"""KV-cached decoding on the B200: the four decode kernels against torch, the engine's prefill + step against its own
recompute path, and ``generate`` against graph-less and per-row recompute decoding."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

dev = torch.device("cuda", 0)


def _attn_oracle(q, kv, lengths, H, dh, slopes, scale):
    d = H * dh
    outs, lses = [], []
    for b, L in enumerate(lengths.tolist()):
        qh = q[b, :d].float().view(H, dh)
        k = kv[b, :L, :d].float().view(L, H, dh)
        v = kv[b, :L, d:].float().view(L, H, dh)
        s = torch.einsum("hd,lhd->hl", qh, k) * scale
        if slopes is not None:
            s = s + slopes[:, None] * (torch.arange(L, device=dev) - (L - 1)).float()[None]
        lses.append(torch.logsumexp(s, -1))
        outs.append(torch.einsum("hl,lhd->hd", torch.softmax(s, -1), v).reshape(d))
    return torch.stack(outs), torch.stack(lses)


@pytest.mark.parametrize("dh", [64, 128])
@pytest.mark.parametrize("alibi", [False, True])
@pytest.mark.parametrize("split", ["one", "max", "auto"])
def test_decode_attention_matches_oracle(dh, alibi, split):
    from photon_b200 import ops
    from photon_b200.models.mpt import alibi_slopes

    H, S_max = 4, 2048
    d = H * dh
    g = torch.Generator(device=dev).manual_seed(dh + 2 * alibi)
    slopes = alibi_slopes(H).to(dev) if alibi else None
    for lens in ([2048], [1, 127, 129], [1, 127, 128, 129, 2048, 5, 640, 1000]):
        B = len(lens)
        kv = torch.full((B, S_max, 2 * d), float("nan"), dtype=torch.bfloat16, device=dev)   # beyond length: never read
        for b, L in enumerate(lens):
            kv[b, :L] = torch.randn(L, 2 * d, generator=g, device=dev).to(torch.bfloat16)
        qkv = torch.randn(B, 3 * d, generator=g, device=dev).to(torch.bfloat16)
        lengths = torch.tensor(lens, dtype=torch.int32, device=dev)
        n_split = {"one": 1, "max": S_max // 32, "auto": 0}[split]
        out = torch.empty(B, d, dtype=torch.bfloat16, device=dev)
        lse = torch.empty(B, H, dtype=torch.float32, device=dev)
        ops.decode_attention(qkv, kv, lengths, slopes, 1.0 / math.sqrt(dh), H, out, lse, n_split=n_split)
        want_o, want_l = _attn_oracle(qkv, kv, lengths, H, dh, slopes, 1.0 / math.sqrt(dh))
        assert torch.isfinite(out.float()).all() and torch.isfinite(lse).all(), lens
        assert (out.float() - want_o).abs().max() < 3e-2, lens
        assert (lse - want_l).abs().max() < 2e-2, lens


@pytest.mark.parametrize("dh", [64, 128])
def test_kv_write_rope_bits_match_rope_kernel(dh):
    from photon_b200 import ops
    from photon_b200.models.mpt import rope_tables

    B, S, H = 3, 256, 4
    d = H * dh
    cos, sin = (t.contiguous() for t in rope_tables(S, dh, 10000.0, dev))
    qkv = torch.randn(B, S, 3 * d, device=dev).to(torch.bfloat16)
    full = ops.rope_(qkv.clone(), cos, sin, H)
    b_idx = torch.tensor([0, 1, 2, 2, 1], dtype=torch.int32, device=dev)
    pos = torch.tensor([0, 1, 127, 128, 255], dtype=torch.int32, device=dev)
    rows = qkv[b_idx.long(), pos.long()].contiguous()
    cache = torch.zeros(B, S, 2 * d, dtype=torch.bfloat16, device=dev)
    ops.kv_write(rows, cache, b_idx, pos, H, rope=(cos, sin))
    want = full[b_idx.long(), pos.long()]
    assert torch.equal(rows.view(torch.int16), want.view(torch.int16))
    assert torch.equal(cache[b_idx.long(), pos.long()].view(torch.int16), want[:, d:].view(torch.int16))
    plain = qkv[b_idx.long(), pos.long()].contiguous()
    cache.zero_()
    ops.kv_write(plain, cache, b_idx, pos, H)
    assert torch.equal(cache[b_idx.long(), pos.long()], plain[:, d:])
    assert torch.equal(plain, qkv[b_idx.long(), pos.long()])      # without rope the row is left as is


def test_embed_at_and_argmax_rows_exact():
    from photon_b200 import ops

    V, d, P = 1000, 256, 64
    wte = torch.randn(V, d, device=dev).to(torch.bfloat16)
    wpe = torch.randn(P, d, device=dev).to(torch.bfloat16)
    ids = torch.tensor([3, 0, V - 1, -5, V + 3, 17], dtype=torch.int64, device=dev)
    pos = torch.tensor([0, 63, 5, 9, 1, 31], dtype=torch.int32, device=dev)
    out = torch.empty(6, d, dtype=torch.bfloat16, device=dev)
    ops.embed_at(ids, pos, wte, wpe, out)
    ref = (wte[ids.clamp(0, V - 1)].float() + wpe[pos.long()].float()).to(torch.bfloat16)
    assert torch.equal(out, ref)
    ops.embed_at(ids, pos, wte, None, out)
    assert torch.equal(out, wte[ids.clamp(0, V - 1)])
    for V in (50368, 1001):
        x = torch.randn(7, V, device=dev).to(torch.bfloat16)
        x[1, 10] = x[1, 4000 % V] = 100.0          # ties -> lowest index
        x[2, :] = 0.0
        x[3, V - 1] = x[3, V - 2] = 50.0
        assert torch.equal(ops.argmax_rows(x), x.float().argmax(-1))
        assert ops.argmax_rows(x)[1] == 10 and ops.argmax_rows(x)[2] == 0


VARIANTS = {"learned": ({}, {}), "alibi": (dict(alibi=True, learned_pos_emb=False), {}), "rope": (dict(rope=True, learned_pos_emb=False), {}),
            "qk_ln": (dict(qk_ln=True), {}), "clip_qkv": (dict(clip_qkv=0.5), {}), "no_bias": (dict(no_bias=True), {}),
            "dh128": (dict(n_heads=2), {}), "ckpt": ({}, dict(activation_checkpointing=True)), "fp8": ({}, dict(precision="amp_fp8"))}


def _engine(variant, msl=512, graph=True):
    from photon_b200.models.engine import B200Engine
    from photon_b200.models.mpt import MPTConfig

    extra, kw = VARIANTS[variant]
    kw = dict(kw)
    cfg = MPTConfig(**{**dict(d_model=256, n_heads=4, n_layers=2, max_seq_len=msl, vocab_size=4096), **extra})
    eng = B200Engine(cfg, dev, kw.pop("precision", "amp_bf16"), {"cuda_graph": graph}, seed=5, **kw)
    eng.train_mode(False)
    assert eng.can_generate
    return eng


def _close(got, want):
    got, want = got.float(), want.float()
    cos = torch.nn.functional.cosine_similarity(got, want, dim=0)
    return cos > 0.999 and (got - want).abs().max() < 5e-2 * want.abs().max(), (float(cos), float((got - want).abs().max()))


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_prefill_and_step_match_engine_recompute(variant):
    eng = _engine(variant)
    g = torch.Generator().manual_seed(1)
    lens = [5, 130, 300]
    ctx = [torch.randint(0, 4096, (n,), generator=g).tolist() for n in lens]
    cont = torch.randint(0, 4096, (3, 64), generator=g)
    dec = eng.decoder(3, max(lens) + 64)
    logits = dec.prefill(ctx)
    for s in range(65):
        for r in range(3):
            ok, err = _close(logits[r], eng.logits(torch.tensor([ctx[r]], device=dev))[0, -1])
            assert ok, (variant, s, r, err)
        if s == 64:
            break
        for r in range(3):
            ctx[r].append(int(cont[r, s]))
        logits = dec.step(cont[:, s].to(dev))
    eng.close()


def _recompute_agrees(eng, prompt, tokens, tol_frac=5e-2):
    """True when ``tokens`` are the recompute path's greedy tokens wherever its top-1/top-2 margin exceeds the logit tolerance
    (after the first near-tie the two continuations may legitimately differ)."""
    ctx = list(prompt)
    for t in tokens:
        lg = eng.logits(torch.tensor([ctx[-eng.cfg.max_seq_len:]], device=dev))[0, -1].float()
        top = lg.topk(2)
        if int(top.indices[0]) != t:
            return float(top.values[0] - top.values[1]) <= tol_frac * float(lg.abs().max())
        ctx.append(t)
    return True


def test_generate_graph_vs_eager_and_recompute():
    eng = _engine("learned")
    g = torch.Generator().manual_seed(2)
    prompts = [torch.randint(0, 4096, (n,), generator=g).tolist() for n in (1, 77, 256, 31)]
    with_graph = eng.generate(prompts, 48)
    eng.use_graph = False
    eng.train_mode(True), eng.train_mode(False)      # drops the cached decoder (and its graph)
    eager = eng.generate(prompts, 48)
    assert with_graph == eager
    assert all(len(t) == 48 for t in eager)
    for p, t in zip(prompts, eager):
        assert _recompute_agrees(eng, p, t)
    eos = eager[1][3]

    def expect(r, seq):
        out = []
        for t in seq:
            if t == eos:
                break
            out.append(t)
            if r == 2 and len(out) == 5:
                break
        return out

    stopped = eng.generate(prompts, 48, eos_id=eos, stop=lambda r, new: r == 2 and len(new) == 5)
    assert stopped == [expect(r, s) for r, s in enumerate(eager)]
    assert len(stopped[1]) <= 3
    eng.close()


def test_generate_row_crossing_max_seq_len_follows_window():
    eng = _engine("learned", msl=512)
    g = torch.Generator().manual_seed(3)
    prompts = [torch.randint(0, 4096, (500,), generator=g).tolist(), torch.randint(0, 4096, (20,), generator=g).tolist(),
               torch.randint(0, 4096, (700,), generator=g).tolist()]      # left-truncated to 512
    out = eng.generate(prompts, 40)
    assert all(len(t) == 40 for t in out)
    for p, t in zip(prompts, out):
        assert _recompute_agrees(eng, p, t)
    eng.close()
