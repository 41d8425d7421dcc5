"""KV-cached greedy decoding on the engine vs per-row recompute, at MPT-125M and MPT-1B with B in {1, 8, 32}, 1024-token prompts
and 256 new tokens (seeded random weights and ids). Per configuration:

* generated tokens/s of ``B200Engine.generate`` (prefill included) and of the recompute path (``ICLEvaluator._generate`` over
  ``B200Engine.logits``, one forward over the whole window per token, one row at a time) on a subset of the rows;
* device-event time of one graph-replayed ``Decoder.step`` (cache filled to ~1100 positions), and the weight bytes one step
  reads (bf16 block matrices + the tied LM head) over that time;
* device-event time of ``decode_attention`` alone on one layer of that cache (256 MiB L2 flush before every timed call), with
  the bytes it must read (sum of lengths * 2d * 2) as achieved HBM bandwidth and share of 7.7 TB/s.

The card's name and power limit are read in the same run and written with the results.

    python scripts/decode_bench.py --out profiles/decode_b200.json
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from photon_b200 import ops  # noqa: E402

HBM_BPS = 7.7e12
dev = torch.device("cuda", 0)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in (q.stdout.splitlines() or [",,"])[0].split(",")][:3]
    return {"name": name or torch.cuda.get_device_name(0), "power_limit": power, "max_sm_clock": clock}


def events_ms(fn, n: int, flush: torch.Tensor | None = None) -> float:
    """Median device time of ``fn`` over ``n`` timed calls (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    ts = []
    for _ in range(n):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


class NullTok:
    eos_token_id = None

    def decode(self, ids):
        return ""


def bench(model: str, B: int, prompt_len: int, new_tokens: int, recompute_rows: int, flush: torch.Tensor) -> dict:
    from photon_b200.config import compose
    from photon_b200.eval.icl import ICLEvaluator
    from photon_b200.models.engine import B200Engine
    from photon_b200.models.mpt import MPTConfig

    cfg = MPTConfig.from_model_cfg(dict(compose([f"llm_config={model}"])["llm_config"]["model"]))
    eng = B200Engine(cfg, dev, "amp_bf16", {}, seed=17)
    eng.train_mode(False)
    g = torch.Generator().manual_seed(B)
    prompts = [torch.randint(0, cfg.vocab_size, (prompt_len,), generator=g).tolist() for _ in range(B)]
    eng.generate(prompts[:1], 4)                                  # module loads / attribute setup outside the timed window
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = eng.generate(prompts, new_tokens)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    n_gen = sum(len(o) for o in out)

    ev = ICLEvaluator(eng.logits, NullTok(), cfg.max_seq_len)
    rows = min(recompute_rows, B)
    ev._generate(prompts[-1], new_tokens, [])                     # noqa: SLF001  (warm-up: every window length is a new shape)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r in range(rows):
        ev._generate(prompts[r], new_tokens, [])                  # noqa: SLF001
    torch.cuda.synchronize()
    t_rec = time.perf_counter() - t0

    # one step, graph-replayed, with the cache filled to prompt_len + 64 positions
    dec = eng.decoder(B, prompt_len + 128)
    dec.prefill(prompts)
    tok = torch.zeros(B, dtype=torch.int64, device=dev)
    for _ in range(64):
        dec.step(tok)
    step_ms = events_ms(dec._graph.replay, 50)                    # noqa: SLF001
    d, L = cfg.d_model, cfg.n_layers
    w_bytes = 2 * (L * (3 * d * d + d * d + 2 * cfg.expansion_ratio * d * d) + cfg.vocab_size * d)
    # decode attention alone: layer 0 of the same cache, lengths as in the step
    lengths = dec.meta[0]
    attn_out = torch.empty(B, d, dtype=torch.bfloat16, device=dev)
    qkv = torch.randn(B, 3 * d, device=dev).to(torch.bfloat16)
    scale = 1.0 / math.sqrt(cfg.d_head)
    attn_ms = events_ms(lambda: ops.decode_attention(qkv, dec.cache[0], lengths, None, scale, cfg.n_heads, attn_out, n_split=dec.n_split),
                        50, flush)
    attn_bytes = int(lengths.sum()) * 2 * d * 2
    res = {"model": model, "batch": B, "prompt_len": prompt_len, "new_tokens": new_tokens,
           "generate": {"tokens": n_gen, "seconds": round(t_gen, 4), "tokens_per_s": round(n_gen / t_gen, 1)},
           "recompute": {"rows": rows, "of_rows": B, "tokens": rows * new_tokens, "seconds": round(t_rec, 4),
                         "tokens_per_s": round(rows * new_tokens / t_rec, 1),
                         "note": "per-row recompute (ICLEvaluator._generate over engine.logits) on a subset of the rows" if rows < B else
                                 "per-row recompute (ICLEvaluator._generate over engine.logits) on every row"},
           "speedup": round((n_gen / t_gen) / (rows * new_tokens / t_rec), 2),
           "step": {"cache_len": prompt_len + 64, "device_ms": round(step_ms, 4), "weight_bytes": w_bytes,
                    "weight_bytes_per_s": round(w_bytes / (step_ms * 1e-3) / 1e12, 3), "weight_bytes_per_s_unit": "TB/s",
                    "share_of_7.7TBps": round(w_bytes / (step_ms * 1e-3) / HBM_BPS, 3),
                    "weight_bound_ms": round(w_bytes / HBM_BPS * 1e3, 4)},
           "decode_attention": {"n_split": dec.n_split, "device_ms": round(attn_ms, 4), "bytes": attn_bytes,
                                "tb_per_s": round(attn_bytes / (attn_ms * 1e-3) / 1e12, 3),
                                "share_of_7.7TBps": round(attn_bytes / (attn_ms * 1e-3) / HBM_BPS, 3), "l2": "flushed (256 MiB) before every call"}}
    del dec
    eng.close()
    del eng
    torch.cuda.empty_cache()
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", default="mpt-125m,mpt-1b")
    ap.add_argument("--batches", default="1,8,32")
    ap.add_argument("--prompt-len", type=int, default=1024)
    ap.add_argument("--new-tokens", type=int, default=256)
    ap.add_argument("--recompute-rows", type=int, default=1, help="rows of each batch decoded by the (slow) per-row recompute path")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("decode_bench needs a CUDA device")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    results = {"card": card(), "torch": torch.__version__, "runs": []}
    for m in a.models.split(","):
        for b in (int(x) for x in a.batches.split(",")):
            r = bench(m, b, a.prompt_len, a.new_tokens, a.recompute_rows, flush)
            print(json.dumps(r), flush=True)
            results["runs"].append(r)
    text = json.dumps(results, indent=1)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
