"""B200Engine — the MPT training step on hand-written sm_100a kernels.

No autograd, no per-op dispatcher: forward and backward are an explicit
schedule of our own kernels over preallocated bf16 activations, flat fp32
master parameters/gradients and a flat bf16 compute shadow
(SURVEY §2.5 (a) K1–K15 → one engine):

* every linear layer = ``csrc/gemm_tcgen05.cu`` (TMA → tcgen05.mma → TMEM →
  fused epilogue): bias, bias+residual, bias+GELU (pre-activation and
  activation written by the same epilogue), dgrad with the stored weight
  consumed MN-major (no transposes), dGELU fused into the dgrad epilogue, wgrad
  with both operands MN-major accumulating in fp32 by TMA reduce-add straight
  into the flat gradient bucket that the DDP all-reduce / optimizer consume;
* LM head + cross-entropy chunked over tokens so the ``[T, 50368]`` logits are
  never materialised (``[chunk, V]`` scratch that stays L2/HBM friendly);
  the chunk's dlogits feed the dgrad/wgrad GEMMs immediately;
* LayerNorm fwd/bwd (+ residual-gradient add), embedding gather/scatter,
  bias-gradient column sums, loss statistics: ``csrc/fused_ops.cu``;
* attention: ``csrc/attention_tcgen05.cu`` (``attention: b200``) or, when
  ``kernels.attention: torch``, cuDNN/FA2 SDPA as an explicit library fallback.

The module tree of :class:`MPTForCausalLM` is kept only as the *owner of names
and initial values*: its parameters are views into the flat fp32 buffer, so the
federated payload / checkpoint order (sorted names) is shared with the torch
backend and the two are directly comparable in tests.
"""
from __future__ import annotations

import math
from typing import Any, Callable

import torch
import torch.nn.functional as F

from photon_b200 import ops
from photon_b200.models.mpt import MPTConfig, MPTForCausalLM, shift_labels
from photon_b200.train.backend import apply_freeze
from photon_b200.utils.flat import FlatParams


class _LayerW:
    """Per-block handles: bf16 weights (shadow plane), fp32 small params and fp32 grads."""

    __slots__ = ("wqkv", "bqkv", "wo", "bo", "wup", "bup", "wdown", "bdown", "g1", "b1", "g2", "b2",
                 "d_wqkv", "d_bqkv", "d_wo", "d_bo", "d_wup", "d_bup", "d_wdown", "d_bdown", "d_g1", "d_b1", "d_g2", "d_b2",
                 "qk_g", "qk_b", "d_qk_g", "d_qk_b")


class B200Engine:
    kind = "b200"

    def __init__(self, cfg: MPTConfig, device: torch.device | str = "cuda", precision: str = "amp_bf16",
                 kernels: dict[str, Any] | None = None, seed: int | None = 17, frozen_layers: list[str] | None = None,
                 unfrozen_layers: list[str] | None = None, unigram_log_probs: torch.Tensor | None = None,
                 lm_head_chunk: int = 18944, grads_storage: torch.Tensor | None = None,
                 activation_checkpointing: bool = False, params_storage: torch.Tensor | None = None,
                 shadow_storage: torch.Tensor | None = None, zero3: Any = None) -> None:
        """``zero3``: a :class:`photon_b200.parallel.zero3.NvlZero3Comm` — full parameter sharding: this rank keeps 1/world of the
        masters / gradients / bf16 weights, block weights are pulled into two rotating buffers one block ahead of the compute
        stream and every block's gradient is reduce-scattered right after its backward (ref: fsdp_config FULL_SHARD)."""
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("B200Engine needs a CUDA (sm_100a) device")
        if precision not in ("amp_bf16", "amp_fp8"):
            raise NotImplementedError(f"B200Engine computes in bf16 (got precision={precision}); use kernels.*=torch for fp32/fp16")
        if frozen_layers or unfrozen_layers:
            raise NotImplementedError("frozen/unfrozen layers run on the torch backend (kernels.*=torch)")
        ops.ext()  # fail loudly if the extension is missing
        self.precision = precision
        self.zero3 = zero3
        if zero3 is not None and precision != "amp_bf16":
            raise NotImplementedError("full parameter sharding runs in amp_bf16 (the fp8 weight copies are quantised from a resident bf16 plane)")
        kernels = dict(kernels or {})
        # amp_fp8 (ref: scripts/centralised_training.sh:91, Composer amp_fp8 -> TransformerEngine): the four GEMMs of every block
        # and their dgrad / wgrad run on tcgen05.mma kind::f8f6f4 (E4M3 activations / weights, E5M2 gradients, per-tensor
        # scaling, fp32 accumulation); LayerNorm, attention, residuals, LM head, loss and optimizer stay bf16 / fp32
        self.fp8 = precision == "amp_fp8"
        self.attn_mode = "torch" if kernels.get("attention", "auto") == "torch" else "b200"
        # kernels.cuda_graph: the ~330 launches of one microbatch are captured once per (batch, seq, loss scaling) and
        # replayed (the schedule is static: preallocated workspace, TMA descriptors baked into the launches)
        # (not under full sharding: the per-block gathers / reductions carry host-side epochs and events)
        self.use_graph = bool(kernels.get("cuda_graph", True)) and zero3 is None
        self._graphs: dict[tuple, Any] = {}
        if self.attn_mode == "b200" and cfg.d_head not in (64, 128):
            # the tcgen05 attention kernels cover d_head 64 and 128 (every shipped MPT config); anything else uses the
            # library attention for BOTH directions (explicit + logged; GEMM/LN/CE/optimizer stay on our kernels)
            print(f"[engine] d_head={cfg.d_head}: attention falls back to SDPA (tcgen05 kernels cover d_head 64 / 128)", flush=True)
            self.attn_mode = "torch"
        self.model = MPTForCausalLM(cfg, device=self.device, seed=seed)
        self.frozen = apply_freeze(self.model, frozen_layers, unfrozen_layers)
        if zero3 is not None:
            from photon_b200.parallel.zero3 import ShardedFlat

            # same initial weights as an unsharded engine with this seed: materialise once, keep the shard, drop the rest
            init = FlatParams(self.model, device=self.device, with_grad=False)
            if init.layout.total != zero3.plan.layout.total or init.layout.names != zero3.plan.layout.names:
                raise ValueError("the ZeRO-3 communicator was planned for a different parameter layout")
            zero3.load_full_params(init.params)
            del init
            self.model = None
            self.flat = ShardedFlat(zero3)
            self.bf16_params = zero3.w16        # this rank's shard of the bf16 weights (what the optimizer kernel writes)
        else:
            self.flat = FlatParams(self.model, device=self.device, params_storage=params_storage, grads_storage=grads_storage)
            # bf16 compute copy; lives in a symmetric arena plane when a fused NVLink step writes it from peer GPUs
            self.bf16_params = shadow_storage if shadow_storage is not None else torch.zeros(
                self.flat.layout.total, dtype=torch.bfloat16, device=self.device)
            if self.bf16_params.numel() != self.flat.layout.total or self.bf16_params.dtype != torch.bfloat16:
                raise ValueError("shadow_storage must be a bf16 tensor with layout.total elements")
        self.unigram_log_probs = unigram_log_probs.to(self.device) if unigram_log_probs is not None else None
        self.lm_head_chunk = int(lm_head_chunk)
        # positional variants of the MPT attention block (ref: SURVEY §5.7): ALiBi slopes enter the attention kernels,
        # RoPE rotates q / k in place after the QKV GEMM (and un-rotates their gradients)
        from photon_b200.models.mpt import alibi_slopes, rope_tables

        self.alibi = alibi_slopes(cfg.n_heads, cfg.alibi_bias_max).to(self.device, torch.float32).contiguous() if cfg.alibi else None
        self.rope = tuple(t.contiguous() for t in rope_tables(cfg.max_seq_len, cfg.d_head, cfg.rope_theta, self.device)) if cfg.rope else None
        # keep only the block inputs h[i]; every block's internals are recomputed right before its backward
        # (fsdp_config.activation_checkpointing, ref: conf/llm_config/mpt-1b.yaml:88): 16·T·d·L bytes of bf16 -> 16·T·d
        self.activation_checkpointing = bool(activation_checkpointing)
        self.collect_activation_stats = False
        self.activation_stats: dict[str, float] = {}
        self.launches_per_microbatch = 0
        self._ws: dict[tuple[int, int], dict[str, Any]] = {}
        self._stats = torch.zeros(4, dtype=torch.float64, device=self.device)
        self._gen_decoder: Decoder | None = None    # kept between generate() calls of one evaluation
        self._bind()
        if self.fp8:
            self._init_fp8(int(kernels.get("fp8_amax_history_len", 16)), int(kernels.get("fp8_margin", 0)))
        self.params_updated()

    # ------------------------------------------------------------------ binding
    def _bind(self) -> None:
        lay, P, G, Sd = self.flat.layout, self.flat.params, self.flat.grads, self.bf16_params
        have = set(lay.names)
        # biases are absent under `no_bias`: every consumer below accepts None (GEMM without bias, LN without beta,
        # no bias-gradient column sums)
        v32 = lambda n: lay.view(P, "transformer." + n) if "transformer." + n in have else None  # noqa: E731
        vg = lambda n: lay.view(G, "transformer." + n) if "transformer." + n in have else None  # noqa: E731
        v16 = lambda n: lay.view(Sd, "transformer." + n)  # noqa: E731
        if self.zero3 is not None:
            # weights: views into the two rotating block buffers (block i -> buffer i % 2) / the resident embedding buffer;
            # 1-D fp32 parameters: the packed resident buffer; gradients: the block's staging plane (reduced after its backward)
            z = self.zero3
            v32 = lambda n: z.small("transformer." + n) if "transformer." + n in have else None  # noqa: E731
            vg = lambda n: z.grad("transformer." + n) if "transformer." + n in have else None  # noqa: E731
            v16 = lambda n: z.weight("transformer." + n)  # noqa: E731
        has_wpe = self.cfg.learned_pos_emb
        self.wte16, self.wpe16 = v16("wte.weight"), (v16("wpe.weight") if has_wpe else None)
        self.d_wte, self.d_wpe = vg("wte.weight"), (vg("wpe.weight") if has_wpe else None)
        self.gf, self.bf, self.d_gf, self.d_bf = v32("norm_f.weight"), v32("norm_f.bias"), vg("norm_f.weight"), vg("norm_f.bias")
        self.layers: list[_LayerW] = []
        for i in range(self.cfg.n_layers):
            p = f"blocks.{i}."
            w = _LayerW()
            w.wqkv, w.wo, w.wup, w.wdown = (v16(p + "attn.Wqkv.weight"), v16(p + "attn.out_proj.weight"),
                                            v16(p + "ffn.up_proj.weight"), v16(p + "ffn.down_proj.weight"))
            w.bqkv, w.bo, w.bup, w.bdown = (v32(p + "attn.Wqkv.bias"), v32(p + "attn.out_proj.bias"),
                                            v32(p + "ffn.up_proj.bias"), v32(p + "ffn.down_proj.bias"))
            w.g1, w.b1, w.g2, w.b2 = v32(p + "norm_1.weight"), v32(p + "norm_1.bias"), v32(p + "norm_2.weight"), v32(p + "norm_2.bias")
            w.d_wqkv, w.d_wo, w.d_wup, w.d_wdown = (vg(p + "attn.Wqkv.weight"), vg(p + "attn.out_proj.weight"),
                                                    vg(p + "ffn.up_proj.weight"), vg(p + "ffn.down_proj.weight"))
            w.d_bqkv, w.d_bo, w.d_bup, w.d_bdown = (vg(p + "attn.Wqkv.bias"), vg(p + "attn.out_proj.bias"),
                                                    vg(p + "ffn.up_proj.bias"), vg(p + "ffn.down_proj.bias"))
            w.d_g1, w.d_b1, w.d_g2, w.d_b2 = vg(p + "norm_1.weight"), vg(p + "norm_1.bias"), vg(p + "norm_2.weight"), vg(p + "norm_2.bias")
            # attn_config.qk_ln: LayerNorm over d_model on the query and key projections
            w.qk_g = [v32(p + "attn.q_ln.weight"), v32(p + "attn.k_ln.weight")]
            w.qk_b = [v32(p + "attn.q_ln.bias"), v32(p + "attn.k_ln.bias")]
            w.d_qk_g = [vg(p + "attn.q_ln.weight"), vg(p + "attn.k_ln.weight")]
            w.d_qk_b = [vg(p + "attn.q_ln.bias"), vg(p + "attn.k_ln.bias")]
            self.layers.append(w)

    def params_updated(self) -> None:
        """Re-cast the bf16 compute shadow from the fp32 masters. Only needed after host-side
        parameter loads: the fused optimizer and the round-broadcast kernels write the shadow
        themselves (the Trainer skips this call in that case)."""
        if self.zero3 is not None:
            self.zero3.before_param_write()
            ops.cast_bf16(self.flat.params, self.bf16_params)
            self.zero3.params_changed()
            return
        ops.cast_bf16(self.flat.params, self.bf16_params)

    # ---------------------------------------------------------------------- fp8
    _DYN_ROLES = ("x_ln1", "x_attn", "x_ln2", "x_u", "g_dqkv", "g_dhmid", "g_dz", "g_dh")   # per block: 4 × E4M3, 4 × E5M2
    _W_ROLES = ("wqkv", "wo", "wup", "wdown")

    def _init_fp8(self, history_len: int, margin: int) -> None:
        """Device-resident scaling state: ``meta`` = [3, n_roles] (scale, 1/scale, running amax). Roles [0, 8L) are activations
        and gradients (delayed scaling: amax history → next scale, ``ops.fp8_update_scales``); roles [8L, 12L) are the weight
        matrices (current scaling, re-quantised from the bf16 shadow at the start of every microbatch — two passes over
        ≤ 2 bytes/param, so whoever wrote the shadow (optimizer, round broadcast, ZeRO step) needs no hook)."""
        L, lay, dev = self.cfg.n_layers, self.flat.layout, self.device
        self._n_dyn = len(self._DYN_ROLES) * L
        n_roles = self._n_dyn + len(self._W_ROLES) * L
        self.fp8_meta = torch.zeros(3, n_roles, dtype=torch.float32, device=dev)
        self.fp8_meta[:2] = 1.0
        self.fp8_hist = torch.zeros(self._n_dyn, max(1, history_len), dtype=torch.float32, device=dev)
        self.fp8_fmax = torch.tensor([ops.FP8_MAX[0 if j < 4 else 1] for _ in range(L) for j in range(8)], dtype=torch.float32, device=dev)
        self.fp8_pos = torch.zeros(1, dtype=torch.int32, device=dev)
        self.fp8_margin_mult = float(2.0 ** margin)
        self.w8 = torch.zeros(lay.total, dtype=torch.uint8, device=dev)      # E4M3 weights at the flat layout's offsets
        seg, self.w8_views = [], []
        for i in range(L):
            views = {}
            for key, name in zip(self._W_ROLES, ("attn.Wqkv.weight", "attn.out_proj.weight", "ffn.up_proj.weight", "ffn.down_proj.weight")):
                j = lay.index(f"transformer.blocks.{i}.{name}")
                seg.append((lay.offsets[j], lay.numels[j]))
                views[key] = lay.view(self.w8, j)
            self.w8_views.append(views)
        self.w8_seg = torch.tensor(seg, dtype=torch.int64, device=dev)
        self._fp8_calibrated = False

    def _role(self, name: str, layer: int) -> int:
        if name in self._DYN_ROLES:
            return layer * len(self._DYN_ROLES) + self._DYN_ROLES.index(name)
        return self._n_dyn + layer * len(self._W_ROLES) + self._W_ROLES.index(name)

    def _fp8_prologue(self, train: bool) -> None:
        """Start of a microbatch: roll the delayed scales (training only) and re-quantise the weights from the shadow."""
        if train:
            ops.fp8_update_scales(self.fp8_meta, self.fp8_hist, self.fp8_fmax, self.fp8_pos, self._n_dyn, self.fp8_margin_mult)
        ops.fp8_quantize_segments(self.bf16_params, self.w8, self.w8_seg, self.fp8_meta, self._n_dyn)

    def fp8_state_dict(self) -> dict[str, Any] | None:
        """Scales / amax histories, checkpointed next to the optimizer so a resumed run casts with the scales it stopped with."""
        if not self.fp8:
            return None
        return {"meta": self.fp8_meta.cpu(), "hist": self.fp8_hist.cpu(), "pos": self.fp8_pos.cpu(), "calibrated": self._fp8_calibrated}

    def load_fp8_state_dict(self, sd: dict[str, Any]) -> None:
        if self.fp8 and sd and "meta" in sd and tuple(sd["meta"].shape) == tuple(self.fp8_meta.shape):
            self.fp8_meta.copy_(sd["meta"]), self.fp8_hist.copy_(sd["hist"]), self.fp8_pos.copy_(sd["pos"])
            self._fp8_calibrated = bool(sd.get("calibrated", True))

    # ---------------------------------------------------------------- workspace
    def _workspace(self, b: int, S: int, fp8: bool | None = None) -> dict[str, Any]:
        """``fp8=False`` on an amp_fp8 engine: bf16 block buffers (the decoder's prefill runs the bf16 GEMMs)."""
        use8 = self.fp8 if fp8 is None else bool(fp8)
        key = (b, S, use8)
        if key in self._ws:
            return self._ws[key]
        self._ws.clear()  # one live shape at a time (activations dominate memory)
        self._graphs.clear()  # captured graphs point into the old workspace
        c, dev = self.cfg, self.device
        T, d, H, L = b * S, c.d_model, c.n_heads, c.n_layers
        bf = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=dev)  # noqa: E731
        f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
        ws: dict[str, Any] = {"h": [bf(T, d) for _ in range(L + 1)], "layers": []}
        for i in range(L):
            if self.activation_checkpointing and i > 0:
                ws["layers"].append(ws["layers"][0])  # ONE set of block internals shared by all layers
                continue
            if use8:   # the GEMM inputs exist only as E4M3 (1 byte): 7·T·d instead of 12·T·d bytes of saved activations
                u8 = lambda *s: torch.empty(*s, dtype=torch.uint8, device=dev)  # noqa: E731
                ws["layers"].append({"ln1": u8(T, d), "m1": f32(T), "r1": f32(T), "qkv": bf(T, 3 * d), "attn": bf(T, d), "attn8": u8(T, d),
                                     "lse": f32(b, H, S), "hmid": bf(T, d), "ln2": u8(T, d), "m2": f32(T), "r2": f32(T),
                                     "z": bf(T, c.expansion_ratio * d), "u": u8(T, c.expansion_ratio * d)})
            else:
                ws["layers"].append({"ln1": bf(T, d), "m1": f32(T), "r1": f32(T), "qkv": bf(T, 3 * d), "attn": bf(T, d),
                                     "lse": f32(b, H, S), "hmid": bf(T, d), "ln2": bf(T, d), "m2": f32(T), "r2": f32(T),
                                     "z": bf(T, c.expansion_ratio * d), "u": bf(T, c.expansion_ratio * d)})
            if c.clip_qkv:
                ws["layers"][-1]["clipmask"] = torch.empty(T, 3 * d, dtype=torch.bool, device=dev)
            if c.qk_ln:   # pre-LayerNorm q / k (inputs of the two LN backward passes) and their row statistics
                ws["layers"][-1].update(qk_pre=[bf(T, d), bf(T, d)], qk_m=[f32(T), f32(T)], qk_r=[f32(T), f32(T)])
        if c.qk_ln:
            ws.update(qk_tmp=bf(T, d), qk_tmp2=bf(T, d))
        ws.update(lnf=bf(T, d), mf=f32(T), rf=f32(T), dlnf=bf(T, d), dh=bf(T, d), dhmid=bf(T, d), dln=bf(T, d),
                  dqkv=bf(T, 3 * d), dattn=bf(T, d), dz=bf(T, c.expansion_ratio * d), delta=f32(b, H, S),
                  logits=bf(min(self.lm_head_chunk, T), c.vocab_size))
        if use8:   # E5M2 copy of the gradient currently flowing backward (one buffer, viewed at the width in use)
            ws["g8"] = torch.empty(T * max(c.expansion_ratio, 3) * d, dtype=torch.uint8, device=dev)
        self._ws[key] = ws
        return ws

    # ------------------------------------------------------------------ forward
    def _attention_fwd(self, lw: dict[str, Any], b: int, S: int) -> None:
        c = self.cfg
        scale = 1.0 / math.sqrt(c.d_head)
        if self.attn_mode == "b200" and S % 128 == 0:
            ops.attention_fwd(lw["qkv"].view(b, S, 3 * c.d_model), lw["attn"].view(b, S, c.d_model), lw["lse"], c.n_heads, scale, True,
                              self.alibi)
            return
        # library attention: kernels.attention=torch, an unsupported d_head, or a sequence length that is not a multiple
        # of the 128-row tiles (the shipped configs use 2048)
        q, k, v = lw["qkv"].view(b, S, 3, c.n_heads, c.d_head).permute(2, 0, 3, 1, 4)
        o = F.scaled_dot_product_attention(q, k, v, scale=scale, **self._sdpa_mask(S, q.dtype))
        lw["attn"].view(b, S, c.n_heads, c.d_head).copy_(o.transpose(1, 2))

    def _sdpa_mask(self, S: int, dtype: torch.dtype) -> dict[str, Any]:
        if self.alibi is None:
            return {"is_causal": True}
        pos = torch.arange(S, device=self.device)
        bias = self.alibi[:, None, None] * (pos[None, :] - pos[:, None]).clamp(max=0).float()[None]
        keep = torch.ones(S, S, dtype=torch.bool, device=self.device).tril()
        return {"attn_mask": bias.masked_fill(~keep, float("-inf")).to(dtype)[None]}

    def _attention_bwd(self, lw: dict[str, Any], ws: dict[str, Any], b: int, S: int) -> None:
        c = self.cfg
        scale = 1.0 / math.sqrt(c.d_head)
        if self.attn_mode == "b200" and S % 128 == 0:
            ops.attention_bwd(lw["qkv"].view(b, S, 3 * c.d_model), lw["attn"].view(b, S, c.d_model),
                              ws["dattn"].view(b, S, c.d_model), lw["lse"], ws["dqkv"].view(b, S, 3 * c.d_model), ws["delta"],
                              c.n_heads, scale, True, self.alibi)
            if self.rope is not None:   # gradients w.r.t. the un-rotated q, k
                ops.rope_(ws["dqkv"].view(b, S, 3 * c.d_model), self.rope[0], self.rope[1], c.n_heads, inverse=True)
            return
        with torch.enable_grad():
            qkv = lw["qkv"].view(b, S, 3, c.n_heads, c.d_head).detach().requires_grad_(True)
            q, k, v = qkv.permute(2, 0, 3, 1, 4)
            o = F.scaled_dot_product_attention(q, k, v, scale=scale, **self._sdpa_mask(S, q.dtype))
            (g,) = torch.autograd.grad(o, qkv, ws["dattn"].view(b, S, c.n_heads, c.d_head).transpose(1, 2))
        ws["dqkv"].view(b, S, 3, c.n_heads, c.d_head).copy_(g)
        if self.rope is not None:
            ops.rope_(ws["dqkv"].view(b, S, 3 * c.d_model), self.rope[0], self.rope[1], c.n_heads, inverse=True)

    def _block_fwd(self, i: int, ws: dict[str, Any], b: int, S: int, fp8: bool | None = None) -> None:
        """h[i] -> h[i+1]; the block internals land in ws["layers"][i] (also the recompute step under checkpointing).
        ``fp8=False`` runs the bf16 GEMMs on an amp_fp8 engine (decoder prefill)."""
        c, h, w, lw = self.cfg, ws["h"], self.layers[i], ws["layers"][i]
        use8 = self.fp8 if fp8 is None else bool(fp8)
        if use8:
            M, w8, R = self.fp8_meta, self.w8_views[i], self._role
            ops.layernorm_fwd_q8(h[i], w.g1, w.b1, lw["ln1"], lw["m1"], lw["r1"], c.norm_eps, M, R("x_ln1", i))
            ops.gemm_fp8(lw["ln1"], w8["wqkv"], lw["qkv"], M, R("x_ln1", i), R("wqkv", i), bias=w.bqkv)
        else:
            ops.layernorm_fwd(h[i], w.g1, w.b1, lw["ln1"], lw["m1"], lw["r1"], c.norm_eps)
            ops.linear_fwd(lw["ln1"], w.wqkv, w.bqkv, lw["qkv"])
        if c.clip_qkv:   # attn_config.clip_qkv: clamp the fused projection; remember where the gradient passes
            torch.logical_and(lw["qkv"] > -c.clip_qkv, lw["qkv"] < c.clip_qkv, out=lw["clipmask"])
            lw["qkv"].clamp_(-c.clip_qkv, c.clip_qkv)
        if c.qk_ln:   # the q / k thirds are strided inside the fused buffer: normalise contiguous copies
            qkv3 = lw["qkv"].view(-1, 3, c.d_model)
            for j in range(2):
                lw["qk_pre"][j].copy_(qkv3[:, j])
                ops.layernorm_fwd(lw["qk_pre"][j], w.qk_g[j], w.qk_b[j], ws["qk_tmp"], lw["qk_m"][j], lw["qk_r"][j], c.norm_eps)
                qkv3[:, j].copy_(ws["qk_tmp"])
        if self.rope is not None:
            ops.rope_(lw["qkv"].view(b, S, 3 * c.d_model), self.rope[0], self.rope[1], c.n_heads)
        self._attention_fwd(lw, b, S)
        if use8:
            ops.colsum_quant(lw["attn"], None, lw["attn8"], ops.E4M3, M, R("x_attn", i))
            ops.gemm_fp8(lw["attn8"], w8["wo"], lw["hmid"], M, R("x_attn", i), R("wo", i), epi=ops.EPI_RESIDUAL, bias=w.bo, aux=h[i])
            ops.layernorm_fwd_q8(lw["hmid"], w.g2, w.b2, lw["ln2"], lw["m2"], lw["r2"], c.norm_eps, M, R("x_ln2", i))
            # gelu(z) leaves the epilogue as E4M3 (the down-projection's operand), gelu'(z) as bf16 (the dgrad multiplier)
            ops.gemm_fp8(lw["ln2"], w8["wup"], lw["z"], M, R("x_ln2", i), R("wup", i), epi=ops.EPI_GELU_GRAD_Q8, bias=w.bup, out2=lw["z"],
                         out8=lw["u"], role_out=R("x_u", i))
            ops.gemm_fp8(lw["u"], w8["wdown"], h[i + 1], M, R("x_u", i), R("wdown", i), epi=ops.EPI_RESIDUAL, bias=w.bdown, aux=lw["hmid"])
            return
        ops.linear_fwd(lw["attn"], w.wo, w.bo, lw["hmid"], residual=h[i])
        ops.layernorm_fwd(lw["hmid"], w.g2, w.b2, lw["ln2"], lw["m2"], lw["r2"], c.norm_eps)
        ops.linear_gelu_grad_fwd(lw["ln2"], w.wup, w.bup, lw["z"], lw["u"])   # lw["z"] holds gelu'(pre-activation)
        ops.linear_fwd(lw["u"], w.wdown, w.bdown, h[i + 1], residual=lw["hmid"])

    def _forward(self, ids: torch.Tensor, ws: dict[str, Any]) -> None:
        c = self.cfg
        b, S = ids.shape
        h = ws["h"]
        z = self.zero3
        if z is not None:
            z.ensure_resident()
        ops.embed_fwd(ids.reshape(-1), self.wte16, self.wpe16, h[0], S)
        for i in range(c.n_layers):
            if z is not None:
                z.acquire(i)          # block i's weights are in buffer i % 2 (stream-ordered wait) ...
                z.prefetch(i + 1)     # ... and block i+1 streams into the other one while block i computes
            self._block_fwd(i, ws, b, S)
            if self.collect_activation_stats:
                x = h[i + 1][:S].float()
                self.activation_stats[f"l2_norm/block_{i}"] = float(x.norm(dim=-1).mean())
                self.activation_stats[f"max/block_{i}"] = float(x.abs().max())
        ops.layernorm_fwd(h[c.n_layers], self.gf, self.bf, ws["lnf"], ws["mf"], ws["rf"], c.norm_eps)

    def _head(self, ws: dict[str, Any], targets: torch.Tensor, grad_scale: float, train: bool) -> None:
        """Chunked LM head + fused CE (+ immediate head backward when training)."""
        T = targets.numel()
        step = ws["logits"].shape[0]
        for lo in range(0, T, step):
            hi = min(T, lo + step)
            logits = ws["logits"][: hi - lo]
            ops.gemm(ws["lnf"][lo:hi], self.wte16, logits)
            ops.cross_entropy(logits, targets[lo:hi], grad_scale, train, self._stats, None, self.unigram_log_probs)
            if train:
                ops.linear_dgrad(logits, self.wte16, ws["dlnf"][lo:hi])
                ops.linear_wgrad(logits, ws["lnf"][lo:hi], self.d_wte, accumulate=True)

    # ----------------------------------------------------------------- backward
    def _linear_bwd(self, i: int, ws: dict[str, Any], dy: torch.Tensor, g_role: str, x: torch.Tensor, x_role: str, w_role: str,
                    w16: torch.Tensor, dw: torch.Tensor, db: torch.Tensor | None, dx: torch.Tensor, mul: torch.Tensor | None = None) -> None:
        """Backward of ``y = x @ w^T + b``: db += colsum(dy); dw += dy^T x; dx = dy w (optionally ``* mul``).
        fp8: the column-sum pass also emits the E5M2 copy of ``dy`` both GEMMs read; ``x`` is the saved E4M3 input."""
        if not self.fp8:
            if db is not None:
                ops.col_sum(dy, db)
            ops.linear_wgrad(dy, x, dw)
            ops.linear_dgrad(dy, w16, dx, mul=mul)
            return
        M, R = self.fp8_meta, self._role
        T, n = dy.shape
        dy8 = ws["g8"][: T * n].view(T, n)
        ops.colsum_quant(dy, db, dy8, ops.E5M2, M, R(g_role, i))
        ops.gemm_fp8(dy8, x, dw, M, R(g_role, i), R(x_role, i), a_mn=True, b_mn=True, epi=ops.EPI_F32, a_fmt=ops.E5M2, b_fmt=ops.E4M3,
                     accumulate=True)
        ops.gemm_fp8(dy8, self.w8_views[i][w_role], dx, M, R(g_role, i), R(w_role, i), b_mn=True, epi=ops.EPI_MUL if mul is not None else ops.EPI_BF16,
                     a_fmt=ops.E5M2, b_fmt=ops.E4M3, aux=mul)

    def _backward(self, ids: torch.Tensor, ws: dict[str, Any]) -> None:
        c = self.cfg
        b, S = ids.shape
        h = ws["h"]
        dh, dhmid, dln = ws["dh"], ws["dhmid"], ws["dln"]
        z = self.zero3
        ops.layernorm_bwd(ws["dlnf"], h[c.n_layers], self.gf, ws["mf"], ws["rf"], None, dh, self.d_gf, self.d_bf)
        for i in range(c.n_layers - 1, -1, -1):
            w, lw = self.layers[i], ws["layers"][i]
            if z is not None:
                z.acquire(i)
                z.prefetch(i - 1)
                z.zero_stage(i)       # this microbatch's gradient of block i (the shard accumulates over microbatches)
            if self.activation_checkpointing and i < c.n_layers - 1:
                self._block_fwd(i, ws, b, S)   # recompute (the shared buffers still hold the LAST block after the forward)
            # ---- FFN: h[i+1] = hmid + down(gelu(up(ln2(hmid))))
            self._linear_bwd(i, ws, dh, "g_dh", lw["u"], "x_u", "wdown", w.wdown, w.d_wdown, w.d_bdown, ws["dz"], mul=lw["z"])
            self._linear_bwd(i, ws, ws["dz"], "g_dz", lw["ln2"], "x_ln2", "wup", w.wup, w.d_wup, w.d_bup, dln)
            ops.layernorm_bwd(dln, lw["hmid"], w.g2, lw["m2"], lw["r2"], dh, dhmid, w.d_g2, w.d_b2)
            # ---- attention: hmid = h[i] + out_proj(attn(qkv(ln1(h[i]))))
            self._linear_bwd(i, ws, dhmid, "g_dhmid", lw["attn8"] if self.fp8 else lw["attn"], "x_attn", "wo", w.wo, w.d_wo, w.d_bo, ws["dattn"])
            self._attention_bwd(lw, ws, b, S)
            if c.qk_ln:
                dqkv3 = ws["dqkv"].view(-1, 3, c.d_model)
                for j in range(2):
                    ws["qk_tmp"].copy_(dqkv3[:, j])
                    ops.layernorm_bwd(ws["qk_tmp"], lw["qk_pre"][j], w.qk_g[j], lw["qk_m"][j], lw["qk_r"][j], None, ws["qk_tmp2"],
                                      w.d_qk_g[j], w.d_qk_b[j])
                    dqkv3[:, j].copy_(ws["qk_tmp2"])
            if c.clip_qkv:
                ws["dqkv"].mul_(lw["clipmask"])
            self._linear_bwd(i, ws, ws["dqkv"], "g_dqkv", lw["ln1"], "x_ln1", "wqkv", w.wqkv, w.d_wqkv, w.d_bqkv, dln)
            ops.layernorm_bwd(dln, h[i], w.g1, lw["m1"], lw["r1"], dhmid, dh, w.d_g1, w.d_b1)
            if z is not None:
                z.reduce(i)           # reduce-scatter: every rank adds the mean of ITS slice into its gradient shard
        ops.embed_bwd(ids.reshape(-1), dh, self.d_wte, self.d_wpe, S)
        if z is not None:
            z.reduce(z.plan.rest)

    # ---------------------------------------------------------------- protocol
    def _fwd_bwd_eager(self, ids: torch.Tensor, grad_scale: float) -> None:
        b, S = ids.shape
        ws = self._workspace(b, S)
        targets = shift_labels(ids).reshape(-1)
        self._stats.zero_()
        if self.fp8:
            self._fp8_prologue(train=True)
        if self.zero3 is not None:
            self.zero3.zero_stage(self.zero3.plan.rest)   # embeddings + final norm collect gradients over the whole backward
        self._forward(ids, ws)
        self._head(ws, targets, grad_scale, train=True)
        self._backward(ids, ws)

    def fwd_bwd(self, ids: torch.Tensor, denom: float, scale: float = 1.0) -> tuple[torch.Tensor, torch.Tensor]:
        """Accumulate d(Σ token-loss · scale / denom) into ``flat.grads``; returns (loss_sum, n_tokens)."""
        b, S = ids.shape
        grad_scale = scale / denom
        if self.fp8 and not self._fp8_calibrated:
            # delayed scaling has no history yet: one discarded pass at scale 1 records every role's amax (gradients would
            # underflow E5M2 unscaled), the next prologue turns them into scales
            saved = self.flat.grads.clone()
            self._fwd_bwd_eager(ids, grad_scale)
            self.flat.grads.copy_(saved)
            self._fp8_calibrated = True
        graphable = self.use_graph and self.attn_mode == "b200" and S % 128 == 0 and not self.collect_activation_stats
        if not graphable:
            n0 = ops.launch_count()
            self._fwd_bwd_eager(ids, grad_scale)
            self.launches_per_microbatch = ops.launch_count() - n0
        else:
            key = (b, S, float(grad_scale))
            g = self._graphs.get(key)
            if g is None:
                g = self._capture(ids, grad_scale, key)
            g["ids"].copy_(ids, non_blocking=True)
            g["graph"].replay()
            ops.add_launch_count(self.launches_per_microbatch)   # replayed launches are still our kernels
        st = self._stats.clone()
        return st[0], st[1]

    def _capture(self, ids: torch.Tensor, grad_scale: float, key: tuple) -> dict[str, Any]:
        """Warm up eagerly on a side stream (lazy allocations, kernel attributes), then capture one microbatch.
        Gradients accumulate into ``flat.grads`` — they are saved around the warm-up / capture passes."""
        if len(self._graphs) >= 4:      # shapes changed (auto microbatch, eval): drop old graphs with their static inputs
            self._graphs.clear()
        static_ids = ids.clone()
        saved = self.flat.grads.clone()
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            n0 = ops.launch_count()
            self._fwd_bwd_eager(static_ids, grad_scale)
            self.launches_per_microbatch = ops.launch_count() - n0
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._fwd_bwd_eager(static_ids, grad_scale)
        self.flat.grads.copy_(saved)
        g = {"graph": graph, "ids": static_ids}
        self._graphs[key] = g
        return g

    @torch.no_grad()
    def eval_stats(self, ids: torch.Tensor) -> dict[str, torch.Tensor]:
        b, S = ids.shape
        ws = self._workspace(b, S)
        targets = shift_labels(ids).reshape(-1)
        self._stats.zero_()
        if self.fp8:
            self._fp8_prologue(train=False)
        self._forward(ids, ws)
        self._head(ws, targets, 0.0, train=False)
        st = self._stats.clone()
        out = {"loss_sum": st[0], "n_tokens": st[1], "n_correct": st[2]}
        if self.unigram_log_probs is not None:
            out["unigram_loss_sum"] = st[3]
        return out

    @torch.no_grad()
    def logits(self, ids: torch.Tensor) -> torch.Tensor:
        """``[B,S] → [B,S,V]`` for the in-context-learning evaluator. ICL prompts are ragged single sequences scored a
        handful of tokens at a time — nothing like the fixed ``[b, 2048]`` schedule the kernel workspace is laid out for — so
        this runs the torch module that shares the fp32 master weights (bf16 autocast, SDPA); it is an evaluation utility,
        not part of the training step."""
        if self.model is None:
            # full parameter sharding: the evaluation utility gets a temporary whole-model copy, pulled from the owners by THIS rank's
            # copy engines (peers only have to leave their shards alone — the trainer keeps them at a barrier during the ICL suite);
            # it is rebuilt when the parameters have changed and dropped by ``train_mode(True)``
            ver = self.zero3.version
            if getattr(self, "_eval_model", None) is None or self._eval_model_version != ver:
                m = MPTForCausalLM(self.cfg, device=self.device, seed=0)
                fp = FlatParams(m, device=self.device, with_grad=False)
                fp.params.copy_(self.flat.full_params())
                m.train(False)
                self._eval_model, self._eval_model_version = m, ver
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return self._eval_model(ids.to(self.device))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return self.model(ids.to(self.device))

    # --------------------------------------------------------------- generation
    @property
    def can_generate(self) -> bool:
        """KV-cached decoding runs on this engine: unsharded weights, the tcgen05 attention path with d_head 64 / 128, and a
        ``max_seq_len`` that is a multiple of the 128-row prefill tiles. Under amp_fp8 decoding reads the bf16 shadow with
        the bf16 GEMMs (there is no fp8 decode path)."""
        return (self.zero3 is None and self.attn_mode == "b200" and self.cfg.d_head in (64, 128)
                and self.cfg.max_seq_len % 128 == 0)

    def decoder(self, batch: int, max_len: int) -> "Decoder":
        """A decoding session for ``batch`` rows of up to ``max_len`` tokens (prompt + generated) over this engine's weights."""
        if not self.can_generate:
            raise NotImplementedError("KV-cached decoding needs zero3=None, attention=b200, d_head 64/128 and max_seq_len % 128 == 0")
        return Decoder(self, batch, max_len)

    @torch.no_grad()
    def generate(self, prompts: list[list[int]], max_new_tokens: int, eos_id: int | None = None,
                 stop: Callable[[int, list[int]], bool] | None = None) -> list[list[int]]:
        """Greedy continuation of every prompt, batched, with a KV cache; returns the new ids of each row.

        Same semantics as per-row recompute (``ICLEvaluator._generate`` over :meth:`logits`): prompts are left-truncated to
        ``max_seq_len``; a row ends at ``eos_id`` (not included), when ``stop(row, new_ids)`` returns True, or after
        ``max_new_tokens``. A row whose context outgrows ``max_seq_len`` continues over its last ``max_seq_len`` ids,
        recomputed through :meth:`logits` at each such step (its positions shift, so the cache no longer applies)."""
        B, msl = len(prompts), self.cfg.max_seq_len
        new: list[list[int]] = [[] for _ in range(B)]
        if B == 0 or max_new_tokens <= 0:
            return new
        ctx = [list(p)[-msl:] for p in prompts]
        need = min(msl, max(len(c) for c in ctx) + max_new_tokens)
        dec = self._gen_decoder
        if dec is None or dec.B != B or dec.S_max < need:
            self._gen_decoder = None     # free the old cache first
            dec = self._gen_decoder = self.decoder(B, need)
        nxt = ops.argmax_rows(dec.prefill(ctx), out=dec.next_ids)
        host = torch.empty(B, dtype=torch.int64, pin_memory=True)
        done, windowed, wtok = [False] * B, [False] * B, [0] * B
        for it in range(max_new_tokens):
            host.copy_(nxt, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            toks = host.tolist()
            for r in range(B):
                if done[r]:
                    continue
                t = wtok[r] if windowed[r] else toks[r]
                if eos_id is not None and t == eos_id:
                    done[r] = True
                    continue
                new[r].append(t)
                ctx[r].append(t)
                if stop is not None and stop(r, new[r]):
                    done[r] = True
            if all(done) or it == max_new_tokens - 1:
                break
            for r in range(B):
                if not done[r] and len(ctx[r]) > msl:
                    windowed[r] = True
                    wtok[r] = int(self.logits(torch.tensor([ctx[r][-msl:]], device=self.device))[0, -1].float().argmax())
            active = [not (done[r] or windowed[r]) for r in range(B)]
            if any(active):
                nxt = ops.argmax_rows(dec.step(nxt, active), out=dec.next_ids)
        return new

    def train_mode(self, on: bool = True) -> None:
        if on:
            self._gen_decoder = None      # the KV cache does not outlive the evaluation
        if self.model is not None:
            self.model.train(on)
        elif on:
            self._eval_model = None       # the whole-model evaluation copy (full sharding) does not outlive the evaluation

    def close(self) -> None:
        self._gen_decoder = None
        self._graphs.clear()
        self._ws.clear()


class Decoder:
    """KV-cached decoding session of a :class:`B200Engine`: the engine's bf16 weight shadow and fp32 small parameters, a
    per-layer cache ``[B, S_max, 2d]`` (k | v, head-major like ``qkv``) and static step buffers.

    :meth:`prefill` runs the engine's own block forward over the right-padded prompts and writes every layer's k | v into
    the cache; :meth:`step` feeds one token per row through LN → QKV GEMM → (clip, qk-LN) → ``kv_write`` (RoPE at the row's
    position) → ``decode_attention`` → out-projection + residual → LN → up + GELU → down + residual, then the final LN and
    the LM head, all with ``M = B``. With ``kernels.cuda_graph`` the step is captured once and replayed: its shapes are
    static and the per-row lengths are read on the device."""

    def __init__(self, eng: B200Engine, batch: int, max_len: int) -> None:
        c, dev = eng.cfg, eng.device
        self.eng, self.B = eng, int(batch)
        if self.B < 1:
            raise ValueError("a decoder needs at least one row")
        self.S_max = min(c.max_seq_len, -(-max(1, int(max_len)) // 128) * 128)
        d, B = c.d_model, self.B
        bf = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=dev)  # noqa: E731
        f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
        self.cache = [bf(B, self.S_max, 2 * d) for _ in range(c.n_layers)]
        self.lengths = [0] * B
        self.meta = torch.zeros(2, B, dtype=torch.int32, device=dev)     # [0] = lengths, [1] = position of the step's token
        self.b_idx = torch.arange(B, dtype=torch.int32, device=dev)
        self.tokens = torch.zeros(B, dtype=torch.int64, device=dev)
        self.next_ids = torch.zeros(B, dtype=torch.int64, device=dev)
        self.h = [bf(B, d), bf(B, d)]
        self.buf = {"ln": bf(B, d), "m": f32(B), "r": f32(B), "qkv": bf(B, 3 * d), "attn": bf(B, d), "hmid": bf(B, d),
                    "z": bf(B, c.expansion_ratio * d), "u": bf(B, c.expansion_ratio * d)}
        if c.qk_ln:
            self.buf.update(qk_pre=bf(B, d), qk_tmp=bf(B, d))
        self.logits = bf(B, c.vocab_size)
        self.n_split = ops.decode_attention_splits(B * c.n_heads, self.S_max)
        self._graph: Any = None

    @torch.no_grad()
    def prefill(self, prompts: list[list[int]]) -> torch.Tensor:
        """Fill the cache with ``prompts`` (one per row, 1..S_max ids); returns the next-token logits ``[B, V]`` of every row."""
        eng, c = self.eng, self.eng.cfg
        if len(prompts) != self.B:
            raise ValueError(f"prefill needs {self.B} prompts, got {len(prompts)}")
        lens = [len(p) for p in prompts]
        if min(lens) < 1 or max(lens) > self.S_max:
            raise ValueError(f"prompt lengths must be within 1..{self.S_max}")
        # right padding to the 128-row attention tiles: every pad key sits after every valid key, so causal attention over
        # the valid positions is unchanged
        S = -(-max(lens) // 128) * 128
        ids = torch.zeros(self.B, S, dtype=torch.int64)
        for r, p in enumerate(prompts):
            ids[r, : len(p)] = torch.tensor(p, dtype=torch.int64)
        ids = ids.to(eng.device)
        ws = eng._workspace(self.B, S, fp8=False)
        ops.embed_fwd(ids.reshape(-1), eng.wte16, eng.wpe16, ws["h"][0], S)
        b_idx = self.b_idx.repeat_interleave(S)
        pos = torch.arange(S, dtype=torch.int32, device=eng.device).repeat(self.B)
        for i in range(c.n_layers):
            eng._block_fwd(i, ws, self.B, S, fp8=False)
            # right after the block: under activation checkpointing the next block overwrites the shared buffers
            ops.kv_write(ws["layers"][i]["qkv"], self.cache[i], b_idx, pos, c.n_heads)
        last = torch.tensor([r * S + n - 1 for r, n in enumerate(lens)], device=eng.device)
        torch.index_select(ws["h"][c.n_layers], 0, last, out=self.h[0])
        self._head(self.h[0])
        self.lengths = lens
        return self.logits

    @torch.no_grad()
    def step(self, tokens: torch.Tensor, active: list[bool] | None = None) -> torch.Tensor:
        """Append ``tokens [B]`` (device int64) at each row's next position; returns the next-token logits ``[B, V]``.
        Rows with ``active[r] = False`` do not advance: their cache is left to be overwritten and their logits are unused."""
        for r in range(self.B):
            if active is None or active[r]:
                if self.lengths[r] >= self.S_max:
                    raise ValueError(f"row {r} is full ({self.S_max} positions)")
                self.lengths[r] += 1
        self.meta.copy_(torch.tensor([self.lengths, [n - 1 for n in self.lengths]], dtype=torch.int32))
        self.tokens.copy_(tokens)
        if not self.eng.use_graph:
            self._step_body()
        else:
            if self._graph is None:
                self._capture()
            self._graph.replay()
        return self.logits

    def _capture(self) -> None:
        side = torch.cuda.Stream(self.eng.device)
        side.wait_stream(torch.cuda.current_stream(self.eng.device))
        with torch.cuda.stream(side):
            self._step_body()        # warm-up: the same step the replay below recomputes
        torch.cuda.current_stream(self.eng.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._step_body()
        self._graph = graph

    def _head(self, h: torch.Tensor) -> None:
        eng, c, bf = self.eng, self.eng.cfg, self.buf
        ops.layernorm_fwd(h, eng.gf, eng.bf, bf["ln"], bf["m"], bf["r"], c.norm_eps)
        ops.gemm(bf["ln"], eng.wte16, self.logits)

    def _step_body(self) -> None:
        eng, c, bf = self.eng, self.eng.cfg, self.buf
        lengths, pos = self.meta[0], self.meta[1]
        ops.embed_at(self.tokens, pos, eng.wte16, eng.wpe16, self.h[0])
        scale = 1.0 / math.sqrt(c.d_head)
        for i, w in enumerate(eng.layers):
            h, h_next = self.h[i % 2], self.h[(i + 1) % 2]
            ops.layernorm_fwd(h, w.g1, w.b1, bf["ln"], bf["m"], bf["r"], c.norm_eps)
            ops.linear_fwd(bf["ln"], w.wqkv, w.bqkv, bf["qkv"])
            if c.clip_qkv:
                bf["qkv"].clamp_(-c.clip_qkv, c.clip_qkv)
            if c.qk_ln:
                qkv3 = bf["qkv"].view(-1, 3, c.d_model)
                for j in range(2):
                    bf["qk_pre"].copy_(qkv3[:, j])
                    ops.layernorm_fwd(bf["qk_pre"], w.qk_g[j], w.qk_b[j], bf["qk_tmp"], bf["m"], bf["r"], c.norm_eps)
                    qkv3[:, j].copy_(bf["qk_tmp"])
            ops.kv_write(bf["qkv"], self.cache[i], self.b_idx, pos, c.n_heads, rope=eng.rope)
            ops.decode_attention(bf["qkv"], self.cache[i], lengths, eng.alibi, scale, c.n_heads, bf["attn"], n_split=self.n_split)
            ops.linear_fwd(bf["attn"], w.wo, w.bo, bf["hmid"], residual=h)
            ops.layernorm_fwd(bf["hmid"], w.g2, w.b2, bf["ln"], bf["m"], bf["r"], c.norm_eps)
            ops.linear_gelu_grad_fwd(bf["ln"], w.wup, w.bup, bf["z"], bf["u"])
            ops.linear_fwd(bf["u"], w.wdown, w.bdown, h_next, residual=bf["hmid"])
        self._head(self.h[c.n_layers % 2])
