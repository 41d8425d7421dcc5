"""Python face of the hand-written sm_100a kernels (``photon_b200._C``).

Every function here launches OUR kernels; nothing silently falls back to a
PyTorch op.  If the extension is missing on a machine that has a CUDA device
the import error is raised loudly (the driver records which ``.so`` files the
GPU tests actually loaded).  On CPU-only machines the extension still imports
(it is cross-compiled) but these wrappers are never called.
"""
from __future__ import annotations

import math
from typing import Any

import torch

_EXT: Any = None


def ext() -> Any:
    """Load (and cache) the in-tree extension; raise loudly if it is absent."""
    global _EXT
    if _EXT is None:
        try:
            from photon_b200 import _C  # type: ignore[attr-defined]
        except ImportError as e:  # pragma: no cover - depends on the box
            raise ImportError(
                "photon_b200._C (sm_100a kernels) is not built. Run `python -m photon_b200.build` "
                "(or __graft_entry__.build()) — refusing to fall back to PyTorch ops on the GPU path.") from e
        _EXT = _C
    return _EXT


def have_ext() -> bool:
    try:
        ext()
        return True
    except ImportError:
        return False


def launch_count() -> int:
    return int(ext().launch_count())


def reset_launch_count() -> None:
    ext().reset_launch_count()


def add_launch_count(n: int) -> None:
    """Account for kernels replayed from a captured CUDA graph (they never pass through the bindings)."""
    ext().add_launch_count(int(n))


# --------------------------------------------------------------------------------- GEMM
EPI_BF16, EPI_RESIDUAL, EPI_GELU_DUAL, EPI_DGELU, EPI_F32, EPI_GELU_GRAD, EPI_MUL, EPI_GELU_GRAD_Q8 = 0, 1, 2, 3, 4, 5, 6, 7
E4M3, E5M2 = 0, 1          # operand formats of the kind::f8f6f4 GEMMs
FP8_MAX = (448.0, 57344.0)


def gemm(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False,
         epi: int = EPI_BF16, bias: torch.Tensor | None = None, aux: torch.Tensor | None = None,
         out2: torch.Tensor | None = None, accumulate: bool = False, alpha: float = 1.0, cluster: int = 0) -> torch.Tensor:
    """``out[M,N] = epilogue(alpha * A @ B^T)`` on tcgen05 tensor cores.

    ``a``: ``[M,K]`` (K-major) or ``[K,M]`` when ``a_mn``; ``b``: ``[N,K]`` or ``[K,N]`` when ``b_mn``."""
    ext().gemm(a, b, out, int(a_mn), int(b_mn), int(epi), bias, aux, out2, bool(accumulate), float(alpha), int(cluster))
    return out


def linear_fwd(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None, out: torch.Tensor,
               residual: torch.Tensor | None = None) -> torch.Tensor:
    """y = x @ w^T + bias (+ residual) — x [T,K], w [N,K] (bf16), bias fp32."""
    return gemm(x, w, out, epi=EPI_RESIDUAL if residual is not None else EPI_BF16, bias=bias, aux=residual)


def linear_gelu_fwd(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None, pre: torch.Tensor,
                    act: torch.Tensor) -> torch.Tensor:
    """pre = x @ w^T + bias ; act = gelu(pre) — both written by the same epilogue."""
    return gemm(x, w, act, epi=EPI_GELU_DUAL, bias=bias, out2=pre)


def linear_gelu_grad_fwd(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None, dact: torch.Tensor,
                         act: torch.Tensor) -> torch.Tensor:
    """z = x @ w^T + bias ; act = gelu(z) ; dact = gelu'(z) — the derivative is what the backward needs, so it is saved
    INSTEAD of z and the dgrad epilogue becomes a plain multiply (no erf / exp in the backward)."""
    return gemm(x, w, act, epi=EPI_GELU_GRAD, bias=bias, out2=dact)


def linear_dgrad(dy: torch.Tensor, w: torch.Tensor, dx: torch.Tensor, gelu_pre: torch.Tensor | None = None,
                 mul: torch.Tensor | None = None) -> torch.Tensor:
    """dx = dy @ w  (w stored [N,K] → consumed MN-major, no transpose); optional ``* gelu'(pre)`` (pre-activation given)
    or ``* mul`` (saved derivative given)."""
    if mul is not None:
        return gemm(dy, w, dx, b_mn=True, epi=EPI_MUL, aux=mul)
    return gemm(dy, w, dx, b_mn=True, epi=EPI_DGELU if gelu_pre is not None else EPI_BF16, aux=gelu_pre)


def linear_wgrad(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, accumulate: bool = True, alpha: float = 1.0) -> torch.Tensor:
    """dw[N,K] (+)= dy^T @ x in fp32 (both operands consumed MN-major; TMA reduce-add when accumulating)."""
    return gemm(dy, x, dw, a_mn=True, b_mn=True, epi=EPI_F32, accumulate=accumulate, alpha=alpha)


# ------------------------------------------------------------------------------ fp8 GEMM
def gemm_fp8(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, meta: torch.Tensor, role_a: int, role_b: int, *,
             a_mn: bool = False, b_mn: bool = False, epi: int = EPI_BF16, a_fmt: int = E4M3, b_fmt: int = E4M3,
             bias: torch.Tensor | None = None, aux: torch.Tensor | None = None, out2: torch.Tensor | None = None,
             accumulate: bool = False, alpha: float = 1.0, cluster: int = 0, out8: torch.Tensor | None = None,
             role_out: int = -1) -> torch.Tensor:
    """``out = epilogue(alpha / (scale[role_a] * scale[role_b]) * A8 @ B8^T)`` — 1-byte operands (E4M3 / E5M2 per operand) on
    ``tcgen05.mma kind::f8f6f4``, fp32 accumulation. ``meta`` = float32 ``[3, n_roles]`` (scale, 1/scale, amax) on the device;
    the de-scales are read by the kernel, so nothing here touches the host. ``EPI_GELU_GRAD_Q8`` writes ``out8`` (E4M3,
    scaled by ``scale[role_out]``, amax recorded) and ``out2`` = gelu'; ``out`` is then unused (pass ``out2``)."""
    ext().gemm_fp8(a, b, out, int(a_mn), int(b_mn), int(epi), int(a_fmt), int(b_fmt), meta, int(role_a), int(role_b), bias, aux, out2,
                   bool(accumulate), float(alpha), int(cluster), out8, int(role_out))
    return out


def mx_quantize(x: torch.Tensor, row_blocks: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
    """bf16 ``[R,K]`` → (E4M3 ``[R,K]`` uint8, E8M0 scale atoms ``[K/128, row_blocks, 512]`` uint8): OCP MXFP8, one power-of-two scale
    per 32 consecutive K elements of a row, stored in the layout ``tcgen05.mma ... block_scale`` reads from TMEM."""
    q, sf = ext().mx_quantize(x, int(row_blocks))
    return q, sf


def gemm_mxfp8(a8: torch.Tensor, b8: torch.Tensor, out: torch.Tensor, sfa: torch.Tensor, sfb: torch.Tensor,
               bias: torch.Tensor | None = None) -> torch.Tensor:
    """``out[M,N] = (A ⊙ SFA) @ (B ⊙ SFB)^T (+ bias)`` with the block scales applied inside the tensor core
    (``tcgen05.mma kind::mxf8f6f4.block_scale``). ``sfb`` needs ``2·ceil(N/256)`` row blocks (``mx_quantize(w, 2 * ceil(N/256))``)."""
    ext().gemm_mxfp8(a8, b8, out, sfa, sfb, bias)
    return out


def layernorm_fwd_q8(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor | None, y8: torch.Tensor, mean: torch.Tensor,
                     rstd: torch.Tensor, eps: float, meta: torch.Tensor, role: int) -> torch.Tensor:
    """LayerNorm whose only output is the E4M3 tensor the next GEMM reads (scaled by ``scale[role]``, ``amax[role]`` updated)."""
    ext().layernorm_fwd_q8(x, gamma, beta, y8, mean, rstd, float(eps), meta, int(role))
    return y8


def colsum_quant(dy: torch.Tensor, out_sum: torch.Tensor | None, y8: torch.Tensor | None, fmt: int = E5M2,
                 meta: torch.Tensor | None = None, role: int = -1) -> None:
    """One read of ``dy`` [T,N]: ``out_sum[j] += Σ_t dy[t,j]`` (bias gradient) and ``y8 = fp8(dy * scale[role])``."""
    ext().colsum_quant(dy, out_sum, y8, int(fmt), meta, int(role))


def fp8_quantize_segments(src_bf16: torch.Tensor, dst8: torch.Tensor, seg: torch.Tensor, meta: torch.Tensor, role0: int) -> None:
    """Per-tensor current scaling of ``seg`` = int64 [n,2] (offset, numel) slices of a flat bf16 plane → E4M3 in ``dst8``."""
    ext().fp8_quantize_segments(src_bf16, dst8, seg, meta, int(role0))


def fp8_update_scales(meta: torch.Tensor, hist: torch.Tensor, fmax: torch.Tensor, pos: torch.Tensor, n: int, margin_mult: float = 1.0) -> None:
    """Delayed scaling for roles [0, n): amax → history ring → scale for the next cast; amax reset."""
    ext().fp8_update_scales(meta, hist, fmax, pos, int(n), float(margin_mult))


# ---------------------------------------------------------------------------- fused ops
def embed_fwd(ids: torch.Tensor, wte: torch.Tensor, wpe: torch.Tensor | None, out: torch.Tensor, seq_len: int) -> torch.Tensor:
    ext().embed_fwd(ids, wte, wpe, out, int(seq_len))
    return out


def embed_bwd(ids: torch.Tensor, dh: torch.Tensor, dwte: torch.Tensor, dwpe: torch.Tensor | None, seq_len: int) -> None:
    ext().embed_bwd(ids, dh, dwte, dwpe, int(seq_len))


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor | None, y: torch.Tensor, mean: torch.Tensor,
                  rstd: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    ext().layernorm_fwd(x, gamma, beta, y, mean, rstd, float(eps))
    return y


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, gamma: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor,
                  dres: torch.Tensor | None, dx: torch.Tensor, dgamma: torch.Tensor | None, dbeta: torch.Tensor | None) -> torch.Tensor:
    ext().layernorm_bwd(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta)
    return dx


def col_sum(dy: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[j] += Σ_t dy[t,j] (bias gradients)."""
    ext().col_sum(dy, out)
    return out


def cross_entropy(logits: torch.Tensor, targets: torch.Tensor, grad_scale: float, write_grad: bool, stats: torch.Tensor,
                  row_lse: torch.Tensor | None = None, unigram_logp: torch.Tensor | None = None) -> None:
    """In place: logits → dlogits (when ``write_grad``); stats[0..3] += (Σloss, #valid, #correct, Σunigram)."""
    ext().cross_entropy(logits, targets, float(grad_scale), bool(write_grad), stats, row_lse, unigram_logp)


_NORM_SCRATCH: dict[int, tuple[torch.Tensor, torch.Tensor]] = {}


def flat_l2_norm(x: torch.Tensor) -> torch.Tensor:
    """‖x‖₂ of a flat fp32 buffer as a 0-dim device tensor (no host sync)."""
    key = x.device.index or 0
    if key not in _NORM_SCRATCH:
        _NORM_SCRATCH[key] = (torch.zeros(1, dtype=torch.float64, device=x.device), torch.zeros(1, dtype=torch.float32, device=x.device))
    scratch, out = _NORM_SCRATCH[key]
    ext().flat_l2_norm(x, scratch, out)
    return out[0]


def axpby_(acc: torch.Tensor, x: torch.Tensor, a: float, b: float) -> torch.Tensor:
    ext().axpby(acc, x, float(a), float(b))
    return acc


def cast_bf16(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    ext().cast_bf16(src, dst)
    return dst


_KIND = {"adopt": 0, "decoupled_adamw": 1, "sgd": 2}


def optimizer_hyper(opt: Any, lr: float) -> dict[str, Any]:
    """Per-step scalar arguments of the fused optimizer kernels for a :class:`FlatOptimizer` at learning rate ``lr``."""
    kind = _KIND[opt.name]
    first = kind == 0 and opt.step_count == 0
    decay, clip, step_size, inv_sqrt_bc2 = 1.0, float("inf"), 0.0, 1.0
    if kind == 0:
        if opt.weight_decay and getattr(opt, "decouple", True):
            decay = 1.0 - lr * opt.weight_decay
        if opt.clip_exp is not None and not first:
            clip = float(opt.step_count) ** opt.clip_exp
    elif kind == 1:
        t = opt.step_count + 1
        decay = 1.0 - (lr / opt.initial_lr) * opt.weight_decay if opt.weight_decay else 1.0
        step_size = lr / (1.0 - opt.beta1 ** t)
        inv_sqrt_bc2 = 1.0 / math.sqrt(1.0 - opt.beta2 ** t)
    else:
        decay = 1.0 - lr * opt.weight_decay if opt.weight_decay else 1.0
    return dict(kind=kind, first=first, lr=float(lr), beta1=opt.beta1, beta2=opt.beta2, eps=opt.eps, decay=float(decay),
                clip=float(clip), step_size=float(step_size), inv_sqrt_bc2=float(inv_sqrt_bc2))


def fused_optimizer_step(opt: Any, lr: float, grad_mult: torch.Tensor | float | None) -> None:
    """One fused multi-tensor step for a :class:`photon_b200.train.optim.FlatOptimizer`."""
    flat = opt.flat
    h = optimizer_hyper(opt, lr)
    gm = None
    if grad_mult is not None:
        gm = grad_mult if torch.is_tensor(grad_mult) else torch.tensor(float(grad_mult), device=flat.params.device)
        gm = gm.to(torch.float32).reshape(1)
    params, grads, shadow = opt.local_views()   # the whole flat buffer, or this rank's slice when the state is sharded
    ext().fused_optimizer(params, grads, opt.exp_avg, opt.exp_avg_sq, shadow, h["kind"], h["first"], h["lr"],
                          h["beta1"], h["beta2"], h["eps"], h["decay"], h["clip"], h["step_size"], h["inv_sqrt_bc2"], gm)


# ---------------------------------------------------------------------------- attention
def attention_fwd(qkv: torch.Tensor, out: torch.Tensor, lse: torch.Tensor, n_heads: int, scale: float, causal: bool = True,
                  alibi_slopes: torch.Tensor | None = None) -> None:
    """``alibi_slopes``: optional fp32 [n_heads]; adds ``slope_h * (key - query)`` to the scores (MPT ``attn_config.alibi``)."""
    ext().attention_fwd(qkv, out, lse, int(n_heads), float(scale), bool(causal), alibi_slopes)


def attention_bwd(qkv: torch.Tensor, out: torch.Tensor, dout: torch.Tensor, lse: torch.Tensor, dqkv: torch.Tensor,
                  delta: torch.Tensor, n_heads: int, scale: float, causal: bool = True,
                  alibi_slopes: torch.Tensor | None = None) -> None:
    ext().attention_bwd(qkv, out, dout, lse, dqkv, delta, int(n_heads), float(scale), bool(causal), alibi_slopes)


def rope_(qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, n_heads: int, inverse: bool = False) -> torch.Tensor:
    """In-place rotary embedding (rotate-half) of the q and k thirds of ``qkv`` [B,S,3d]; ``inverse`` applies the
    transposed rotation (what the gradients of q and k need)."""
    ext().rope(qkv, cos, sin, int(n_heads), bool(inverse))
    return qkv


# ---------------------------------------------------------------------------- KV-cached decoding
def embed_at(ids: torch.Tensor, pos: torch.Tensor, wte: torch.Tensor, wpe: torch.Tensor | None, out: torch.Tensor) -> torch.Tensor:
    """``out[t] = wte[ids[t]] (+ wpe[pos[t]])``: int64 ids, int32 explicit positions (``embed_fwd`` derives them as ``t % S``).
    Out-of-range ids are clamped as in ``embed_fwd``."""
    ext().embed_at(ids, pos, wte, wpe, out)
    return out


def decode_attention_splits(bh: int, s_max: int) -> int:
    """The key-split count :func:`decode_attention` picks for ``bh`` (row, head) pairs over an ``s_max`` cache."""
    return int(ext().decode_attention_splits(int(bh), int(s_max)))


def decode_attention(q: torch.Tensor, kv: torch.Tensor, lengths: torch.Tensor, alibi_slopes: torch.Tensor | None, scale: float,
                     n_heads: int, out: torch.Tensor, lse: torch.Tensor | None = None, n_split: int = 0) -> torch.Tensor:
    """One query per row against a ragged KV cache (split-KV flash-decoding).

    ``q``: bf16 rows ``[B, >= d]`` (the q third of the step's ``qkv [B, 3d]`` is ``qkv`` itself: only the first ``d`` columns
    are read); ``kv``: bf16 ``[B, S_max, 2d]`` (k | v, head-major); ``lengths``: int32 ``[B]`` valid keys per row on the device,
    the current token included; ``alibi_slopes``: optional fp32 ``[H]`` (adds ``slope_h * (key - (length - 1))``). Keys at or
    beyond ``length`` are never read. ``out``: bf16 ``[B, d]``; ``lse``: optional fp32 ``[B, H]`` (natural log).
    ``n_split`` = 0 picks :func:`decode_attention_splits`; it depends only on shapes, so a captured step stays valid."""
    ext().decode_attention(q, kv, lengths, alibi_slopes, float(scale), int(n_heads), int(n_split), out, lse)
    return out


def kv_write(qkv: torch.Tensor, cache: torch.Tensor, b_idx: torch.Tensor, pos: torch.Tensor, n_heads: int,
             rope: tuple[torch.Tensor, torch.Tensor] | None = None) -> None:
    """``cache[b_idx[t], pos[t]] = k | v`` of ``qkv [T, 3d]`` row ``t`` (int32 coordinates). With ``rope`` = (cos, sin) the
    row's q and k are first rotated in place at ``pos[t]``, bit-identical to :func:`rope_` at that position."""
    cos, sin = rope if rope is not None else (None, None)
    ext().kv_write(qkv, cache, b_idx, pos, cos, sin, int(n_heads))


def argmax_rows(logits: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """int64 ``[R]`` index of the largest value of every bf16 row of ``logits [R, V]``; ties go to the lowest index."""
    if out is None:
        out = torch.empty(logits.shape[0], dtype=torch.int64, device=logits.device)
    ext().argmax_rows(logits, out)
    return out
