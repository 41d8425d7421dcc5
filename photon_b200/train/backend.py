"""Compute backends behind the Trainer.

``TorchBackend`` = MPT in stock PyTorch ops with autograd (CPU path, numerics
oracle, and the "reference-equivalent" GPU baseline: cuBLAS GEMMs, SDPA/FA2
attention, ATen LN/GELU/CE under ``torch.autocast`` — what the reference gets
from Composer + llm-foundry, ref: photon/clients/trainer_utils.py:1615-1719).

``photon_b200.models.engine.B200Engine`` implements the same protocol with the
hand-written sm_100a kernels and an explicit (autograd-free) backward; the
Trainer does not care which one it drives.

Protocol
--------
``flat``                      :class:`FlatParams` (fp32 master params + grads)
``fwd_bwd(ids, denom, scale)``  accumulate d(Σ token-loss · scale / denom) into ``flat.grads``;
                              returns device scalars ``(loss_sum, n_tokens)``
``eval_stats(ids)``           ``{"loss_sum","n_tokens","n_correct"[, "unigram_loss_sum"]}``
``params_updated()``          hook after optimizer / parameter load (refresh shadows)
``generate(prompts, max_new_tokens, eos_id, stop)``  batched greedy decoding (the engine: with a KV cache)
"""
from __future__ import annotations

import contextlib
from typing import Any, Callable

import torch
import torch.nn.functional as F

from photon_b200.models.mpt import MPTConfig, MPTForCausalLM, shift_labels
from photon_b200.utils.flat import FlatParams


def autocast_ctx(device: torch.device, precision: str) -> Any:
    if precision == "fp32":
        return contextlib.nullcontext()
    dt = torch.float16 if precision == "amp_fp16" else torch.bfloat16
    return torch.autocast(device_type=device.type, dtype=dt)


def apply_freeze(model: torch.nn.Module, frozen: list[str] | None, unfrozen: list[str] | None) -> list[str]:
    """Exact-name freeze lists (ref: photon/utils.py:322-387). Frozen tensors drop out of
    the exchanged parameter list because only ``requires_grad`` tensors are flat-packed."""
    if frozen and unfrozen:
        raise ValueError("frozen_layers and unfrozen_layers are mutually exclusive")
    names = [n for n, _ in model.named_parameters()]
    touched = []
    if frozen:
        missing = [n for n in frozen if n not in names]
        if missing:
            raise KeyError(f"frozen_layers not in model: {missing[:4]}")
        for n, p in model.named_parameters():
            if n in frozen:
                p.requires_grad_(False)
                touched.append(n)
    elif unfrozen:
        missing = [n for n in unfrozen if n not in names]
        if missing:
            raise KeyError(f"unfrozen_layers not in model: {missing[:4]}")
        for n, p in model.named_parameters():
            if n not in unfrozen:
                p.requires_grad_(False)
                touched.append(n)
    return touched


class TorchBackend:
    kind = "torch"

    def __init__(self, cfg: MPTConfig, device: torch.device | str = "cpu", precision: str = "amp_bf16",
                 seed: int | None = 17, frozen_layers: list[str] | None = None,
                 unfrozen_layers: list[str] | None = None, unigram_log_probs: torch.Tensor | None = None,
                 grads_storage: torch.Tensor | None = None, activation_checkpointing: bool = False,
                 params_storage: torch.Tensor | None = None, shadow_storage: torch.Tensor | None = None) -> None:
        self.cfg = cfg
        self.device = torch.device(device)
        self.precision = precision
        self.model = MPTForCausalLM(cfg, device=self.device, seed=seed)
        self.model.activation_checkpointing = bool(activation_checkpointing)
        self.frozen = apply_freeze(self.model, frozen_layers, unfrozen_layers)
        self.flat = FlatParams(self.model, device=self.device, params_storage=params_storage, grads_storage=grads_storage)
        self.bf16_params = shadow_storage   # only kept so a fused NVLink step has a plane to write (autocast casts on the fly)
        self.fp8_layers: list[str] = []
        if precision == "amp_fp8":          # E4M3 forward / E5M2 backward GEMM operands with delayed scaling, bf16 elsewhere
            from photon_b200.train.fp8 import enable_fp8

            self.fp8_layers = enable_fp8(self.model)
        self.unigram_log_probs = unigram_log_probs.to(self.device) if unigram_log_probs is not None else None
        self.collect_activation_stats = False
        self.activation_stats: dict[str, float] = {}
        self.launches_per_microbatch = 0  # stock torch ops are not "our" kernels

    # -- training ---------------------------------------------------------------------
    def fwd_bwd(self, ids: torch.Tensor, denom: float, scale: float = 1.0) -> tuple[torch.Tensor, torch.Tensor]:
        with autocast_ctx(self.device, self.precision):
            loss_sum, n = self.model.loss(ids, reduction="sum")
        (loss_sum * (scale / denom)).backward()
        if self.collect_activation_stats:
            self._act_stats(ids)
        return loss_sum.detach(), n

    @torch.no_grad()
    def _act_stats(self, ids: torch.Tensor) -> None:
        t = self.model.transformer
        x = t.wte(ids[:1])
        if self.cfg.learned_pos_emb:
            x = x + t.wpe(torch.arange(ids.shape[1], device=ids.device))[None]
        rope, alibi = self.model._aux(ids.shape[1], ids.device)  # noqa: SLF001
        for i, blk in enumerate(t.blocks):
            x = blk(x, rope, alibi)
            self.activation_stats[f"l2_norm/block_{i}"] = float(x.float().norm(dim=-1).mean())
            self.activation_stats[f"max/block_{i}"] = float(x.abs().max())

    # -- evaluation -------------------------------------------------------------------
    @torch.no_grad()
    def eval_stats(self, ids: torch.Tensor) -> dict[str, torch.Tensor]:
        with autocast_ctx(self.device, self.precision):
            logits = self.model(ids)
        targets = shift_labels(ids)
        lf = logits.float().view(-1, logits.shape[-1])
        tf = targets.view(-1)
        out = {"loss_sum": F.cross_entropy(lf, tf, ignore_index=-100, reduction="sum"),
               "n_tokens": (tf != -100).sum(),
               "n_correct": ((lf.argmax(-1) == tf) & (tf != -100)).sum()}
        if self.unigram_log_probs is not None:
            from photon_b200.metrics.language import unigram_loss_sum

            out["unigram_loss_sum"] = unigram_loss_sum(tf, self.unigram_log_probs)
        return out

    @torch.no_grad()
    def logits(self, ids: torch.Tensor) -> torch.Tensor:
        """``[B,S] → [B,S,V]`` next-token logits (the in-context-learning evaluator's view of the model)."""
        with autocast_ctx(self.device, self.precision):
            return self.model(ids.to(self.device))

    @torch.no_grad()
    def generate(self, prompts: list[list[int]], max_new_tokens: int, eos_id: int | None = None,
                 stop: Callable[[int, list[int]], bool] | None = None) -> list[list[int]]:
        """Greedy continuation of every prompt by batched recompute (no cache); returns the new ids of each row.

        Each step runs the unfinished rows' windows (the last ``max_seq_len`` ids) right-padded in one batch and takes every
        row's argmax at its last valid position; causal attention keeps the padding out of the valid positions. A row ends
        at ``eos_id`` (not included), when ``stop(row, new_ids)`` returns True, or after ``max_new_tokens``."""
        msl = self.cfg.max_seq_len
        ctx = [list(p) for p in prompts]
        new: list[list[int]] = [[] for _ in prompts]
        done = [False] * len(prompts)
        for _ in range(max_new_tokens):
            rows = [r for r in range(len(prompts)) if not done[r]]
            if not rows:
                break
            wins = [ctx[r][-msl:] for r in rows]
            ids = torch.zeros(len(rows), max(len(w) for w in wins), dtype=torch.long)
            for j, w in enumerate(wins):
                ids[j, : len(w)] = torch.tensor(w, dtype=torch.long)
            logits = self.logits(ids)
            last = torch.tensor([len(w) - 1 for w in wins], device=logits.device)
            nxt = logits[torch.arange(len(rows), device=logits.device), last].float().argmax(-1).tolist()
            for r, t in zip(rows, nxt):
                if eos_id is not None and t == eos_id:
                    done[r] = True
                    continue
                ctx[r].append(t)
                new[r].append(t)
                if stop is not None and stop(r, new[r]):
                    done[r] = True
        return new

    def params_updated(self) -> None:
        pass

    def train_mode(self, on: bool = True) -> None:
        self.model.train(on)

    def close(self) -> None:
        pass


def build_backend(model_cfg: MPTConfig, device: torch.device, precision: str, kernels: dict[str, Any] | None = None,
                  **kw: Any) -> Any:
    """Pick the compute backend. On a CUDA device the B200 engine is THE path (and fails
    loudly if its extension is missing); ``kernels.gemm: torch`` etc. selects the stock
    PyTorch baseline explicitly; CPU always uses stock PyTorch."""
    kernels = dict(kernels or {})
    modes = [kernels.get(k, "auto") for k in ("gemm", "attention", "norm", "loss", "optimizer")]
    want_engine = device.type == "cuda" and not all(m == "torch" for m in modes)
    if any(m == "b200" for m in modes) and device.type != "cuda":
        raise RuntimeError("kernels.*=b200 requires a CUDA (sm_100a) device")
    if want_engine:
        unsupported = []
        if precision not in ("amp_bf16", "amp_fp8"):
            unsupported.append(f"precision={precision}")
        if kw.get("frozen_layers") or kw.get("unfrozen_layers"):
            unsupported.append("frozen/unfrozen layers")
        if unsupported:
            print(f"[backend] {', '.join(unsupported)} not covered by the sm_100a engine -> stock PyTorch backend "
                  "(explicit, logged; set kernels.*=torch to silence)", flush=True)
            kw.pop("zero3", None)
            return TorchBackend(model_cfg, device=device, precision=precision, **kw)
        from photon_b200.models.engine import B200Engine

        return B200Engine(model_cfg, device=device, precision=precision, kernels=kernels, **kw)
    if kw.pop("zero3", None) is not None:
        raise RuntimeError("full parameter sharding (NvlZero3Comm) needs the sm_100a engine on a CUDA device")
    return TorchBackend(model_cfg, device=device, precision=precision, **kw)
