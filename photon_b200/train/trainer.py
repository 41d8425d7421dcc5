"""Trainer: the local-training engine a federated client (or the centralised
entry point) drives.

Replaces the Composer ``Trainer`` the reference wraps (ref:
photon/clients/trainer_utils.py:1675-1719 construction; photon/clients/
llm_client_functions.py:206-208 ``trainer.fit(duration=local_steps)``;
photon/centralised_train.py:151-153).  Semantics kept:

* ``fit(duration=X)`` trains X *more* from the current timestamp;
* a batch is split into microbatches of ``device_train_microbatch_size``
  (``auto`` = halve on CUDA OOM, ranks agree on the min);
* DDP "forced sync": every microbatch accumulates locally, ONE gradient
  all-reduce after the last one (ref: trainer_utils.py:1714) — here a single
  fused NVLink kernel on the flat grad buffer instead of 148 NCCL calls;
* algorithms → grad clipping; optimizer step; scheduler stepped every batch
  and indexed by the global batch counter;
* checkpoints ``ep{E}-ba{B}-rank{R}.pt`` + ``latest-rank{R}.pt`` with
  ``save_num_checkpoints_to_keep`` and glob ``load_ignore_keys``.

B200-first differences: one flat fp32 parameter/gradient/moment buffer, H2D
copies on a side stream from pinned memory, device-side loss/clip scalars (no
per-step host sync besides the configurable metric read-back).
"""
from __future__ import annotations

import fnmatch
import os
import time
from dataclasses import dataclass, field
from pathlib import Path
from typing import Any, Iterable, Iterator

import torch
import torch.distributed as dist

from photon_b200.metrics.language import Metric, build_metrics, sync_metrics, unigram_loss_sum
from photon_b200.models.mpt import MPTConfig, shift_labels
from photon_b200.train.backend import build_backend
from photon_b200.train.callbacks import Callback, InMemoryLogger, Logger
from photon_b200.train.optim import FlatOptimizer, build_optimizer, clip_coefficient
from photon_b200.train.schedulers import Scheduler, build_scheduler
from photon_b200.train.timestamp import Time, Timestamp
from photon_b200.utils.flat import FlatParams


@dataclass
class TrainerState:
    backend: Any
    flat: FlatParams
    optimizer: FlatOptimizer
    scheduler: Scheduler
    timestamp: Timestamp = field(default_factory=Timestamp)
    eval_timestamp: Timestamp = field(default_factory=Timestamp)
    train_metrics: dict[str, Metric] = field(default_factory=dict)
    eval_metrics: dict[str, dict[str, Metric]] = field(default_factory=dict)
    run_name: str = "run"

    @property
    def model(self) -> Any:
        return getattr(self.backend, "model", self.backend)

    @property
    def train_metric_values(self) -> dict[str, float]:
        return {k: m.compute() for k, m in self.train_metrics.items() if m.count}

    @property
    def eval_metric_values(self) -> dict[str, float]:
        out: dict[str, float] = {}
        for label, ms in self.eval_metrics.items():
            for k, m in ms.items():
                if m.count:
                    out[f"{label}/{k}" if label else k] = m.compute()
        return out


class GradScaler:
    """Dynamic loss scaling for ``amp_fp16`` (growth 2× / 2000 good steps, back-off ½)."""

    def __init__(self, init: float = 2.0 ** 16, growth_interval: int = 2000) -> None:
        self.scale, self.growth_interval, self._good = float(init), growth_interval, 0

    def update(self, found_inf: bool) -> None:
        if found_inf:
            self.scale, self._good = max(self.scale * 0.5, 1.0), 0
        else:
            self._good += 1
            if self._good % self.growth_interval == 0:
                self.scale *= 2.0


def shard_bounds(total: int, world_size: int, align: int = 256) -> list[tuple[int, int]]:
    """Contiguous, ``align``-element-aligned [lo, hi) slices of the flat index space, one per rank."""
    per = -(-total // world_size)
    per = -(-per // align) * align
    return [(min(total, r * per), min(total, (r + 1) * per)) for r in range(world_size)]


def _is_oom(e: BaseException) -> bool:
    return isinstance(e, torch.cuda.OutOfMemoryError) or "out of memory" in str(e).lower()


class Trainer:
    def __init__(self, model_cfg: MPTConfig | dict[str, Any], *, optimizer_cfg: dict[str, Any],
                 scheduler_cfg: dict[str, Any] | None = None, train_loader: Any = None,
                 eval_loaders: dict[str, Any] | None = None, global_train_batch_size: int = 8,
                 device_train_microbatch_size: int | str = "auto", device_eval_batch_size: int | None = None,
                 precision: str = "amp_bf16", max_duration: str | int | None = None,
                 grad_clip_norm: float | None = None, callbacks: Iterable[Callback] = (),
                 loggers: Iterable[Logger] = (), save_folder: str | None = None, save_interval: str | int | None = None,
                 save_num_checkpoints_to_keep: int = -1, save_overwrite: bool = True,
                 eval_interval: str | int | None = None, eval_subset_num_batches: int = -1,
                 device: torch.device | str | None = None, rank: int = 0, world_size: int = 1,
                 process_group: Any = None, grad_comm: Any = None, kernels: dict[str, Any] | None = None,
                 seed: int = 17, run_name: str = "run", use_unigram_metrics: bool = False,
                 unigram_log_probs: torch.Tensor | None = None, frozen_layers: list[str] | None = None,
                 unfrozen_layers: list[str] | None = None, metric_sync_interval: int = 1,
                 backend: Any = None, shard_optimizer_state: bool = False, activation_checkpointing: bool = False,
                 device_eval_microbatch_size: int | str | None = None, grad_clip_value: float | None = None,
                 save_filename: str | None = None, save_latest_filename: str | None = None, save_weights_only: bool = False,
                 save_ignore_keys: Iterable[str] | None = None, train_subset_num_batches: int = -1) -> None:
        self.model_cfg = model_cfg if isinstance(model_cfg, MPTConfig) else MPTConfig.from_model_cfg(model_cfg)
        self.device = torch.device(device) if device is not None else torch.device(
            "cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        self.rank, self.world_size, self.process_group = int(rank), int(world_size), process_group
        self.precision = precision
        if global_train_batch_size % self.world_size:
            raise ValueError(f"global_train_batch_size={global_train_batch_size} not divisible by world_size={world_size}")
        self.global_batch = int(global_train_batch_size)
        self.device_batch = self.global_batch // self.world_size
        self.microbatch = device_train_microbatch_size
        self._auto_mb = self.device_batch if device_train_microbatch_size == "auto" else None
        self.device_eval_batch_size = device_eval_batch_size or self.device_batch
        self.eval_microbatch: int | str | None = device_eval_microbatch_size
        self._eval_mb_auto = device_eval_microbatch_size == "auto"
        self.grad_clip_norm = grad_clip_norm
        self.grad_clip_value = float(grad_clip_value) if grad_clip_value is not None else None   # element-wise clamp (clipping_type: value)
        self.train_loader, self.eval_loaders = train_loader, dict(eval_loaders or {})
        self.callbacks, self.loggers = list(callbacks), list(loggers) or [InMemoryLogger()]
        self.save_folder, self.save_overwrite = save_folder, save_overwrite
        self.save_keep = int(save_num_checkpoints_to_keep)
        self.save_filename = save_filename or "ep{epoch}-ba{batch}-rank{rank}.pt"     # the per-client resume logic parses this default
        self.save_latest_filename = save_latest_filename or "latest-rank{rank}.pt"
        self.save_weights_only, self.save_ignore_keys = bool(save_weights_only), list(save_ignore_keys or [])
        self.eval_subset_num_batches = int(eval_subset_num_batches)
        self.train_subset_num_batches = int(train_subset_num_batches if train_subset_num_batches is not None else -1)
        self.metric_sync_interval = max(1, int(metric_sync_interval))
        self.grad_comm = grad_comm
        self.seed = seed
        self.scaler = GradScaler() if precision == "amp_fp16" else None
        self._pending: dict[str, float] = {}
        self._saved: list[Path] = []
        self._train_iter: Iterator[Any] | None = None
        self.fit_start_batch, self.fit_end_batch = 0, None
        self.closed = False
        self.last_batch_stats: dict[str, float] = {}
        self.icl_suite: Any = None              # callable(logits_fn) -> metrics; set by get_trainer_object from icl_tasks_config
        self.last_icl_metrics: dict[str, float] = {}

        seq = self.model_cfg.max_seq_len
        self.max_duration = Time.parse(max_duration) if max_duration is not None else None
        geom = dict(samples_per_batch=self.global_batch, tokens_per_batch=self.global_batch * seq,
                    batches_per_epoch=len(train_loader) if train_loader is not None and hasattr(train_loader, "__len__") else None)
        self._geom = geom
        self.save_interval = Time.parse(save_interval).to_batches(max_duration=self.max_duration, **geom) if save_interval else None
        self.eval_interval = Time.parse(eval_interval).to_batches(max_duration=self.max_duration, **geom) if eval_interval else None

        be = backend or build_backend(self.model_cfg, self.device, precision, kernels, seed=seed,
                                      frozen_layers=frozen_layers, unfrozen_layers=unfrozen_layers,
                                      unigram_log_probs=unigram_log_probs,
                                      grads_storage=getattr(grad_comm, "grads", None),
                                      params_storage=getattr(grad_comm, "params", None),
                                      shadow_storage=getattr(grad_comm, "shadow", None),
                                      activation_checkpointing=activation_checkpointing,
                                      **({"zero3": grad_comm} if getattr(grad_comm, "zero3", False) else {}))
        if hasattr(grad_comm, "bind_layout"):
            grad_comm.bind_layout(be.flat.layout)
        shadow = getattr(be, "bf16_params", None)
        use_kernel = (kernels or {}).get("optimizer", "auto") != "torch" and self.device.type == "cuda"
        shard_kw: dict[str, Any] = {}
        self.fused_comm_step = (bool(getattr(grad_comm, "fused_step", False)) and self.world_size > 1 and self.scaler is None
                                and grad_clip_value is None)   # the fused NVLink step clips by norm only
        if self.fused_comm_step:
            # reduce-scatter + clip + optimizer + all-gather in one NVLink kernel: moments sharded like the arena
            shard_kw = dict(shard=grad_comm.shard(), shard_bounds=grad_comm.shard_bounds(), group=process_group)
        elif shard_optimizer_state and self.world_size > 1 and not getattr(be.flat, "is_sharded", False):
            # (under full parameter sharding the optimizer already sees nothing but this rank's shard)
            # ZeRO-style state sharding inside the client (the reference's fsdp_config FULL_SHARD / SHARD_GRAD_OP)
            bounds = shard_bounds(be.flat.params.numel(), self.world_size)
            shard_kw = dict(shard=bounds[self.rank], shard_bounds=bounds, group=process_group)
        opt = build_optimizer(optimizer_cfg, be.flat, use_kernel=use_kernel, bf16_shadow=shadow, **shard_kw)
        sched = build_scheduler(scheduler_cfg, max_duration=self.max_duration, **geom)
        self.state = TrainerState(backend=be, flat=be.flat, optimizer=opt, scheduler=sched, run_name=run_name,
                                  train_metrics=build_metrics(use_unigram_metrics),
                                  eval_metrics={lbl: build_metrics(use_unigram_metrics) for lbl in self.eval_loaders})
        self._copy_stream = torch.cuda.Stream(self.device) if self.device.type == "cuda" else None

    # ------------------------------------------------------------------ helpers
    def log(self, metrics: dict[str, float]) -> None:
        self._pending.update(metrics)

    def _flush_logs(self) -> None:
        if self._pending:
            step = self.state.timestamp.batch
            for lg in self.loggers:
                lg.log_metrics(self._pending, step)
            self._pending = {}

    def flops_per_token(self) -> float:
        return self.model_cfg.flops_per_token()

    def peak_flops(self) -> float | None:
        if self.device.type != "cuda":
            return None
        from photon_b200.utils.hw import measured_peaks

        return measured_peaks().get("bf16_flops")

    def _emit(self, event: str) -> None:
        for cb in self.callbacks:
            getattr(cb, event)(self)

    def _to_device(self, ids: torch.Tensor) -> torch.Tensor:
        if self.device.type != "cuda":
            return ids.to(self.device)
        assert self._copy_stream is not None
        with torch.cuda.stream(self._copy_stream):
            out = ids.to(self.device, non_blocking=True)
        torch.cuda.current_stream(self.device).wait_stream(self._copy_stream)
        return out

    def _next_batch(self) -> dict[str, torch.Tensor]:
        if self.train_loader is None:
            raise RuntimeError("Trainer has no train_loader")
        empty_epochs = 0
        while True:
            fresh = self._train_iter is None
            if fresh:
                self._train_iter = iter(self.train_loader)
            limit = self.train_subset_num_batches
            try:
                if limit >= 0 and self.state.timestamp.batch_in_epoch >= limit:
                    raise StopIteration       # train_subset_num_batches: the epoch ends early
                return next(self._train_iter)
            except StopIteration:
                if hasattr(self._train_iter, "close"):
                    self._train_iter.close()
                self._train_iter = None
                self.state.timestamp.advance_epoch()
                empty_epochs = empty_epochs + 1 if fresh else 0
                if empty_epochs >= 2:   # a whole epoch without a single batch (dataset < one batch with drop_last, subset of 0)
                    raise RuntimeError("the train loader yields no batches per epoch (dataset smaller than one batch with drop_last, "
                                       "or train_subset_num_batches=0): nothing to train on")

    def _agree_min(self, v: int) -> int:
        if self.world_size > 1 and dist.is_initialized():
            t = torch.tensor([v], device=self.device if dist.get_backend(self.process_group) == "nccl" else "cpu")
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.process_group)
            return int(t.item())
        return v

    # ------------------------------------------------------------------ training
    def _train_batch(self, batch: dict[str, torch.Tensor]) -> None:
        st = self.state
        ids_host = batch["input_ids"]
        B, S = ids_host.shape
        n_tok_target = float(B * (S - 1))  # packed sequences: only the last position is ignored
        scale = self.scaler.scale if self.scaler else 1.0
        while True:
            mb = int(self._auto_mb if self._auto_mb is not None else self.microbatch)
            mb = max(1, min(mb, B))
            try:
                st.flat.zero_grad()
                loss_sum = torch.zeros((), device=self.device, dtype=torch.float32)
                n_tok = torch.zeros((), device=self.device, dtype=torch.float32)
                uni_logp = getattr(st.backend, "unigram_log_probs", None)
                uni_sum = torch.zeros((), device=self.device, dtype=torch.float32) if uni_logp is not None else None
                for lo in range(0, B, mb):
                    ids = self._to_device(ids_host[lo:lo + mb])
                    ls, n = st.backend.fwd_bwd(ids, n_tok_target, scale)
                    loss_sum += ls.float()
                    n_tok += n.float() if torch.is_tensor(n) else float(n)
                    if uni_sum is not None:  # CE of the unigram model needs the targets only (K15: no second pass over logits)
                        uni_sum += unigram_loss_sum(shift_labels(ids).view(-1), uni_logp).float()
                break
            except RuntimeError as e:  # auto microbatch: halve on OOM (ref: SURVEY App. C)
                if self._auto_mb is None or not _is_oom(e) or mb == 1:
                    raise
                if self.device.type == "cuda":
                    torch.cuda.empty_cache()
                self._auto_mb = self._agree_min(max(1, mb // 2))
                print(f"[trainer] CUDA OOM at microbatch {mb}; retrying with {self._auto_mb}")
        if self._auto_mb is not None and self.world_size > 1 and st.timestamp.batch == self.fit_start_batch:
            self._auto_mb = self._agree_min(self._auto_mb)

        if self.fused_comm_step:
            # N1 + K11 + K12 fused: nothing else to do for this batch
            self._emit("after_backward")
            gnorm = self.grad_comm.step(st.optimizer, st.optimizer.initial_lr * float(st.scheduler(st.timestamp.batch)),
                                        self.grad_clip_norm, 1.0 / scale)
            if self.grad_clip_norm is not None:
                self.log({"l2_norm/grad/clipped_from": gnorm})
            self.last_batch_stats = {"loss_sum": loss_sum, "n_tokens": n_tok, **({"unigram_loss_sum": uni_sum} if uni_sum is not None else {})}
            st.timestamp.advance_batch(samples=B * self.world_size, tokens=B * S * self.world_size)
            return
        # N1: ONE gradient all-reduce on the flat bucket (mean over ranks)
        if self.world_size > 1:
            self._allreduce_grads()
        if self.grad_clip_value is not None:
            lim = self.grad_clip_value * scale
            st.flat.grads.clamp_(-lim, lim)
        self._emit("after_backward")

        grad_mult: torch.Tensor | float | None = None
        skip = False
        if self.grad_clip_norm is not None or self.scaler is not None:
            gnorm = self._grad_norm() / scale
            if self.scaler is not None:
                skip = not bool(torch.isfinite(gnorm))
                self.scaler.update(skip)
            coef = clip_coefficient(gnorm, self.grad_clip_norm) if self.grad_clip_norm is not None else 1.0
            grad_mult = coef / scale if scale != 1.0 else coef
            self.log({"l2_norm/grad/clipped_from": gnorm})  # device scalar; floated lazily below
        if not skip:
            z3 = self.grad_comm if getattr(self.grad_comm, "zero3", False) else None
            if z3 is not None:
                z3.before_param_write()       # peers have finished pulling this step's weights from this rank's shard
            st.optimizer.step(st.scheduler(st.timestamp.batch), grad_mult)
            if z3 is not None:
                z3.params_changed()           # every shard is new before anybody pulls for the next step
            if not (st.optimizer.use_kernel and st.optimizer.bf16_shadow is not None):
                st.backend.params_updated()
        self.last_batch_stats = {"loss_sum": loss_sum, "n_tokens": n_tok, **({"unigram_loss_sum": uni_sum} if uni_sum is not None else {})}
        st.timestamp.advance_batch(samples=B * self.world_size, tokens=B * S * self.world_size)

    def _grad_norm(self) -> torch.Tensor:
        g = self.state.flat.grads
        if hasattr(self.grad_comm, "grad_norm"):     # sharded gradients: the norm spans every rank's shard
            return self.grad_comm.grad_norm(g)
        if g.is_cuda and self.state.optimizer.use_kernel:
            from photon_b200 import ops

            return ops.flat_l2_norm(g)
        return g.norm()

    def _allreduce_grads(self) -> None:
        g = self.state.flat.grads
        if self.grad_comm is not None:
            self.grad_comm.all_reduce_mean_(g)  # fused NVLink kernel (photon_b200.parallel.ddp)
            return
        dist.all_reduce(g, group=self.process_group)
        g.div_(self.world_size)

    def fit(self, duration: str | int | None = None, reset_time: bool = False) -> None:
        """Train ``duration`` more (default: until ``max_duration``)."""
        if self.closed:
            raise RuntimeError("Trainer is closed")
        st = self.state
        if reset_time:
            st.timestamp.reset()
        if duration is not None:
            n = Time.parse(duration).to_batches(max_duration=self.max_duration, **self._geom)
            end = st.timestamp.batch + n
        elif self.max_duration is not None:
            end = self.max_duration.to_batches(**self._geom)
        else:
            raise ValueError("fit() needs a duration or max_duration")
        self.fit_start_batch, self.fit_end_batch = st.timestamp.batch, end
        st.backend.train_mode(True)
        for m in st.train_metrics.values():
            m.reset()
        self._emit("fit_start")
        while st.timestamp.batch < end:
            t0 = time.perf_counter()
            self._emit("batch_start")
            self._train_batch(self._next_batch())
            if (st.timestamp.batch - self.fit_start_batch) % self.metric_sync_interval == 0 or st.timestamp.batch == end:
                self._collect_train_metrics()
            st.timestamp.total_wct_s += time.perf_counter() - t0
            self._emit("batch_end")
            self._flush_logs()
            if self.save_interval and self.save_folder and st.timestamp.batch % self.save_interval == 0:
                self.save_checkpoint()
            if self.eval_interval and self.eval_loaders and st.timestamp.batch % self.eval_interval == 0 \
                    and st.timestamp.batch < end:
                self.eval()
                st.backend.train_mode(True)
        self._emit("fit_end")
        self._flush_logs()

    def _collect_train_metrics(self) -> None:
        """D2H read of the step's loss (the only host sync in the step)."""
        stats = {k: float(v) for k, v in self.last_batch_stats.items()}
        if self.world_size > 1 and dist.is_initialized():
            keys = sorted(stats)
            t = torch.tensor([stats[k] for k in keys], dtype=torch.float64,
                             device=self.device if dist.get_backend(self.process_group) == "nccl" else "cpu")
            dist.all_reduce(t, group=self.process_group)
            stats = dict(zip(keys, t.tolist()))
        for m in self.state.train_metrics.values():
            m.update(stats)
        loss = stats["loss_sum"] / max(stats["n_tokens"], 1.0)
        out = {"loss/train/total": loss, "metrics/train/LanguageCrossEntropy": loss}
        for k, v in list(self._pending.items()):
            if torch.is_tensor(v):
                self._pending[k] = float(v)
        self.log(out)

    # ---------------------------------------------------------------- evaluation
    @torch.no_grad()
    def eval(self, subset_num_batches: int | None = None) -> dict[str, float]:
        st = self.state
        st.backend.train_mode(False)
        limit = self.eval_subset_num_batches if subset_num_batches is None else subset_num_batches
        st.eval_timestamp.reset()
        for label, loader in self.eval_loaders.items():
            metrics = st.eval_metrics.setdefault(label, build_metrics(bool(getattr(st.backend, "unigram_log_probs", None) is not None)))
            for m in metrics.values():
                m.reset()
            for i, batch in enumerate(loader):
                if 0 <= limit <= i:
                    break
                ids = self._to_device(batch["input_ids"])
                stats = self._eval_batch_stats(ids)
                for m in metrics.values():
                    m.update(stats)
                st.eval_timestamp.advance_batch(samples=ids.shape[0] * self.world_size,
                                                tokens=ids.numel() * self.world_size)
            if self.world_size > 1:     # the Trainer's OWN data-parallel group; a 1-rank trainer inside a bigger job must not
                sync_metrics(metrics, self.process_group)      # all-reduce over the job's WORLD group (the other ranks are not evaluating)
        vals = st.eval_metric_values
        self.log({f"metrics/{k}": v for k, v in vals.items()})
        if self.icl_suite is not None:   # llm-foundry's ICL evaluators + EvalGauntlet run as part of every trainer.eval()
            # generation tasks decode batched through the backend (on the engine: KV-cached, on its own kernels)
            gen = st.backend.generate if st.backend.kind == "torch" or getattr(st.backend, "can_generate", False) else None
            icl = {k: v for k, v in self.icl_suite(st.backend.logits, gen).items() if isinstance(v, (int, float))} if self.rank == 0 else {}
            self.last_icl_metrics = icl
            if self.world_size > 1 and dist.is_initialized():
                # the suite runs on rank 0 only and can take minutes: the others wait HERE, on the host, instead of inside the next
                # step's NVLink kernel (whose peer spins are time-bounded) — and leave their parameter shards alone meanwhile
                dist.barrier(group=self.process_group)
            self.log({(k if k.startswith("icl/") else f"metrics/icl/{k}"): float(v) for k, v in icl.items()})
            vals = {**vals, **{(k if k.startswith("icl/") else f"icl/{k}"): float(v) for k, v in icl.items()}}
        self._emit("eval_end")
        self._flush_logs()
        return vals

    def _eval_batch_stats(self, ids: torch.Tensor) -> dict[str, float]:
        """Sum-type statistics of one eval batch, computed in ``device_eval_microbatch_size`` slices (``auto`` halves the
        slice on an out-of-memory error and remembers the size that worked — same policy as the train microbatch)."""
        B = ids.shape[0]
        while True:
            mb = self.eval_microbatch
            mb = B if mb in (None, "auto") else max(1, min(int(mb), B))
            try:
                total: dict[str, float] = {}
                for lo in range(0, B, mb):
                    for k, v in self.state.backend.eval_stats(ids[lo:lo + mb]).items():
                        total[k] = total.get(k, 0.0) + float(v)
                return total
            except RuntimeError as e:
                if not self._eval_mb_auto or not _is_oom(e) or mb == 1:
                    raise
                if self.device.type == "cuda":
                    torch.cuda.empty_cache()
                self.eval_microbatch = max(1, mb // 2)
                print(f"[trainer] CUDA OOM at eval microbatch {mb}; retrying with {self.eval_microbatch}")

    # --------------------------------------------------------------- checkpoints
    def state_dict(self) -> dict[str, Any]:
        st = self.state
        names = st.flat.layout.names
        return {
            "state": {
                "model": (lambda full: {n: st.flat.layout.view(full, i).detach().cpu().clone() for i, n in enumerate(names)})(
                    st.flat.full_params()),
                "optimizers": {type(st.optimizer).__name__: st.optimizer.state_dict()},
                "schedulers": {"lr": {"last_batch": st.timestamp.batch}},
                "timestamp": st.timestamp.state_dict(),
                "dataset_state": {"train": self.train_loader.state_dict() if hasattr(self.train_loader, "state_dict") else {}},
                "callbacks": {type(c).__name__: c.state_dict() for c in self.callbacks},
                "run_name": st.run_name,
                "scaler": {"scale": self.scaler.scale} if self.scaler else None,
                "fp8": self._fp8_state(),
            },
            "rng": {"torch": torch.get_rng_state(), "seed": self.seed},
        }

    def _fp8_state(self) -> dict[str, Any] | None:
        """amax histories / scales of an ``amp_fp8`` run (the delayed-scaling recipe resumes with the scales it stopped with)."""
        if hasattr(self.state.backend, "fp8_state_dict"):      # the sm_100a engine keeps its scales on the device
            return self.state.backend.fp8_state_dict()
        if not getattr(self.state.backend, "fp8_layers", None):
            return None
        from photon_b200.train.fp8 import fp8_state_dict

        return fp8_state_dict(self.state.backend.model)

    def checkpoint_name(self) -> str:
        ts = self.state.timestamp
        return self.save_filename.format(epoch=ts.epoch, batch=ts.batch, rank=self.rank, run_name=self.state.run_name)

    def _pruned_state_dict(self) -> dict[str, Any]:
        """``state_dict()`` minus what ``save_weights_only`` / ``save_ignore_keys`` (Composer glob paths such as ``*optim*`` or
        ``state/dataset_state``) exclude — e.g. the reference drops optimizer state from client checkpoints when
        ``fl.reset_optimizer`` (ref: clients/utils.py:229-238)."""
        sd = self.state_dict()
        if self.save_weights_only:
            return {"state": {"model": sd["state"]["model"], "run_name": sd["state"]["run_name"]}}
        for key in list(sd["state"]):
            if any(fnmatch.fnmatch(key, pat) or fnmatch.fnmatch("state/" + key, pat) for pat in self.save_ignore_keys):
                del sd["state"][key]
        if any(fnmatch.fnmatch("rng", pat) for pat in self.save_ignore_keys):
            sd.pop("rng", None)
        return sd

    def save_checkpoint(self, folder: str | None = None) -> Path:
        folder_p = Path(folder or self.save_folder or ".")
        folder_p.mkdir(parents=True, exist_ok=True)
        path = folder_p / self.checkpoint_name()
        if path.exists() and not self.save_overwrite:
            raise FileExistsError(path)
        tmp = path.with_suffix(".pt.tmp")
        torch.save(self._pruned_state_dict(), tmp)
        os.replace(tmp, path)
        latest = folder_p / self.save_latest_filename.format(rank=self.rank, run_name=self.state.run_name)
        if latest.is_symlink() or latest.exists():
            latest.unlink()
        latest.symlink_to(path.name)
        self._saved.append(path)
        if self.save_keep >= 0:
            while len(self._saved) > max(self.save_keep, 1):
                old = self._saved.pop(0)
                if old.exists() and old != path:
                    old.unlink()
        return path

    def load_checkpoint(self, path: str | os.PathLike, ignore_keys: Iterable[str] = (), *, weights_only: bool = False,
                        strict_model_weights: bool = False) -> None:
        """``weights_only`` = Composer's ``load_weights_only`` (model tensors, nothing else); ``strict_model_weights`` refuses a
        checkpoint whose tensor names do not match the model's exactly (otherwise names in common are loaded)."""
        ck = torch.load(path, map_location="cpu", weights_only=False)
        pats = list(ignore_keys) + (["optimizers", "timestamp", "dataset_state", "scaler", "fp8", "rng", "callbacks"] if weights_only else [])
        if strict_model_weights:
            have, want = set(ck["state"].get("model", {})), set(self.state.flat.layout.names)
            if have != want:
                raise KeyError(f"checkpoint / model tensor names differ: missing {sorted(want - have)[:3]}, unexpected {sorted(have - want)[:3]}")

        def ignored(key: str) -> bool:
            return any(fnmatch.fnmatch(key, p) or fnmatch.fnmatch("state/" + key, p) for p in pats)

        s = ck["state"]
        st = self.state
        if not ignored("model"):
            with torch.no_grad():
                full = st.flat.full_params()      # the buffer itself, or a gathered copy under full parameter sharding
                for i, n in enumerate(st.flat.layout.names):
                    if n in s["model"]:
                        st.flat.layout.view(full, i).copy_(s["model"][n])
                if getattr(st.flat, "is_sharded", False):
                    st.flat.load_full_params(full)
            st.backend.params_updated()
        if not ignored("optimizers") and s.get("optimizers"):
            sd = s["optimizers"].get(type(st.optimizer).__name__)
            if sd is not None:
                st.optimizer.load_state_dict(sd)
        if not ignored("timestamp") and "timestamp" in s:     # absent from weights-only / pruned checkpoints
            st.timestamp.load_state_dict(s["timestamp"])
        if not ignored("dataset_state") and hasattr(self.train_loader, "load_state_dict"):
            ds = (s.get("dataset_state") or {}).get("train")
            if ds:
                self.train_loader.load_state_dict(ds)
                self._train_iter = None
        if self.scaler and s.get("scaler") and not ignored("scaler"):
            self.scaler.scale = float(s["scaler"]["scale"])
        if s.get("fp8") and not ignored("fp8"):
            if hasattr(st.backend, "load_fp8_state_dict"):
                st.backend.load_fp8_state_dict(s["fp8"])
            elif getattr(st.backend, "fp8_layers", None):
                from photon_b200.train.fp8 import load_fp8_state_dict

                load_fp8_state_dict(st.backend.model, s["fp8"])
        if not ignored("rng") and "rng" in ck and "torch" in ck["rng"]:
            torch.set_rng_state(ck["rng"]["torch"])

    # --------------------------------------------------------------------- close
    def close(self) -> None:
        if self.closed:
            return
        for lg in self.loggers:
            lg.close()
        self.state.backend.close()
        self.closed = True
