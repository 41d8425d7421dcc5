"""Build (and re-use) the per-client Trainer from the resolved config.

``get_trainer_object`` is the B200 engine's counterpart of the reference's fork
of llm-foundry ``train.py`` (ref: photon/clients/trainer_utils.py:1117-1721):
device pick from ``APPOINTED_CUDA_DEVICE``, process-group bring-up, per-client
streams, loaders, evaluators, callbacks, loggers, optimizer, scheduler,
algorithms (gradient clipping), checkpoint policy.  ``reconfigure_trainer`` is
the "mutables" path (ref: ``get_trainer_mutables_from_config`` +
``set_mutables_trainer*``, :330-1114): a live Trainer — and its CUDA context,
workspace and compiled kernels — survives across rounds/clients; only loaders,
save folder, loggers and clocks are swapped.
"""
from __future__ import annotations

import dataclasses
import os
from pathlib import Path
from typing import Any

import torch
import torch.distributed as dist

from photon_b200.clients import llm_config_functions as lcf
from photon_b200.data.synthetic import TOKENIZER_VOCAB
from photon_b200.data.streaming import build_text_loader
from photon_b200.metrics.language import unigram_log_probs
from photon_b200.models.mpt import MPTConfig
from photon_b200.train.callbacks import build_callbacks, build_loggers
from photon_b200.train.timestamp import Time
from photon_b200.train.trainer import Trainer
from photon_b200.utils.core import add_unigram_metrics, appointed_cuda_devices  # noqa: F401 - add_unigram_metrics: reference name of this module


def pick_device(local_rank: int = 0) -> torch.device:
    if not torch.cuda.is_available():
        return torch.device("cpu")
    appointed = appointed_cuda_devices()
    idx = appointed[local_rank % len(appointed)] if appointed else local_rank % torch.cuda.device_count()
    torch.cuda.set_device(idx)
    return torch.device("cuda", idx)


def initialize_dist(device: torch.device, timeout_s: float = 600.0) -> tuple[int, int]:
    """Bring up the intra-client process group from torchrun-style env (NCCL on GPU, gloo on CPU)
    and smoke-test it with a barrier (ref: trainer_utils.py:403-405,1249-1251)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1 and not dist.is_initialized():
        import datetime

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if device.type == "cuda" else "gloo", rank=rank, world_size=world,
                                timeout=datetime.timedelta(seconds=timeout_s))
        dist.barrier()
    return rank, world


def _prepare_train_cfg(cfg: Any, cid: int | str | None, split_eval: bool, n_devices: int, log_name: str) -> tuple[Any, dict[str, Any]]:
    t = lcf.get_train_config(cfg["llm_config"], run_uuid=str(cfg.get("run_uuid", "run")))
    lcf.adapt_train_batch_size_to_num_devices(t, n_devices)
    lcf.set_n_workers_dataloaders(t, n_devices)
    evals = lcf.client_set_data_config(t, cid, split_eval)
    lcf.set_dataset_default_params(t)
    lcf.set_client_loggers(t, log_name)
    return t, evals


def _grad_clip(train_cfg: Any, kind: str = "norm") -> float | None:
    """``algorithms.gradient_clipping`` → threshold for ``kind`` (``norm``: global L2, the reference's setting; ``value``:
    element-wise clamp — Composer's two non-adaptive types). None when the algorithm is absent or of the other kind."""
    gc = ((train_cfg.get("algorithms") or {}).get("gradient_clipping") or None)
    if not gc:
        return None
    have = str(gc.get("clipping_type", "norm"))
    if have not in ("norm", "value"):
        raise NotImplementedError(f"gradient_clipping.clipping_type={have!r}: norm and value are supported (adaptive is not)")
    return float(gc["clipping_threshold"]) if have == kind else None


def _with_profiler(t: Any) -> dict[str, Any]:
    """``llm_config.callbacks`` plus the optional ``llm_config.profiler`` node (ref: trainer_utils.py:1456-1482)."""
    cbs = dict(t.get("callbacks") or {})
    if t.get("profiler"):
        cbs["profiler"] = dict(t["profiler"])
    return cbs


def apply_runtime_env(llm_cfg: Any) -> dict[str, str]:
    """Process-level knobs of ``llm_config`` that must be in the environment before CUDA / the process group come up
    (ref: trainer_utils.py:1278-1298): caching-allocator configuration (``max_split_size_mb``, ``expandable_segments``),
    lazy CUDA module loading, python log level. Returns what was set."""
    import logging

    out: dict[str, str] = {}
    alloc = []
    if llm_cfg.get("max_split_size_mb") is not None:
        alloc.append(f"max_split_size_mb:{int(llm_cfg['max_split_size_mb'])}")
    if llm_cfg.get("expandable_segments"):
        alloc.append("expandable_segments:True")
    if alloc:
        out["PYTORCH_CUDA_ALLOC_CONF"] = ",".join(alloc)
    if llm_cfg.get("cuda_load_lazy"):
        out["CUDA_MODULE_LOADING"] = "LAZY"
    os.environ.update(out)
    level = llm_cfg.get("python_log_level")
    if level:
        logging.getLogger("photon_b200").setLevel(str(level).upper())
        out["python_log_level"] = str(level).upper()
    return out


def get_trainer_object(cfg: Any, cid: int | str | None, *, log_name: str = "", device: torch.device | None = None,
                       rank: int | None = None, world_size: int | None = None, process_group: Any = None,
                       grad_comm: Any = None, split_eval: bool = False, use_unigram_metrics: bool = False,
                       allow_unigram_metrics_failures: bool = False, frozen_layers: list[str] | None = None,
                       unfrozen_layers: list[str] | None = None, resize_vocab: int | None = None,
                       no_data: bool = False, backend: Any = None) -> tuple[Trainer, Any]:
    """Returns ``(trainer, train_cfg)``. ``cid=None`` = all streams (centralised / evaluation)."""
    apply_runtime_env(cfg["llm_config"])
    device = device or pick_device(int(os.environ.get("LOCAL_RANK", "0")))
    if rank is None or world_size is None:
        rank, world_size = initialize_dist(device, timeout_s=float(cfg["llm_config"].get("dist_timeout") or 600.0))
    t, evals = _prepare_train_cfg(cfg, cid, split_eval, world_size, log_name)
    if t.get("compile_config"):
        print("[trainer] compile_config is ignored: the GPU step is an explicit kernel schedule replayed as a CUDA graph")
    if t.get("tp_config"):
        raise ValueError("tp_config must be null (TP is plumbing-only in the reference)")
    model_node = dict(t["model"])
    if resize_vocab:
        model_node["vocab_size"] = int(resize_vocab)  # ref: clients/utils.py:245-249
    mcfg = MPTConfig.from_model_cfg(model_node)
    if device.type == "cpu" and mcfg.attn_impl == "flash":
        mcfg.attn_impl = "torch"  # README.md:82-84: CPU runs use the eager attention path
    precision = t.get("precision", "amp_bf16")
    gbs = int(t["global_train_batch_size"])
    seed = int(t.get("seed", 17))
    uni = None
    if use_unigram_metrics:
        freq = lcf.get_stream_freq_dict_for_client(t, cid, allow_failures=allow_unigram_metrics_failures)
        if freq is not None:
            uni = unigram_log_probs(freq, mcfg.vocab_size)
        elif not allow_unigram_metrics_failures:
            raise RuntimeError("unigram metrics requested but no 1_gram.json found")
    syn_vocab = min(int(mcfg.vocab_size), TOKENIZER_VOCAB)   # synthetic streams stay inside the model's embedding table
    train_loader = None if no_data else build_text_loader(t["train_loader"], gbs // world_size, rank, world_size, seed, syn_vocab)
    eval_bs = int(t.get("device_eval_batch_size", 1))
    eval_loaders = {} if no_data else {lbl: build_text_loader(lc, eval_bs, rank, world_size, seed + 1, syn_vocab) for lbl, lc in evals.items()}
    save_root = t.get("save_folder") or "."
    interval = t.get("console_log_interval", "1ba")
    loggers = build_loggers(t.get("loggers"), Path(str(save_root)).parent if t.get("save_folder") else ".", str(t["run_name"]),
                            console_interval=Time.parse(interval).to_batches(), log_to_console=bool(t.get("log_to_console", True)), rank=rank,
                            progress_bar=bool(t.get("progress_bar", False)),
                            total_batches=(Time.parse(t["max_duration"]).to_batches() if str(t.get("max_duration", "")).endswith("ba") else None))
    kernels = dict(cfg.get("kernels") or {})
    if mcfg.attn_impl == "torch" and device.type == "cuda" and kernels.get("attention", "auto") == "auto":
        kernels["attention"] = "torch"
    # fsdp_config present (YAML default) → shard the optimizer state over the client's GPUs; the launch scripts delete the
    # node (or set NO_SHARD) for plain DDP (ref: scripts/cen_125m_example.sh:87, trainer_utils.py:1378-1393: 1 GPU → DDP)
    fsdp = t.get("fsdp_config") or None
    shard_state = bool(fsdp) and world_size > 1 and str(dict(fsdp).get("sharding_strategy", "FULL_SHARD")).upper() != "NO_SHARD"
    tr = Trainer(mcfg, optimizer_cfg=dict(t["optimizer"]), scheduler_cfg=dict(t.get("scheduler") or {}),
                 train_loader=train_loader, eval_loaders=eval_loaders, global_train_batch_size=gbs,
                 device_train_microbatch_size=t.get("device_train_microbatch_size", "auto"),
                 device_eval_batch_size=eval_bs, device_eval_microbatch_size=t.get("device_eval_microbatch_size"),
                 precision=precision, max_duration=t.get("max_duration"),
                 grad_clip_norm=_grad_clip(t), grad_clip_value=_grad_clip(t, "value"), callbacks=build_callbacks(_with_profiler(t)), loggers=loggers,
                 save_folder=t.get("save_folder"), save_interval=t.get("save_interval"),
                 save_num_checkpoints_to_keep=int(t.get("save_num_checkpoints_to_keep", -1)),
                 save_overwrite=bool(t.get("save_overwrite", False)), save_filename=t.get("save_filename"),
                 save_latest_filename=t.get("save_latest_filename"), save_weights_only=bool(t.get("save_weights_only", False)),
                 save_ignore_keys=t.get("save_ignore_keys"), train_subset_num_batches=int(t.get("train_subset_num_batches", -1) or -1),
                 eval_interval=t.get("eval_interval"),
                 eval_subset_num_batches=int(t.get("eval_subset_num_batches", -1)), device=device, rank=rank,
                 world_size=world_size, process_group=process_group, grad_comm=grad_comm, kernels=kernels, seed=seed,
                 run_name=str(t["run_name"]), use_unigram_metrics=uni is not None, unigram_log_probs=uni,
                 frozen_layers=frozen_layers, unfrozen_layers=unfrozen_layers, backend=backend,
                 shard_optimizer_state=shard_state,
                 # host read-back of the loss: every `metric_sync_interval` batches (default: whenever the console logs) — between
                 # two reads the step path has no host synchronisation at all
                 metric_sync_interval=int(t.get("metric_sync_interval") or max(1, Time.parse(interval).to_batches())),
                 activation_checkpointing=bool(fsdp) and bool(dict(fsdp).get("activation_checkpointing", False)))
    tr.icl_suite = build_icl_suite(cfg, mcfg.max_seq_len)
    return tr, t


def build_icl_suite(cfg: Any, max_seq_len: int) -> Any:
    """``icl_tasks_config`` (+ ``eval_gauntlet_config``) → a callable the Trainer runs at every ``eval()``
    (ref: centralised_train.py:120-136 and llm-foundry ``build_evaluators`` / ``EvalGauntlet``). None when no task is listed."""
    tasks = ((cfg.get("icl_tasks_config") or {}).get("icl_tasks")) or []
    if not tasks:
        return None
    from photon_b200.dataset.utils import build_tokenizer
    from photon_b200.eval.icl import run_icl_suite

    tok_cfg = dict((cfg["llm_config"].get("tokenizer") or {}))
    tokenizer = build_tokenizer(str(tok_cfg.get("name", "EleutherAI/gpt-neox-20b")))
    return lambda logits_fn, generate_fn=None: run_icl_suite(logits_fn, tokenizer, cfg, max_seq_len, generate_fn=generate_fn)


@dataclasses.dataclass
class TrainerMutableAttributes:
    """What changes on a live Trainer between clients / rounds (ref: trainer_utils.py:172-202): the client's loaders, its loggers and
    callbacks, the per-client training config and the checkpoint file templates. Everything else — model, optimizer planes, CUDA
    context, kernel workspace, captured graphs — is kept."""

    train_loader: Any
    evaluators: dict[str, Any] | None
    callbacks: list[Any] | None
    loggers: list[Any] | None
    train_cfg: Any
    save_latest_filename: str | None = None
    save_filename: str = "ep{epoch}-ba{batch}-rank{rank}.pt"


def get_trainer_mutables_from_config(cfg: Any, cid: int | str | None, trainer: Trainer, *, log_name: str = "", split_eval: bool = False,
                                     rebuild_loggers: bool = False) -> TrainerMutableAttributes:
    """Build the per-client mutables from the resolved config for the geometry of ``trainer`` (rank, world size, device batch)
    (ref: trainer_utils.py:330-653). Loggers / callbacks are rebuilt only on request: re-opening a wandb run or a tensorboard
    writer every round is what the reference's per-client logger names exist for, the default keeps the Trainer's own."""
    t, evals = _prepare_train_cfg(cfg, cid, split_eval, trainer.world_size, log_name)
    seed = int(t.get("seed", 17))
    syn_vocab = min(int(trainer.model_cfg.vocab_size), TOKENIZER_VOCAB)
    train_loader = build_text_loader(t["train_loader"], trainer.device_batch, trainer.rank, trainer.world_size, seed, syn_vocab)
    evaluators = {lbl: build_text_loader(lc, trainer.device_eval_batch_size, trainer.rank, trainer.world_size, seed + 1, syn_vocab)
                  for lbl, lc in evals.items()}
    loggers = callbacks = None
    if rebuild_loggers:
        save_root = t.get("save_folder") or "."
        interval = t.get("console_log_interval", "1ba")
        loggers = build_loggers(t.get("loggers"), Path(str(save_root)).parent if t.get("save_folder") else ".", str(t["run_name"]),
                                console_interval=Time.parse(interval).to_batches(), log_to_console=bool(t.get("log_to_console", True)),
                                rank=trainer.rank, progress_bar=bool(t.get("progress_bar", False)))
        callbacks = build_callbacks(_with_profiler(t))
    return TrainerMutableAttributes(train_loader, evaluators, callbacks, loggers, t, t.get("save_latest_filename"),
                                    t.get("save_filename") or "ep{epoch}-ba{batch}-rank{rank}.pt")


def set_mutables_trainer_train_dataloader(trainer: Trainer, train_dataloader: Any, client_config: Any = None) -> None:
    """(ref: trainer_utils.py:911-982) the iterator restarts with the new loader; the data position of a resumed client comes back
    with its checkpoint (``load_trainer_checkpoint``)."""
    del client_config
    trainer.train_loader = train_dataloader
    trainer._train_iter = None  # noqa: SLF001


def set_mutables_trainer_eval_dataloader(trainer: Trainer, eval_dataloader: dict[str, Any] | None, train_cfg: Any = None) -> None:
    """(ref: trainer_utils.py:985-1068) one evaluator per label; metric objects are created lazily per label by ``Trainer.eval``."""
    del train_cfg
    trainer.eval_loaders = dict(eval_dataloader or {})


def set_mutables_trainer_callbacks_and_loggers(trainer: Trainer, callbacks: list[Any] | None, loggers: list[Any] | None, train_cfg: Any,
                                               save_latest_filename: str | None = None, save_filename: str | None = None) -> None:
    """(ref: trainer_utils.py:656-908) new loggers / callbacks replace the old ones (which are closed), and the checkpoint policy
    of the client — folder, file templates — is installed."""
    if loggers is not None:
        for lg in trainer.loggers:
            lg.close()
        trainer.loggers = list(loggers)
    if callbacks is not None:
        trainer.callbacks = list(callbacks)
    trainer.save_folder = train_cfg.get("save_folder")
    trainer._saved = []  # noqa: SLF001
    if save_filename:
        trainer.save_filename = save_filename
    if save_latest_filename:
        trainer.save_latest_filename = save_latest_filename
    trainer.state.run_name = str(train_cfg["run_name"])


def set_mutables_trainer(trainer: Trainer, trainer_mutable_attributes: TrainerMutableAttributes, client_config: Any = None,
                         reset_timestamp: bool = False) -> None:
    """Install a :class:`TrainerMutableAttributes` on a live Trainer (ref: trainer_utils.py:1071-1114). The reference always
    zeroes the clocks here and restores them from the client checkpoint; ``reset_timestamp`` makes that explicit."""
    m = trainer_mutable_attributes
    set_mutables_trainer_callbacks_and_loggers(trainer, m.callbacks, m.loggers, m.train_cfg, m.save_latest_filename, m.save_filename)
    set_mutables_trainer_train_dataloader(trainer, m.train_loader, client_config)
    set_mutables_trainer_eval_dataloader(trainer, m.evaluators, m.train_cfg)
    trainer.closed = False
    if reset_timestamp:
        trainer.state.timestamp.reset()


def reconfigure_trainer(trainer: Trainer, cfg: Any, cid: int | str | None, *, log_name: str = "", split_eval: bool = False,
                        reset_timestamp: bool = False, use_unigram_metrics: bool | None = None,
                        allow_unigram_metrics_failures: bool = False) -> Any:
    """Swap the per-client mutables on a live Trainer (loaders, save folder, run name, clocks, and — when
    ``use_unigram_metrics`` — the unigram table of THIS client's streams; ref: trainer_utils.py:278-327,656-1114):
    ``get_trainer_mutables_from_config`` + ``set_mutables_trainer`` in one call. Returns the client's training config."""
    m = get_trainer_mutables_from_config(cfg, cid, trainer, log_name=log_name, split_eval=split_eval)
    if use_unigram_metrics:
        freq = lcf.get_stream_freq_dict_for_client(m.train_cfg, cid, allow_failures=allow_unigram_metrics_failures)
        if freq is not None:
            add_unigram_metrics(trainer, freq)
        elif not allow_unigram_metrics_failures:
            raise RuntimeError("unigram metrics requested but no 1_gram.json found")
    set_mutables_trainer(trainer, m, reset_timestamp=reset_timestamp)
    return m.train_cfg


def load_trainer_checkpoint(trainer: Trainer, load_path: str, ignore_keys: list[str] | None = None) -> None:
    """``load_path`` may contain ``{rank}`` (ref: trainer_utils.py:229-275)."""
    trainer.load_checkpoint(load_path.format(rank=trainer.rank), ignore_keys or [])


def load_kwargs_from_config(train_cfg: Any) -> dict[str, Any]:
    """``load_weights_only`` / ``load_strict_model_weights`` / ``load_ignore_keys`` of ``llm_config`` as ``load_checkpoint`` kwargs."""
    return dict(ignore_keys=list(train_cfg.get("load_ignore_keys") or []), weights_only=bool(train_cfg.get("load_weights_only", False)),
                strict_model_weights=bool(train_cfg.get("load_strict_model_weights", False)))


def trainer_clean_up(trainer: Trainer) -> None:
    """Close loggers and drop the workspace; barrier so every rank leaves together
    (ref: trainer_utils.py:205-226)."""
    trainer.close()
    if dist.is_available() and dist.is_initialized() and trainer.world_size > 1:
        dist.barrier(group=trainer.process_group)
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
