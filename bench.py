#!/usr/bin/env python
"""Headline benchmark of photon_b200 — one script for every BASELINE.json config.

    python bench.py --gpus 1 --steps 4 --warmup 3                       # config #2 (default): MPT-125M, 8 federated clients
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W [--mode fed|ddp|fed4x2] [--model mpt-1b --server fedadam --precision amp_fp8]

``--mode fed``  (configs #2 / #4)  ``fed_125m_example``: 8 clients per round spread over the N GPUs (8/N per GPU, time-multiplexed on the
    node's persistent Trainer), local batch 32 × 2048, ADOPT (125M) / DecoupledAdamW (1B+), FedAvg ≡ Nesterov η=1 μ=0 or FedAdam;
    one "step" = every client advances one local optimizer step (8 × 32 × 2048 tokens); the timed region is ONE full round of K
    local steps per client PLUS the round's aggregate + server optimizer + broadcast (the fused NVLink kernel).
``--mode ddp``  (config #3)  ``cen_125m_example``: centralised training, global batch 256 over the N GPUs, DecoupledAdamW, no clipping,
    DDP with the fused NVLink all-reduce on the flat gradient bucket; one step = one optimizer step (256 × 2048 tokens).
``--mode fed4x2`` (config #5)  4 clients × 2 GPUs: DDP inside every client (fused all-reduce), federated round across the clients.

Total work per step is fixed in every mode → ``"scaling": "strong"``.  Two measurements of the same work:
* ``value``      device time (CUDA events on the launching stream, max over ranks; per-rank min/max printed as ``rank_dev_ms``);
* ``e2e.value``  wall clock around the public API call (``FederationRuntime.run_clients_fit`` + ``finish_round`` / ``Trainer.fit``):
                 every step copies its inputs H2D from pinned host memory and reads the loss back D2H (bytes counted).

In the same invocation the reference-EQUIVALENT arm is measured too (``torch_arm``: stock PyTorch ops — cuBLAS, SDPA, ATen LN/GELU/CE,
torch optimizer — with the reference's communication pattern: per-parameter NCCL all-reduce for DDP, host shared-memory round for the
federation), same K, same batch, microbatch ``auto`` (32 unless it runs out of memory); ``vs_torch_arm`` = ours ÷ that.
``--impl reference`` must run the UNMODIFIED reference from ``baseline/_ref``; it cannot be installed offline here (DESIGN.md §0), so
that arm prints ``unavailable``.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_CLIENTS = 8
LOCAL_BATCH = 32
SEQ = 2048
DDP_GLOBAL_BATCH = 256
MODEL_NAMES = {"mpt-125m": "MPT-125M", "mpt-1b": "MPT-1B", "mpt-3b": "MPT-3B", "mpt-7b": "MPT-7B"}
DUMP_PARAMS = 1 << 22       # --dump-outputs: at most this many fp32 parameters (16 MiB), a seeded sample of larger models
DUMP_MAX_BYTES = 64 << 20


def reference_arm() -> None:
    why = ("reference not installable offline: `pip install --no-index --no-build-isolation --find-links /opt/wheelhouse [--no-deps] "
           "--target baseline/_ref` fails with ModuleNotFoundError: poetry (build backend poetry-core absent from image and wheelhouse); "
           "its runtime deps flwr/composer/llm-foundry/streaming (git forks), ray, hydra, omegaconf, torchmetrics are absent too "
           "(DESIGN.md §0); the same-box stand-in is the `torch_arm` key of the default run")
    ref = ROOT / "baseline" / "_ref" / "photon"
    if ref.exists():
        try:
            sys.path.insert(0, str(ref.parent))
            import photon.server_app  # noqa: F401  (would need flwr)
        except Exception as e:  # noqa: BLE001
            why = f"baseline/_ref present but not importable: {type(e).__name__}: {e}"
    if int(os.environ.get("RANK", "0")) == 0:   # one line per job, also under torchrun
        print(json.dumps({"impl": "reference", "unavailable": why}))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): ONE long-lived
    ``nvidia-smi -lms 200`` child started before the region (no fork/exec while the step is being timed)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, enabled: bool = True) -> None:
        self.idx, self.rows, self.proc, self.enabled = gpu_index, [], None, enabled

    def start(self) -> "ClockSampler":
        if self.enabled:
            try:
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx),
                                              "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:  # noqa: BLE001
                self.proc = None
        return self

    def stop(self) -> None:
        if self.proc is None:
            return
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
            out = ""
        self.rows = [[x.strip() for x in line.split(",")] for line in out.splitlines() if line.strip()]

    def summary(self) -> dict:
        load = [r for r in self.rows if len(r) > 3 and r[3].replace(".", "").isdigit() and float(r[3]) > 300.0] or self.rows
        sm = sorted(float(r[1]) for r in load if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = max((float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()), default=0.0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in load for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm),
                "note": "median over samples with power draw > 300 W (under load)"}


# ------------------------------------------------------------------------------------------------------------------ configs
def _common_overrides(args, impl: str) -> list[str]:
    ov = [f"llm_config={args.model}", "run_uuid=bench", f"llm_config.precision={args.precision}", "llm_config.log_to_console=false",
          "~llm_config.loggers.wandb", "~llm_config.loggers.tensorboard", "llm_config.save_folder=null", "llm_config.save_interval=1000000ba",
          "llm_config.eval_interval=1000000ba", "~llm_config.callbacks", "photon.checkpoint=false",
          "++llm_config.metric_sync_interval=1",    # the loss is read back EVERY step: that D2H is part of the e2e number
          "dataset.train.root_local=synthetic://c4", "dataset.val.root_local=synthetic://c4"]
    if impl == "ours":
        ov += [f"kernels.attention={args.attention}"]
    else:   # reference-equivalent stock path
        ov += ["kernels.gemm=torch", "kernels.attention=torch", "kernels.norm=torch", "kernels.loss=torch", "kernels.optimizer=torch"]
    return ov


def fed_cfg(args, impl: str, steps: int, n_clients: int, microbatch):
    from photon_b200.config import compose

    ov = _common_overrides(args, impl) + [
        f"fl.n_total_clients={n_clients}", f"fl.n_clients_per_round={n_clients}", "fl.strategy_name=NESTOROV",
        "fl.strategy_kwargs.server_learning_rate=1.0", "fl.strategy_kwargs.server_momentum=0.0", "fl.reset_optimizer=false",
        "fl.eval_period=null", f"llm_config.global_train_batch_size={LOCAL_BATCH}", f"llm_config.device_train_microbatch_size={microbatch}",
        f"llm_config.local_steps={steps}ba", "llm_config.max_duration=40960ba", "llm_config.scheduler.schedulers.lr.t_max=40960ba",
        "llm_config.scheduler.schedulers.lr.t_warmup=800ba", "photon.comm_stack.shm=false"]
    if args.mode == "fed4x2":
        ov += ["~llm_config.fsdp_config"]      # plain DDP inside the client (the launch scripts' choice, ref: cen_125m_example.sh:87)
    if args.server == "fedadam":   # BASELINE config #4 flavour
        ov += ["fl.strategy_name=fedadam", "fl.strategy_kwargs={eta: 0.1, beta_1: 0.9, beta_2: 0.95, tau: 1.0e-9}", "fl.reset_optimizer=true"]
    ov += ["photon.comm_stack.nvl=true"] if impl == "ours" else ["photon.comm_stack.shm=true"]
    return compose(ov)


def ddp_cfg(args, impl: str, microbatch):
    from photon_b200.config import compose

    ov = _common_overrides(args, impl) + [
        f"llm_config.global_train_batch_size={DDP_GLOBAL_BATCH}", f"llm_config.device_train_microbatch_size={microbatch}",
        "llm_config.scheduler.schedulers.lr.name=constant_with_sqrt_cooldown_with_warmup", "llm_config.scheduler.schedulers.lr.t_warmup=100ba",
        "++llm_config.scheduler.schedulers.lr.t_cooldown=240ba", "llm_config.scheduler.schedulers.lr.t_max=5120ba",
        "llm_config.max_duration=5120ba", "~llm_config.algorithms.gradient_clipping",
        "llm_config.optimizer={name: decoupled_adamw, lr: 6.0e-4, betas: [0.9, 0.95], eps: 1.0e-8, weight_decay: 0.0}",
        "dataset/streams@dataset.train.streams=centralised", "centralized.store_init_model=false", "centralized.store_final_model=false"]
    # plain DDP is the launch scripts' choice for the small models (ref: cen_125m_example.sh:87 deletes fsdp_config); the 7B config
    # keeps its fsdp_config (FULL_SHARD + activation checkpointing, ref: mpt-7b.yaml:85-91) -> full parameter sharding here
    sharding = args.sharding if args.sharding != "auto" else ("zero3" if args.model == "mpt-7b" else "none")
    if sharding == "none" or impl != "ours":
        ov += ["~llm_config.fsdp_config"]
    else:
        ov += [f"kernels.param_sharding={sharding}"]
    return compose(ov)


# ------------------------------------------------------------------------------------------------------------------ arms
class Env:
    """Process-wide state shared by the arms of one invocation."""

    def __init__(self, args) -> None:
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {args.gpus}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py measures the sm_100a engine: it needs a CUDA (B200) device and does not fall back to the CPU")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", rank=self.rank, world_size=self.world, device_id=self.dev)
        from photon_b200.utils.hw import L2_BYTES

        self.flush = torch.empty(max(2 * L2_BYTES, 1 << 28), dtype=torch.uint8, device=self.dev)

    def sync(self) -> None:
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def reduce(self, vals: list[float]) -> tuple[list[float], list[float]]:
        """(max over ranks, min over ranks) of each value."""
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        lo = t.clone()
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(lo, op=self.dist.ReduceOp.MIN)
        return [float(x) for x in t.tolist()], [float(x) for x in lo.tolist()]

    def timed(self, fn):
        """(device ms, result) of ``fn`` bracketed by barrier + synchronize on both sides, L2 flushed before."""
        torch = self.torch
        self.flush.zero_()
        self.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        self.sync()
        return e0.elapsed_time(e1), out

    def walled(self, fn):
        self.flush.zero_()
        self.sync()
        t0 = time.perf_counter()
        out = fn()
        self.sync()
        return time.perf_counter() - t0, out


# ------------------------------------------------------------------------------------------------------------------ outputs
def param_sample(flat):
    """A flat parameter vector as float32 on the host: whole up to ``DUMP_PARAMS`` elements, else the elements at ``DUMP_PARAMS``
    positions drawn with a fixed seed (sorted, repeats dropped), so the same model size always yields the same positions."""
    import numpy as np
    import torch

    flat = flat.detach().reshape(-1)
    if flat.numel() > DUMP_PARAMS:
        idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), DUMP_PARAMS))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    return flat.float().cpu().numpy()


def fed_outputs(rt, results: list) -> dict:
    """What a caller of one round receives: the new global model and every client's fit result, clients in id order.
    ``num_examples`` is local steps x local batch; the cross-entropy is the mean over the client's local steps."""
    import numpy as np

    failed = [r for r in results if r.status.code != 0]
    if failed:
        raise SystemExit(f"bench round had failed clients: {failed[0].status.message}")
    res = sorted(results, key=lambda r: int(r.cid))
    n_layers = len(rt.model_layout.names)
    return {"global_params": param_sample(rt.round_backend.global_params()),
            "client_num_examples": np.array([r.num_examples for r in res], dtype=np.float64),
            "client_cross_entropy": np.array([r.metrics["LanguageCrossEntropy"] for r in res], dtype=np.float64),
            "client_pseudo_gradient_l2_norm": np.array([r.metrics["client/l2_norm_pseudo_gradient"] for r in res], dtype=np.float64),
            "client_layer_pseudo_gradient_l2_norm": np.array(
                [[r.metrics[f"client/layer/{i}/l2_norm_of_pseudo_gradient"] for i in range(n_layers)] for r in res], dtype=np.float64)}


def ddp_outputs(tr, K: int) -> dict:
    """What a caller of ``Trainer.fit`` receives: the trained parameters (this rank's, when they are sharded) and the loss of each
    of the K steps of the call."""
    import numpy as np

    loss = [v for _, v in tr.loggers[0].data["loss/train/total"][-K:]]
    return {"params": param_sample(tr.state.flat.params), "train_loss": np.array(loss, dtype=np.float64)}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np

    nbytes = sum(a.nbytes for a in arrays.values())
    if nbytes > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {nbytes} bytes exceed the {DUMP_MAX_BYTES} byte budget")
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(d / f"{name}.npy", a)


def run_fed(env: Env, args, impl: str, K: int, W: int) -> dict:
    """Configs #2 / #4 / #5: one federated round of K local steps per client + the round exchange."""
    torch = env.torch
    from photon_b200 import ops
    from photon_b200.federation import FederationRuntime
    from photon_b200.server.broadcast_utils import broadcast_parameters_to_nodes
    from photon_b200.utils.hw import NVLINK_PEER_GBS, measured_peaks

    gpc = 2 if args.mode == "fed4x2" else 1
    n_clients = 4 if args.mode == "fed4x2" else N_CLIENTS
    if env.world % gpc or n_clients % (env.world // gpc):
        raise SystemExit(f"--mode {args.mode}: --gpus must be a multiple of {gpc} dividing {n_clients * gpc}")
    default_mb = LOCAL_BATCH // gpc if args.model == "mpt-125m" else 8
    mb = args.microbatch or (default_mb if impl == "ours" else "auto")
    rt = FederationRuntime(fed_cfg(args, impl, W, n_clients, mb), device=env.dev, rank=env.rank, world_size=env.world, gpus_per_client=gpc)
    rt.build()
    broadcast_parameters_to_nodes(rt, rt.initial_parameters())
    sampled = list(range(n_clients))

    mid = {"ev": None}

    def one_round(server_round: int) -> list:
        res = rt.run_clients_fit(server_round, sampled)       # K local steps on each of this rank's clients
        mid["ev"] = torch.cuda.Event(enable_timing=True)      # this rank's own compute ends here; the round kernel then waits for the slowest peer
        mid["ev"].record()
        rt.finish_round(server_round)                         # aggregate + server optimizer + broadcast
        return res

    one_round(1)                                              # warm-up: a W-step round (workspaces, kernels, arena, CUDA graphs)
    env.sync()
    rt.cfg["llm_config"]["local_steps"] = f"{K}ba"
    if impl == "ours":
        ops.reset_launch_count()
    clk = ClockSampler(env.local, enabled=(env.rank == 0)).start()
    env.flush.zero_()
    env.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = one_round(2)
    e1.record()
    env.sync()
    dev_ms, own_ms = e0.elapsed_time(e1), e0.elapsed_time(mid["ev"])     # whole round / this rank's local training only
    launches = ops.launch_count() if impl == "ours" else 0
    failed = [r for r in res if r.status.code != 0]
    if failed:
        raise SystemExit(f"bench round had failed clients: {failed[0].status.message}")
    e2e_s, res = env.walled(lambda: one_round(3))
    clk.stop()
    outputs = fed_outputs(rt, res) if args.dump_outputs and impl == args.impl else None
    # the round exchange alone (aggregate + server optimizer + broadcast) on a freshly filled accumulator: device time of the
    # transport's launch, and wall clock of the whole public call (adds the host-side status agreement of the control plane)
    def fill() -> None:
        rt.round_backend.begin_round()
        if rt.is_leader:
            rt.round_backend.add_client(rt.trainer.state.flat.params, 1.0)

    fill()
    agg_ms, _ = env.timed(lambda: rt.round_backend.finish_round(4))
    fill()
    agg_host_s, _ = env.walled(lambda: rt.finish_round(5))
    (dev_max, e2e_max, agg_max, agg_host_max, own_max), (dev_min, _, agg_min, _, own_min) = env.reduce([dev_ms, e2e_s, agg_ms, agg_host_s, own_ms])
    total = rt.layout.total
    n_srv = int(rt.strategy.n_moments)     # server moment planes the kernel reads and writes (Nesterov: 1 even with mu = 0, FedAdam: 2)
    if env.world == 1:      # HBM roofline: read the client sum + x (+ moments), write x fp32 + bf16 (+ moments)
        roof_ms = total * (4 + 4 + 4 + 2 + 8 * n_srv) / measured_peaks()["hbm_bytes_per_s"] * 1e3
    else:                   # NVLink roofline: (N-1)/N of the fp32 plane in (reduce) and out again (fp32 + bf16 broadcast), per direction
        roof_ms = total * ((env.world - 1) / env.world) * (4 + 4 + 2) / (NVLINK_PEER_GBS * 1e9) * 1e3
    mcfg = rt.trainer.model_cfg
    out = dict(dev_ms=dev_max, dev_ms_min=dev_min, e2e_s=e2e_max, agg_ms=agg_max, agg_ms_min=agg_min, agg_roofline_ms=roof_ms,
               agg_host_ms=agg_host_max * 1e3, own_ms_min=own_min, own_ms_max=own_max, launches=int(launches), clocks=clk.summary(), tokens=n_clients * K * LOCAL_BATCH * SEQ,
               flops_per_token=float(mcfg.flops_per_token(SEQ)), optimizer=str(rt.cfg["llm_config"]["optimizer"]["name"]),
               comm_stack=rt.round_backend.name, microbatch=int(getattr(rt.trainer, "_auto_mb", None) or rt.trainer.microbatch),
               clients_per_node=n_clients // rt.n_nodes, gpus_per_client=gpc, n_clients=n_clients,
               h2d=(n_clients // rt.n_nodes) * (LOCAL_BATCH // gpc) * SEQ * 8, d2h=(n_clients // rt.n_nodes) * 2 * 8, outputs=outputs)
    rt.close()
    return out


def run_ddp(env: Env, args, impl: str, K: int, W: int) -> dict:
    """Config #3: centralised DDP — K optimizer steps of global batch 256 through ``run_centralised`` / ``Trainer.fit``."""
    torch = env.torch
    from photon_b200 import ops
    from photon_b200.centralised_train import run_centralised
    from photon_b200.parallel.ddp import NcclPerTensorGradComm
    from photon_b200.utils.hw import NVLINK_PEER_GBS

    if DDP_GLOBAL_BATCH % env.world:
        raise SystemExit("--gpus must divide 256")
    per_gpu = DDP_GLOBAL_BATCH // env.world
    # the reference's device_train_microbatch_size: 32 fits MPT-125M, the larger configs use 8 (ref: conf/llm_config/mpt-{1b,3b,7b}.yaml)
    default_mb = min(LOCAL_BATCH if args.model == "mpt-125m" else 8, per_gpu)
    mb = args.microbatch or (default_mb if impl == "ours" else "auto")
    cfg = ddp_cfg(args, impl, mb)
    kw = {}
    if impl != "ours" and env.world > 1:
        kw["grad_comm"] = NcclPerTensorGradComm()     # the reference's FORCED_SYNC: one NCCL all-reduce per parameter tensor
    tr = run_centralised(cfg, device=env.dev, rank=env.rank, world_size=env.world, duration=f"{W}ba", **kw)
    env.sync()
    if impl == "ours":
        ops.reset_launch_count()
    clk = ClockSampler(env.local, enabled=(env.rank == 0)).start()
    dev_ms, _ = env.timed(lambda: tr.fit(duration=f"{K}ba"))
    launches = ops.launch_count() if impl == "ours" else 0
    e2e_s, _ = env.walled(lambda: tr.fit(duration=f"{K}ba"))
    clk.stop()
    outputs = ddp_outputs(tr, K) if args.dump_outputs and impl == args.impl else None
    # the gradient all-reduce alone on the live bucket
    ar_ms = 0.0
    # (fully sharded: reduced per block inside the backward; fused ZeRO-1 step: the reduction is part of the step kernel)
    if env.world > 1 and not getattr(tr.state.flat, "is_sharded", False) and not getattr(tr, "fused_comm_step", False):
        g = tr.state.flat.grads
        for _ in range(3):
            tr._allreduce_grads()  # noqa: SLF001
        ts = []
        for _ in range(5):
            t, _ = env.timed(tr._allreduce_grads)  # noqa: SLF001
            ts.append(t)
        ar_ms = sorted(ts)[len(ts) // 2]
        g.zero_()
    (dev_max, e2e_max, ar_max), (dev_min, _, _) = env.reduce([dev_ms, e2e_s, ar_ms])
    total = tr.state.flat.layout.total
    roof_ms = total * 4 * 2 * ((env.world - 1) / env.world) / (NVLINK_PEER_GBS * 1e9) * 1e3 if env.world > 1 else 0.0
    out = dict(dev_ms=dev_max, dev_ms_min=dev_min, e2e_s=e2e_max, agg_ms=ar_max, agg_ms_min=ar_max, agg_roofline_ms=roof_ms, launches=int(launches),
               clocks=clk.summary(), tokens=K * DDP_GLOBAL_BATCH * SEQ, flops_per_token=float(tr.model_cfg.flops_per_token(SEQ)),
               optimizer="decoupled_adamw", comm_stack=type(tr.grad_comm).__name__ if tr.grad_comm is not None else "none",
               microbatch=int(getattr(tr, "_auto_mb", None) or tr.microbatch), clients_per_node=1, gpus_per_client=env.world, n_clients=1,
               h2d=per_gpu * SEQ * 8, d2h=2 * 8, outputs=outputs)
    free_b, total_b = torch.cuda.mem_get_info(env.dev)
    out["gpu_mem_used_gb"] = round((total_b - free_b) / 2**30, 1)     # whole device, arena planes included (after the run)
    out["torch_peak_alloc_gb"] = round(torch.cuda.max_memory_allocated(env.dev) / 2**30, 1)
    gc_ = tr.grad_comm
    tr.close()
    if gc_ is not None:
        gc_.close()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch"])
    ap.add_argument("--mode", default="fed", choices=["fed", "ddp", "fed4x2"])
    ap.add_argument("--model", default="mpt-125m")
    ap.add_argument("--precision", default="amp_bf16", choices=["amp_bf16", "amp_fp8"])
    ap.add_argument("--attention", default="b200", choices=["b200", "torch"])
    ap.add_argument("--microbatch", type=int, default=0, help="device microbatch (0 = 32 for mpt-125m, 8 otherwise; torch arm: auto)")
    ap.add_argument("--server", default="fedavg", choices=["fedavg", "fedadam"])
    ap.add_argument("--sharding", default="auto", choices=["auto", "none", "zero1", "zero3"],
                    help="ddp mode: none = replicated DDP, zero1 = fused sharded-optimizer step, zero3 = full parameter sharding "
                         "(auto = zero3 for mpt-7b, none otherwise)")
    ap.add_argument("--global-batch", type=int, default=0, help="ddp mode: sequences per optimizer step (default 256, BASELINE config #3)")
    ap.add_argument("--torch-arm", default="auto", choices=["auto", "on", "off"],
                    help="also measure the reference-equivalent stock-PyTorch arm in this invocation (auto = yes for mpt-125m)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps write what the timed path computed in its last step (fed: the new global model and the "
                         "clients' fit results; ddp: the parameters and the step losses) as DIR/<name>.npy, float32 / float64, at most "
                         "64 MiB; parameters of models above 4 Mi of them are a fixed, seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.global_batch:
        global DDP_GLOBAL_BATCH
        DDP_GLOBAL_BATCH = int(args.global_batch)
    if args.impl == "reference":
        reference_arm()
        return
    env = Env(args)
    K, W = args.steps, max(args.warmup, 3)
    run = run_ddp if args.mode == "ddp" else run_fed
    t_ours = time.time()
    r = run(env, args, args.impl, K, W)
    t_ours = time.time() - t_ours
    if args.dump_outputs and env.rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"])

    def emit(torch_arm) -> None:
        if env.rank == 0:
            print(json.dumps(result_line(env, args, r, K, W, torch_arm)), flush=True)

    torch_arm = None
    want_torch = args.impl == "ours" and (args.torch_arm == "on" or (args.torch_arm == "auto" and args.model == "mpt-125m"))
    if want_torch:
        # The stand-in arm must never cost the headline: if it hangs (e.g. one rank failing while the others sit in a collective)
        # a watchdog prints OUR line without it and ends every rank.
        import threading

        def bail() -> None:
            emit({"error": "the stock-PyTorch arm did not finish within its time limit; headline printed without it"})
            os._exit(0)

        dog = threading.Timer(min(420.0, max(180.0, 8.0 * t_ours)), bail)     # bounded: the whole invocation stays far below the driver's limit
        dog.daemon = True
        dog.start()
        gc.collect()
        env.torch.cuda.empty_cache()
        try:
            t = run(env, args, "torch", K, W)
            torch_arm = {"value": t["tokens"] / (t["dev_ms"] / 1e3), "ms_per_step": t["dev_ms"] / K, "e2e_value": t["tokens"] / t["e2e_s"],
                         "exchange_ms": t["agg_ms"], "microbatch": t["microbatch"], "comm_stack": t["comm_stack"],
                         "what": "stock PyTorch ops (cuBLAS, SDPA, ATen, torch optimizer) + the reference's communication pattern, same K and batch"}
        except Exception as e:  # noqa: BLE001 - the stand-in arm must never take the headline down
            torch_arm = {"error": f"{type(e).__name__}: {e}"[:300]}
        dog.cancel()
    emit(torch_arm)
    if env.world > 1:
        env.dist.destroy_process_group()


def result_line(env, args, r: dict, K: int, W: int, torch_arm) -> dict:
    from photon_b200.utils.hw import measured_peaks

    if True:
        world = env.world
        value = r["tokens"] / (r["dev_ms"] / 1e3)
        peak = measured_peaks()
        model = MODEL_NAMES.get(args.model, args.model)
        metric = {"fed": f"tokens/sec (whole box, device-timed, max over ranks) {model} 8-client fed round",
                  "ddp": f"tokens/sec (whole box, device-timed, max over ranks) {model} centralised_train DDP global batch {DDP_GLOBAL_BATCH}",
                  "fed4x2": f"tokens/sec (whole box, device-timed, max over ranks) {model} 4 clients x 2 GPUs fed round"}[args.mode]
        par = {"fed": f"fed{N_CLIENTS}clients_on_{world}gpu", "ddp": f"dp{world}", "fed4x2": f"fed4clients_x_dp2_on_{world}gpu"}[args.mode]
        exch = "round_aggregate_broadcast_ms" if args.mode != "ddp" else "allreduce_ms"
        out = {
            "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": r["dev_ms"] / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "fp8 GEMMs (E4M3/E5M2, fp32 accumulate) + bf16" if args.precision == "amp_fp8" else "bf16",
            "data": "synthetic C4-shaped tokens, random-init weights", "impl": args.impl,
            "config": {"model": args.model, "mode": args.mode, "global_batch": DDP_GLOBAL_BATCH if args.mode == "ddp" else r["n_clients"] * LOCAL_BATCH,
                       "seq_len": SEQ, "parallelism": par, "clients_per_gpu_group": r["clients_per_node"], "gpus_per_client": r["gpus_per_client"],
                       "local_steps_per_round": K if args.mode != "ddp" else None, "local_batch": LOCAL_BATCH if args.mode != "ddp" else None,
                       "microbatch": r["microbatch"], "precision": args.precision, "optimizer": r["optimizer"],
                       "server": None if args.mode == "ddp" else ("fedavg(nesterov lr=1 mu=0)" if args.server == "fedavg" else "fedadam"),
                       "comm_stack": r["comm_stack"], "attention": args.attention if args.impl == "ours" else "sdpa",
                       "l2_flush": "256 MiB memset before each timed region; per-step activations (~19 GB) exceed L2",
                       "timed_region": "K optimizer steps" if args.mode == "ddp" else "one full round: K local steps x clients + aggregate + server-opt + broadcast"},
            exch: r["agg_ms"], exch.replace("_ms", "_roofline_ms"): r["agg_roofline_ms"],
            exch.replace("_ms", "_roofline_fraction"): (r["agg_roofline_ms"] / r["agg_ms"]) if r["agg_ms"] > 0 else None,
            **({"round_exchange_wall_ms_incl_host_agreement": r["agg_host_ms"]} if "agg_host_ms" in r else {}),
            "rank_dev_ms": {"min": r["dev_ms_min"], "max": r["dev_ms"], "spread_pct": 100.0 * (r["dev_ms"] - r["dev_ms_min"]) / r["dev_ms"]},
            **({"rank_local_training_ms": {"min": r["own_ms_min"], "max": r["own_ms_max"],
                                           "straggler_pct": 100.0 * (r["own_ms_max"] - r["own_ms_min"]) / r["own_ms_max"],
                                           "note": "device time of each rank's own K local steps (before the round kernel's start barrier makes everyone wait for the slowest)"}}
               if "own_ms_max" in r else {}),
            "mfu_of_measured_bf16_peak": value / world * r["flops_per_token"] / peak["bf16_flops"],
            "clocks": r["clocks"],
            "e2e": {"value": r["tokens"] / r["e2e_s"], "unit": "tokens/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "api": "Trainer.fit via run_centralised (wall clock)" if args.mode == "ddp" else "FederationRuntime.run_clients_fit + finish_round (wall clock)"},
            "gpu_launches": r["launches"],
        }
        if "gpu_mem_used_gb" in r:
            out["memory"] = {"gpu_mem_used_gb": r["gpu_mem_used_gb"], "torch_peak_alloc_gb": r["torch_peak_alloc_gb"],
                             "note": "device memory in use after the run (arena planes included) / peak of the torch allocator"}
        if torch_arm is not None:
            out["torch_arm"] = torch_arm
            if "value" in torch_arm:
                out["vs_torch_arm"] = value / torch_arm["value"]
                out["e2e_vs_torch_arm"] = out["e2e"]["value"] / torch_arm["e2e_value"]
        return out


if __name__ == "__main__":
    main()
