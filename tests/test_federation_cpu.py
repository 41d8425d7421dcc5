"""Federation plumbing on CPU: SPMD runtime end to end (resume, fault injection, transports),
node manager + worker processes over shm, plumbing config #1, gloo world_size 2."""
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest
import torch

from photon_b200.config import compose
from conftest import free_port as _free_port  # noqa: E402

TINY = ["llm_config.model.d_model=32", "llm_config.model.n_heads=2", "llm_config.model.n_layers=1", "llm_config.max_seq_len=16",
        "llm_config.global_train_batch_size=4", "llm_config.device_train_microbatch_size=2", "llm_config.device_eval_batch_size=4",
        "llm_config.local_steps=2ba", "llm_config.precision=fp32", "llm_config.model.attn_config.attn_impl=torch",
        "llm_config.eval_subset_num_batches=1", "llm_config.log_to_console=false", "~llm_config.loggers.wandb", "~llm_config.loggers.tensorboard",
        "~llm_config.callbacks", "llm_config.optimizer.lr=1.0e-2", "llm_config.scheduler.schedulers.lr.t_warmup=1ba",
        "fl.n_total_clients=4", "fl.n_clients_per_round=2", "photon.resume_round=null"]


def _cfg(tmp, *extra):
    return compose(TINY + [f"photon.saving_path={tmp}", f"llm_config.save_folder={tmp}/clients", "llm_config.save_interval=2ba", *extra])


def test_federated_rounds_checkpoint_and_resume(tmp_path):
    from photon_b200.checkpoint import CheckpointStore
    from photon_b200.server_app import run_server

    cfg = _cfg(tmp_path, "run_uuid=r1", "photon.checkpoint=true", "fl.n_rounds=2", "fl.strategy_name=fedadam",
               "fl.strategy_kwargs={eta: 0.01, beta_1: 0.9, beta_2: 0.99, tau: 0.001}")
    h = run_server(cfg)
    assert [r for r, _ in h.metrics_distributed_fit["server/l2_norm_pseudo_gradient"]] == [1, 2]
    assert len(h.losses_distributed) == 3                      # eval at round 0, 1, 2
    store = CheckpointStore(tmp_path, "checkpoints")
    keys = ["current_server_parameters", "current_momentum_vector", "current_second_momentum_vector"]
    assert store.obtain_sorted_rounds("r1", keys) == [0, 1, 2]
    with np.load(store.round_dir("r1", 2) / "current_server_parameters.npz") as z:
        assert len(z.files) == 16 and z["arr_0"].shape == (96,)     # arr_0 = transformer.blocks.0.attn.Wqkv.bias (sorted names)
    # resume: 2 more rounds continue from round 2 with replayed sampling and restored steps
    cfg2 = _cfg(tmp_path, "run_uuid=r1", "photon.checkpoint=true", "fl.n_rounds=4", "photon.resume_round=-1", "fl.strategy_name=fedadam",
                "fl.strategy_kwargs={eta: 0.01, beta_1: 0.9, beta_2: 0.99, tau: 0.001}")
    h2 = run_server(cfg2)
    assert [r for r, _ in h2.metrics_distributed_fit["server/l2_norm_pseudo_gradient"]] == [1, 2, 3, 4]
    assert store.obtain_sorted_rounds("r1", keys) == [0, 1, 2, 3, 4]
    # an uninterrupted 4-round run must sample the same clients in rounds 3-4 (RNG replay)
    import random

    rng = random.Random(1337)
    expect = [rng.sample(range(4), 2) for _ in range(4)]
    from photon_b200.federation import FederationRuntime

    rt = FederationRuntime(cfg2, device=torch.device("cpu"), rank=0, world_size=1)
    rt.replay_sampling(2)
    assert [rt.sample_clients(), rt.sample_clients()] == expect[2:]
    # and the resumed federation is bit-identical to one that never stopped (server moments, client clocks, data positions)
    cfg3 = _cfg(tmp_path / "straight", "run_uuid=r1", "photon.checkpoint=true", "fl.n_rounds=4", "fl.strategy_name=fedadam",
                "fl.strategy_kwargs={eta: 0.01, beta_1: 0.9, beta_2: 0.99, tau: 0.001}")
    run_server(cfg3)
    a = np.load(store.round_dir("r1", 4) / "current_server_parameters.npz")
    b = np.load(CheckpointStore(tmp_path / "straight", "checkpoints").round_dir("r1", 4) / "current_server_parameters.npz")
    assert all(np.array_equal(a[k], b[k]) for k in a.files)


def test_fault_injection_accept_and_ignore(tmp_path):
    from photon_b200.server.fit_utils import TooManyFailuresError
    from photon_b200.server_app import run_server

    base = ["run_uuid=f1", "fl.n_rounds=1", "fl.n_clients_per_round=4", "fl.eval_period=null", "fl.fault_injection={round: 1, cid: 2, kind: drop}"]
    with pytest.raises(TooManyFailuresError):
        run_server(_cfg(tmp_path, *base))
    h = run_server(_cfg(tmp_path, *base, "fl.accept_failures_cnt=1"))          # survivors are aggregated
    assert h.latest("server/n_failures") == 1 and h.latest("server/l2_norm_pseudo_gradient") > 0
    h = run_server(_cfg(tmp_path, *base, "fl.ignore_failed_rounds=true"))       # round skipped, model kept
    assert h.latest("server/round_ignored") == 1


@pytest.mark.parametrize("stack", ["shm", "ray", "s3"])
def test_transports_agree(tmp_path, stack):
    from photon_b200.server_app import run_server
    from photon_b200.federation import FederationRuntime

    outs = {}
    for s in ("shm", stack):
        cs = {k: (k == s) for k in ("s3", "shm", "ray", "nvl")}
        cfg = _cfg(tmp_path / s, f"run_uuid=t-{s}", "fl.n_rounds=2", "fl.eval_period=null",
                   *[f"photon.comm_stack.{k}={str(v).lower()}" for k, v in cs.items()])
        rt = FederationRuntime(cfg, device=torch.device("cpu"), rank=0, world_size=1)
        run_server(cfg, runtime=rt)
        outs[s] = rt.round_backend.global_params().clone()
        rt.close()
    assert torch.allclose(outs["shm"], outs[stack], atol=1e-6)


def test_plumbing_config_1_mpt125m_one_cpu_step(tmp_path):
    """BASELINE config #1: MPT-125M centralised_train, fp32, attn_impl=torch, 1 step on CPU, synthetic tokens."""
    from photon_b200.centralised_train import run_centralised

    cfg = compose(["run_uuid=plumb", "llm_config.precision=fp32", "llm_config.model.attn_config.attn_impl=torch",
                   "llm_config.global_train_batch_size=1", "llm_config.device_train_microbatch_size=1", "llm_config.max_seq_len=256",
                   "llm_config.log_to_console=false", "~llm_config.loggers.wandb", "~llm_config.loggers.tensorboard", "~llm_config.callbacks",
                   "llm_config.save_folder=null", "dataset/streams@dataset.train.streams=centralised", "centralized.store_final_model=false"])
    tr = run_centralised(cfg, device=torch.device("cpu"), rank=0, world_size=1, duration="1ba")
    assert tr.state.flat.layout.n_params == 125_311_488 - (2048 - 256) * 768 and len(tr.state.flat.names) == 148
    loss = tr.state.train_metric_values["LanguageCrossEntropy"]
    assert 9.0 < loss < 13.0 and tr.state.timestamp.batch == 1
    tr.close()


def test_node_manager_workers_over_shm(tmp_path):
    from photon_b200.client_app import ClientApp
    from photon_b200.clients.configs import get_photon_fit_config_fn
    from photon_b200.clients.utils import get_initial_parameters
    from photon_b200.messages import ClientState, Code, Message
    from photon_b200.server.server_util import fit_or_evaluate_ins

    cfg = _cfg(tmp_path, "run_uuid=nm", "llm_config.save_folder=null")
    arrays, layout = get_initial_parameters(cfg)
    app = ClientApp(cfg, n_workers=1)
    with app.lifespan():
        ack = app.handle(Message("query", {"type": "broadcast_parameters", "parameters": arrays}))
        assert ack.content == {"broadcast": {"status": "OK"}}
        fn = get_photon_fit_config_fn(cfg)
        states = {c: ClientState() for c in range(4)}
        msg = fit_or_evaluate_ins("train", 1, [0, 3], states, 0, {c: fn(1, c, states, 0).to_wire() for c in (0, 3)})
        reply = app.handle(msg)
        res = reply.content
        assert [r.cid for r in res] == [0, 3] and all(r.status.code == Code.OK and r.num_examples == 8 for r in res)
        new = res[0].parameters.data
        assert len(new) == len(arrays) and any(not np.array_equal(a, b) for a, b in zip(new, arrays))
        assert "client/l2_norm_pseudo_gradient" in res[0].metrics
        # a failing worker is reported, the pool is rebuilt and the retry succeeds
        res2 = app.nm.fit({1: {"fit_config": fn(1, 1, states, 0).to_wire(), "inject_failure": True}})
        assert res2[0].status.code == Code.OK and all(w.is_alive() for w in app.nm.workers)
        # a worker that hangs (alive, silent) is caught by photon.task_timeout_s: pool torn down, respawned, client retried
        app.nm.task_timeout_s = 15.0   # must exceed a respawn + one tiny fit (worker start-up imports torch)
        old_pids = [w.pid for w in app.nm.workers]
        res3 = app.nm.fit({2: {"fit_config": fn(1, 2, states, 0).to_wire(), "inject_hang": True}})
        assert res3[0].status.code == Code.OK and [w.pid for w in app.nm.workers] != old_pids


def test_two_rank_gloo_federation(tmp_path):
    """world_size=2 over gloo: SPMD runtime with the collective transport; both ranks end with the same model."""
    script = tmp_path / "run.py"
    script.write_text(textwrap.dedent(f"""
        import os, sys, torch, torch.distributed as dist
        sys.path.insert(0, {str(Path(__file__).resolve().parents[1])!r})
        from photon_b200.config import compose
        from photon_b200.federation import FederationRuntime
        from photon_b200.server_app import run_server
        dist.init_process_group("gloo")
        cfg = compose({TINY!r} + ["run_uuid=g2", "fl.n_rounds=2", "fl.eval_period=null", "photon.comm_stack.shm=false", "photon.comm_stack.ray=true",
                                "llm_config.save_folder=null", "fl.n_clients_per_round=4", "fl.use_noise_scale_metric=true",
                                "fl.strategy_kwargs={{server_learning_rate: 1.0, server_momentum: 0.0, track_inplace_aggregation: true}}"])
        rt = FederationRuntime(cfg, device=torch.device("cpu"), rank=dist.get_rank(), world_size=2)
        h = run_server(cfg, runtime=rt)
        x = rt.round_backend.global_params().clone()
        ref = x.clone(); dist.broadcast(ref, src=0)
        assert torch.equal(x, ref)
        if dist.get_rank() == 0:
            fit = h.metrics_distributed_fit
            assert [v for _, v in fit["noise_scale/b_big"]] == [4, 4]          # per-client statistics reduced over both ranks
            assert all(v < 1e-4 for _, v in fit["server/l2_norm_fedavg_gap"])   # transport aggregate == textbook mean
            print("OK", float(x.norm()))
        dist.destroy_process_group()
    """))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", str(_free_port()), str(script)], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and "OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]


@pytest.mark.parametrize("extra,check", [
    (["fl.aggregate_momenta=true", "fl.reset_optimizer=false", "llm_config.optimizer.name=decoupled_adamw"], "momenta"),
    (["fl.personalized_layers=[transformer.wpe.weight]"], "personalized"),
    (["fl.random_layers=[transformer.blocks.0.ffn.up_proj.weight]", "fl.random_init_freq=1"], "random"),
    (["fl.frozen_layers=[transformer.wpe.weight]", "fl.split_eval=true"], "frozen"),
])
def test_client_side_model_surgery_features(tmp_path, extra, check):
    """SURVEY App. B features run end to end through the round loop (ref: clients/utils.py:405-652)."""
    from photon_b200.federation import FederationRuntime
    from photon_b200.server_app import run_server

    cfg = _cfg(tmp_path, f"run_uuid=s-{check}", "fl.n_rounds=2", "fl.n_clients_per_round=2", *extra)
    rt = FederationRuntime(cfg, device=torch.device("cpu"), rank=0, world_size=1)
    h = run_server(cfg, runtime=rt)
    fit = h.metrics_distributed_fit
    assert [r for r, _ in fit["server/l2_norm_pseudo_gradient"]] == [1, 2]
    assert all(np.isfinite(v) for _, v in fit["server/l2_norm_model"])
    if check == "momenta":
        # three planes travelled: [params | exp_avg | exp_avg_sq]; the aggregated Adam moments are non-zero after a round
        total = rt.model_layout.total
        g = rt.round_backend.global_params()
        assert g.numel() == 3 * total == rt.layout.total and len(rt.layout.names) == 3 * len(rt.model_layout.names)
        assert float(g[total:2 * total].abs().sum()) > 0 and float(g[2 * total:].min()) >= 0 and float(g[2 * total:].sum()) > 0
        assert any("exp_avg" in k or "momentum" in k for k in fit if k.startswith("client/"))
    if check == "frozen":
        assert "transformer.wpe.weight" not in rt.layout.names
        assert len(h.losses_distributed) >= 2
    rt.close()


_MATRIX = {
    "noise_scale+unigram": ["fl.use_noise_scale_metric=true", "fl.use_unigram_metrics=true"],
    "resize_vocab+eval_every_round": ["fl.resize_vocab=96", "fl.eval_period=1"],
    "fedmom": ["fl.strategy_name=fedmom", "fl.strategy_kwargs={server_learning_rate: 1.0, server_momentum: 0.5}"],
    "fedyogi": ["fl.strategy_name=fedyogi"],
    "sqrt_scaling+gap_metric": ["fl.strategy_kwargs={server_learning_rate: 1.0, server_momentum: 0.0, scaling_fn: sqrt, track_inplace_aggregation: true}"],
    "per_round_cleanup": ["photon.checkpoint=true", "cleanup_checkpoints_per_round=true"],
    "rope+qk_ln+clip": ["++llm_config.model.attn_config.rope=true", "++llm_config.model.learned_pos_emb=false",
                        "++llm_config.model.attn_config.qk_ln=true", "++llm_config.model.attn_config.clip_qkv=0.5"],
    "alibi+no_bias": ["++llm_config.model.attn_config.alibi=true", "++llm_config.model.learned_pos_emb=false", "++llm_config.model.no_bias=true"],
    "sqrt_cooldown+adamw": ["llm_config.scheduler.schedulers.lr.name=constant_with_sqrt_cooldown_with_warmup",
                            "++llm_config.scheduler.schedulers.lr.t_cooldown=1ba", "~llm_config.scheduler.schedulers.lr.alpha_f",
                            "llm_config.optimizer.name=decoupled_adamw"],
    "keep_optimizer+reset_timestamp": ["fl.reset_optimizer=false", "fl.reset_timestamp=true", "llm_config.save_overwrite=true"],
    "more_clients_than_nodes": ["fl.n_total_clients=8", "fl.n_clients_per_round=5"],
}


@pytest.mark.parametrize("name", sorted(_MATRIX))
def test_option_matrix_runs_two_clean_rounds(tmp_path, name):
    """Every documented ``fl.*`` / ``llm_config.*`` switch combination runs two federated rounds without a client failure."""
    from photon_b200.server_app import run_server

    h = run_server(_cfg(tmp_path, "run_uuid=mx", "fl.n_rounds=2", *_MATRIX[name]))
    fit = h.metrics_distributed_fit
    assert [v for _, v in fit["server/n_failures"]] == [0, 0]
    assert [r for r, _ in fit["server/l2_norm_pseudo_gradient"]] == [1, 2]
    assert len(h.losses_distributed) == 3 and all(np.isfinite(v) for _, v in h.losses_distributed)
    if "gap_metric" in name:
        assert all(v < 1e-4 for _, v in fit["server/l2_norm_fedavg_gap"])
    if "noise_scale" in name:
        assert any(k.startswith("noise_scale/") for k in fit) and any("Unigram" in k for k in fit)


def test_centralised_warm_starts_and_federation_restores(tmp_path, monkeypatch):
    """``store_*_model`` → ``pretrained_model_path`` / ``wte_parameters_path`` / ``eval_only`` in a second centralised run,
    ``photon.restore_cent_run_uuid`` seeding a federation, and ``photon.restore_run_uuid`` importing another run's round
    (ref: centralised_train.py:98-166, server/init_utils.py:43-125, server/s3_utils.py:275-345)."""
    from photon_b200.centralised_train import run_centralised
    from photon_b200.checkpoint import CheckpointStore
    from photon_b200.federation import FederationRuntime
    from photon_b200.server_app import run_server
    from photon_b200.utils.core import load_model_parameters_from_file

    monkeypatch.chdir(tmp_path)
    cen = [a for a in TINY if not a.startswith(("fl.", "llm_config.local_steps"))] + [f"photon.saving_path={tmp_path}", "llm_config.save_folder=null"]
    a = run_centralised(compose(cen + ["run_uuid=cA", "centralized.store_init_model=true", "centralized.store_final_model=true"]),
                        device=torch.device("cpu"), duration="3ba")
    final = tmp_path / "cA-3-checkpoint.npz"
    assert (tmp_path / "cA-0-checkpoint.npz").exists() and final.exists()
    trained = load_model_parameters_from_file(final)
    assert all(np.array_equal(x, y) for x, y in zip(trained, a.state.flat.to_ndarrays()))
    a.close()
    # eval-only run on the trained weights: no optimizer step, weights untouched
    b = run_centralised(compose(cen + ["run_uuid=cB", f"pretrained_model_path={final}", "centralized.eval_only=true"]), device=torch.device("cpu"))
    assert b.state.timestamp.batch == 0 and all(np.array_equal(x, y) for x, y in zip(trained, b.state.flat.to_ndarrays()))
    assert "eval/LanguageCrossEntropy" in b.state.eval_metric_values
    b.close()
    # embedding transplant: everything fresh except wte, which comes from the donor file
    c = run_centralised(compose(cen + ["run_uuid=cC", f"wte_parameters_path={final}", "centralized.eval_only=true", "llm_config.seed=99"]),
                        device=torch.device("cpu"))
    names = list(c.state.flat.names)
    got = c.state.flat.to_ndarrays()
    i = names.index("transformer.wte.weight")
    assert np.array_equal(got[i], trained[i]) and not np.array_equal(got[i - 1], trained[i - 1])
    c.close()
    # a federation seeded from the centralised run starts at its weights (round-0 checkpoint proves it)
    fed = _cfg(tmp_path, "run_uuid=fA", "photon.checkpoint=true", "fl.n_rounds=1", "photon.restore_cent_run_uuid=cA", "photon.restore_cent_run_batches=3")
    run_server(fed)
    store = CheckpointStore(tmp_path, "checkpoints")
    r0 = load_model_parameters_from_file(store.round_dir("fA", 0) / "current_server_parameters.npz")
    assert all(np.array_equal(x, y) for x, y in zip(r0, trained))
    # a NEW run importing fA's last round continues from round 1 → runs only round 2
    fed2 = _cfg(tmp_path, "run_uuid=fB", "photon.checkpoint=true", "fl.n_rounds=2", "photon.restore_run_uuid=fA", "photon.resume_round=-1")
    h = run_server(fed2)
    assert [r for r, _ in h.metrics_distributed_fit["server/l2_norm_pseudo_gradient"]][-1] == 2
    assert store.obtain_sorted_rounds("fB", ["current_server_parameters", "current_momentum_vector"])[-2:] == [1, 2]
    r1a = load_model_parameters_from_file(store.round_dir("fA", 1) / "current_server_parameters.npz")
    r1b = load_model_parameters_from_file(store.round_dir("fB", 1) / "current_server_parameters.npz")
    assert all(np.array_equal(x, y) for x, y in zip(r1a, r1b))


def test_node_fleet_topology_matches_spmd_runtime(tmp_path):
    """``photon.topology=nodes``: server → 2 ClientApps → NodeManagers → worker processes, work queue over 3 sampled
    clients, broadcast over the shm side channel, streaming aggregation — and the same global model as the SPMD runtime."""
    from photon_b200.federation import FederationRuntime
    from photon_b200.server.fleet import NodeFleetRuntime, split_devices
    from photon_b200.server_app import run_server

    assert split_devices(8, 3) == [[0, 1, 2], [3, 4, 5], [6, 7]] and split_devices(0, 2) == [None, None]
    common = ["fl.n_rounds=2", "fl.n_clients_per_round=3", "llm_config.save_folder=null", "fl.strategy_name=fedavg"]
    cfg = _cfg(tmp_path / "a", "run_uuid=fleet", "photon.topology=nodes", "photon.n_nodes=2", *common)
    rt = NodeFleetRuntime(cfg)
    try:
        h = run_server(cfg, runtime=rt)
        fit = h.metrics_distributed_fit
        assert [v for _, v in fit["server/n_failures"]] == [0, 0] and [v for _, v in fit["server/n_nodes"]] == [2, 2]
        assert len(h.losses_distributed) == 3 and "node_training_time_s" in fit
        x_nodes = rt.round_backend.global_params().clone()
    finally:
        rt.close()
    cfg2 = _cfg(tmp_path / "b", "run_uuid=spmd", *common)
    rt2 = FederationRuntime(cfg2, device=torch.device("cpu"), rank=0, world_size=1)
    run_server(cfg2, runtime=rt2)
    x_spmd = rt2.round_backend.global_params()
    assert torch.allclose(x_nodes, x_spmd, atol=1e-5), float((x_nodes - x_spmd).abs().max())
    rt2.close()


def test_node_fleet_two_workers_collaborate_on_one_client(tmp_path):
    """All workers of a node train ONE client together (intra-client DDP over gloo here, NCCL/NVLink on GPUs)."""
    from photon_b200.server.fleet import NodeFleetRuntime
    from photon_b200.server_app import run_server

    cfg = _cfg(tmp_path, "run_uuid=f2", "photon.topology=nodes", "fl.n_rounds=1", "fl.n_clients_per_round=2", "llm_config.save_folder=null")
    rt = NodeFleetRuntime(cfg, n_nodes=1, workers_per_node=2)
    try:
        h = run_server(cfg, runtime=rt)
        assert h.metrics_distributed_fit["server/n_failures"] == [(1, 0)] and len(h.losses_distributed) == 2
        assert len(rt.apps[0].nm.workers) == 2 and all(w.is_alive() for w in rt.apps[0].nm.workers)
    finally:
        rt.close()


def test_centralised_autoresume_continues_from_latest_checkpoint(tmp_path, monkeypatch):
    """A restarted centralised run picks up ``latest-rank0.pt`` (weights, optimizer, clock, data position) and only trains
    the remaining batches; the result equals an uninterrupted run (ref: Composer autoresume, trainer_utils.py:437-450)."""
    from photon_b200.centralised_train import run_centralised

    monkeypatch.chdir(tmp_path)
    cen = [a for a in TINY if not a.startswith(("fl.", "llm_config.local_steps"))] + [
        f"photon.saving_path={tmp_path}", "llm_config.save_interval=1ba", "llm_config.scheduler.schedulers.lr.t_max=5ba"]
    a = run_centralised(compose(cen + ["run_uuid=ar", f"llm_config.save_folder={tmp_path}/ar", "llm_config.max_duration=3ba"]), device=torch.device("cpu"))
    assert a.state.timestamp.batch == 3
    a.close()
    b = run_centralised(compose(cen + ["run_uuid=ar", f"llm_config.save_folder={tmp_path}/ar", "llm_config.max_duration=5ba"]), device=torch.device("cpu"))
    assert b.state.timestamp.batch == 5 and b.fit_start_batch == 3      # resumed at 3, trained 2
    import json

    from photon_b200.centralised_train import dump_metrics

    rec = json.loads(dump_metrics(b, tmp_path / "m.json").read_text())
    assert rec["timestamp"]["batch"] == 5 and [s for s, _ in rec["metrics"]["loss/train/total"]] == [4, 5]
    resumed = b.state.flat.params.clone()
    b.close()
    c = run_centralised(compose(cen + ["run_uuid=one", f"llm_config.save_folder={tmp_path}/one", "llm_config.max_duration=5ba"]), device=torch.device("cpu"))
    assert torch.allclose(resumed, c.state.flat.params, atol=1e-6), float((resumed - c.state.flat.params).abs().max())
    c.close()


def test_runs_from_the_reference_yaml_tree(tmp_path):
    """A user of the reference can point this framework at THEIR config directory: the composer resolves the reference's
    defaults lists / interpolations / schema, and both entry points run from it (keys that only exist here take defaults).
    The directory is the reference's ``photon/conf`` YAML tree, stored under ``tests/golden/reference_conf``."""
    from photon_b200.centralised_train import run_centralised
    from photon_b200.server_app import run_server

    ref = str(Path(__file__).resolve().parent / "golden" / "reference_conf")
    for size, d, opt in (("mpt-125m", 768, "adopt"), ("mpt-1b", 2048, "decoupled_adamw"), ("mpt-3b", 2560, "decoupled_adamw"), ("mpt-7b", 4096, "decoupled_adamw")):
        c = compose([f"llm_config={size}"], config_dir=ref)
        assert c.llm_config.model.d_model == d and c.llm_config.optimizer.name == opt and c.photon.comm_stack.nvl is False
    cfg = compose(TINY + [f"photon.saving_path={tmp_path}", f"llm_config.save_folder={tmp_path}/clients", "run_uuid=refconf", "fl.n_rounds=1",
                          "photon.checkpoint=true"], config_dir=ref)
    h = run_server(cfg)
    assert h.metrics_distributed_fit["server/n_failures"] == [(1, 0)] and len(h.losses_distributed) == 2
    cen = [a for a in TINY if not a.startswith(("fl.", "llm_config.local_steps"))]
    tr = run_centralised(compose(cen + [f"photon.saving_path={tmp_path}", "llm_config.save_folder=null", "run_uuid=refcen",
                                        "llm_config.max_duration=2ba"], config_dir=ref), device=torch.device("cpu"))
    assert tr.state.timestamp.batch == 2
    tr.close()


def test_restore_run_brings_client_checkpoints_along(tmp_path):
    """``photon.restore_run_uuid`` + ``copy_client_checkpoints``: the new run finds the old run's per-client checkpoints under its
    own save folder, so clients keep optimizer state and data position (ref: server/s3_utils.py:1478-1608)."""
    from photon_b200.server_app import run_server

    def cfg_for(uuid, *extra):
        return compose(TINY + [f"photon.saving_path={tmp_path}", f"llm_config.save_folder={tmp_path}/{uuid}/clients", "llm_config.save_interval=2ba",
                               f"run_uuid={uuid}", "photon.checkpoint=true", "fl.reset_optimizer=false", *extra])

    run_server(cfg_for("old", "fl.n_rounds=1"))
    old = sorted(p.relative_to(tmp_path / "old").as_posix() for p in (tmp_path / "old" / "clients").rglob("ep*-rank0.pt"))
    assert old, "the first run wrote no client checkpoints"
    h = run_server(cfg_for("new", "fl.n_rounds=2", "photon.restore_run_uuid=old", "photon.resume_round=-1"))
    new = sorted(p.relative_to(tmp_path / "new").as_posix() for p in (tmp_path / "new" / "clients").rglob("ep*-rank0.pt"))
    assert set(old) <= set(new)
    assert [r for r, _ in h.metrics_distributed_fit["server/n_failures"]][-1] == 2


def test_round_lost_by_a_server_crash_is_rebuilt_from_client_checkpoints(tmp_path):
    """The server dies after the clients finished round 2 but before the round was checkpointed. On restart round 2 runs again;
    every client finds its ``ba == target`` checkpoint, skips training and returns those weights, so the rebuilt round equals
    the lost one bit for bit (ref: llm_config_functions.py:724-761 skip/resume, llm_client_functions.py:163,207)."""
    import shutil

    from photon_b200.checkpoint import CheckpointStore
    from photon_b200.server_app import run_server

    base = ["run_uuid=mid", "photon.checkpoint=true", "fl.n_clients_per_round=4", "fl.n_rounds=2", "llm_config.save_num_checkpoints_to_keep=-1"]
    run_server(_cfg(tmp_path, *base))
    store = CheckpointStore(tmp_path, "checkpoints")
    with np.load(store.round_dir("mid", 2) / "current_server_parameters.npz") as z:
        want = [z[k] for k in z.files]
    shutil.rmtree(store.round_dir("mid", 2))
    h = run_server(_cfg(tmp_path, *base, "photon.resume_round=-1"))
    with np.load(store.round_dir("mid", 2) / "current_server_parameters.npz") as z:
        assert all(np.array_equal(a, z[k]) for a, k in zip(want, z.files))
    assert h.metrics_distributed_fit["client/fit_time"][-1][1] < 0.05      # nobody trained: the weights came from the checkpoints


def test_killed_server_leaves_no_orphan_workers_and_no_shm_segments(tmp_path):
    """SIGKILL the node-topology server mid-run: its worker processes notice the missing parent, exit on their own and take the
    node manager's /dev/shm segments with them (the reference leaks both)."""
    import signal
    import time

    script = tmp_path / "srv.py"
    script.write_text(textwrap.dedent(f"""
        import sys
        sys.path.insert(0, {str(Path(__file__).resolve().parents[1])!r})
        if __name__ == "__main__":
            from photon_b200.config import compose
            from photon_b200.server.fleet import NodeFleetRuntime
            from photon_b200.server_app import run_server
            cfg = compose({TINY!r} + ["run_uuid=orphan", "photon.topology=nodes", "photon.n_nodes=1", "fl.n_rounds=100000", "fl.eval_period=null",
                                    "llm_config.save_folder=null", "photon.saving_path={tmp_path}"])
            rt = NodeFleetRuntime(cfg)
            rt.build()
            print("NM", rt.apps[0].nm.nm_uuid, " ".join(str(w.pid) for w in rt.apps[0].nm.workers), flush=True)
            run_server(cfg, runtime=rt)
    """))
    proc = subprocess.Popen([sys.executable, str(script)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    try:
        line = ""
        t0 = time.time()
        while not line.startswith("NM ") and time.time() - t0 < 120:
            line = proc.stdout.readline()
        assert line.startswith("NM "), "server did not come up"
        _, nm_uuid, *pids = line.split()
        time.sleep(3.0)                                     # a few rounds in
        assert any(n.startswith(nm_uuid) for n in os.listdir("/dev/shm"))
        proc.send_signal(signal.SIGKILL)
        proc.wait(timeout=30)
        deadline = time.time() + 60
        alive = lambda pid: Path(f"/proc/{pid}").exists() and "zombie" not in Path(f"/proc/{pid}/status").read_text().lower()  # noqa: E731
        while time.time() < deadline and (any(alive(p) for p in pids) or any(n.startswith(nm_uuid) for n in os.listdir("/dev/shm"))):
            time.sleep(0.5)
        assert not any(alive(p) for p in pids), "worker processes outlived the killed server"
        assert not [n for n in os.listdir("/dev/shm") if n.startswith(nm_uuid)], "node-manager segments were left in /dev/shm"
    finally:
        if proc.poll() is None:
            proc.kill()


def test_history_json_dump(tmp_path):
    import json

    from photon_b200.server_app import dump_history, run_server

    h = run_server(_cfg(tmp_path, "run_uuid=hj", "fl.n_rounds=1"))
    rec = json.loads(dump_history(h, tmp_path / "history.json").read_text())
    assert rec["losses_distributed"][0][0] == 0 and rec["metrics_distributed_fit"]["server/n_failures"] == [[1, 0.0]]
    assert "server/round_time" in rec["metrics_centralized"] and "server/broadcast_pre_time" in rec["metrics_centralized"]


def test_round_two_trains_from_the_broadcast_global_not_the_client_checkpoint(tmp_path, monkeypatch):
    """With client checkpoints on (save_folder set, reset_checkpoint=false) the client's checkpoint is loaded BEFORE the round's
    parameters are installed: right before ``fit()`` in every round the trainer holds exactly the broadcast global model, not the
    client's own stale weights (ref order: photon/clients/llm_client_functions.py:126-168)."""
    from photon_b200.federation import FederationRuntime
    from photon_b200.server.broadcast_utils import broadcast_parameters_to_nodes
    from photon_b200.train.trainer import Trainer

    cfg = _cfg(tmp_path, "run_uuid=order", "fl.n_total_clients=2", "fl.n_clients_per_round=2", "fl.strategy_name=fedavg")
    rt = FederationRuntime(cfg, device=torch.device("cpu"), rank=0, world_size=1)
    rt.build()
    broadcast_parameters_to_nodes(rt, rt.initial_parameters())
    seen = []
    real_fit = Trainer.fit

    def spy(self, *a, **k):
        seen.append(bool(torch.equal(self.state.flat.params, rt.round_backend.global_params()[: self.state.flat.layout.total])))
        return real_fit(self, *a, **k)

    monkeypatch.setattr(Trainer, "fit", spy)
    for rnd in (1, 2, 3):
        res = rt.run_clients_fit(rnd, [0, 1])
        assert all(r.status.code == 0 for r in res), [r.status.message for r in res]
        for r in res:
            rt.client_states[r.cid] = rt.client_states[r.cid]
        rt.finish_round(rnd)
        rt.server_steps_cumulative += 2
    assert len(seen) == 6 and all(seen), seen
    assert list((tmp_path / "clients").rglob("*.pt")), "client checkpoints were expected on disk"
    rt.close()


def test_client_state_cache_is_bounded_lru():
    """Per-client optimizer moments kept between participations never grow with the number of clients: device budget, then host
    budget, then the least recently used client is dropped (it restarts from a fresh state, like an unseen client)."""
    from photon_b200.federation import ClientStateCache

    one = 2 * 256 * 4                                     # bytes of one entry (two fp32 planes of 256 elements)
    c = ClientStateCache(device_bytes=0, host_bytes=3 * one)      # CPU box: everything counts as host
    for cid in range(5):
        c.put(cid, torch.full((256,), float(cid)), torch.zeros(256), cid)
    assert len(c) == 3 and 0 not in c and 1 not in c and 4 in c
    m, _, step = c.get(2)                                  # touching 2 makes it the most recent
    assert float(m[0]) == 2.0 and step == 2
    c.put(5, torch.ones(256), torch.ones(256), 5)
    assert 3 not in c and 2 in c and 5 in c               # 3 was the least recently used
    assert c.pop(2)[2] == 2 and 2 not in c
