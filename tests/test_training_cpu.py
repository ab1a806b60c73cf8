"""Integration tests of the CLI entry points on CPU/gloo (torchrun, world_size 2), mirroring the reference's
tests/test_training/test_train.py: checkpoint/resume loss-curve continuity for the plain data-parallel path (atol 1e-3)
and for 2 DiLoCo workers (atol 1e-2), plus the train_diloco_torch entry (BASELINE.json config #1)."""
import os
import pickle
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def free_port() -> int:
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def torchrun(nproc: int, module: str, args: list[str], timeout: int = 900, extra_env: dict | None = None) -> None:
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="2", WANDB_MODE="disabled", **(extra_env or {}))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), "-m", module, *args]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    if res.returncode != 0:
        pytest.fail(f"{' '.join(cmd)}\n{res.stdout[-3000:]}\n{res.stderr[-3000:]}")


BASE = ["--path_model", "2m", "--fake_data", "--no-torch_compile", "--lr", "1e-2", "--per_device_train_batch_size", "4",
        "--total_batch_size", "16", "--seq_length", "64", "--metric_logger_type", "dummy", "--precision", "bf16-mixed",
        "--warmup_steps", "4", "--total_steps", "100"]


def _load(path):
    with open(path, "rb") as f:
        return {d["step"]: (d["Loss"], d["lr"]) for d in pickle.load(f)}


def test_full_shard_gathers_parameters_and_matches_zero2(tmp_path):
    """FULL_SHARD (ZeRO-3: compute weights kept as per-rank shards, all-gathered for forward and again for backward) must
    train exactly like SHARD_GRAD_OP (ZeRO-2): same kernels, same reduction order, only the residency of the weights
    differs (reference: utils.py:138-152 -> FSDP ShardingStrategy)."""
    logs = {}
    for strat in ("SHARD_GRAD_OP", "FULL_SHARD"):          # HYBRID_SHARD takes the same code path as FULL_SHARD
        logs[strat] = f"{tmp_path}/{strat}.pkl"
        torchrun(2, "opendiloco_b200.train_fsdp", BASE + ["--max_steps", "6", "--sharding_strategy", strat, "--project", logs[strat]])
    a = _load(logs["SHARD_GRAD_OP"])
    for strat in ("FULL_SHARD",):
        b = _load(logs[strat])
        assert set(a) == set(b) == set(range(1, 7))
        for s in a:
            assert a[s][0] == b[s][0], f"{strat}: loss at step {s}: {a[s][0]} vs {b[s][0]}"


@pytest.mark.parametrize("sharding", ["NO_SHARD", "SHARD_GRAD_OP", "FULL_SHARD"])
def test_ckpt_resume_data_parallel(tmp_path, sharding):
    ckpt = f"{tmp_path}/ckpt"
    log1, log2 = f"{tmp_path}/log1.pkl", f"{tmp_path}/log2.pkl"
    common = BASE + ["--max_steps", "12", "--sharding_strategy", sharding]
    torchrun(2, "opendiloco_b200.train_fsdp", common + ["--ckpt.path", ckpt, "--ckpt.interval", "4", "--project", log1])
    assert os.path.isfile(f"{ckpt}/model_step_8/global_state_dict.pt") and os.path.isfile(f"{ckpt}/model_step_8/.metadata")
    torchrun(2, "opendiloco_b200.train_fsdp", common + ["--ckpt.path", ckpt, "--ckpt.resume", f"{ckpt}/model_step_8", "--project", log2])
    a, b = _load(log1), _load(log2)
    common_steps = set(a) & set(b)
    assert common_steps == {9, 10, 11, 12}
    for s in common_steps:
        assert np.allclose(a[s][0], b[s][0], atol=1e-3), f"Loss at step {s} is different: {a[s][0]} vs {b[s][0]}"
        assert a[s][1] == b[s][1], f"Lr at step {s} is different"


def test_ckpt_resume_two_diloco_workers(tmp_path):
    """2 DiLoCo workers x 1 rank, H=5, resume from a step that is NOT a multiple of H (the reference silently moves the
    outer anchor in that case; we restore theta_outer and the inner-step phase)."""
    ckpt = f"{tmp_path}/ckpt"
    log1, log2 = f"{tmp_path}/log1.pkl", f"{tmp_path}/log2.pkl"
    hv = ["--hv.local_steps", "5", "--hv.galaxy_size", "2", "--hv.skip_load_from_peers", "--hv.fail_rank_drop", "--hv.matchmaking_time", "1",
          "--total_batch_size", "8", "--max_steps", "16"]
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--ckpt.path", ckpt, "--ckpt.interval", "7", "--project", log1])
    assert os.path.isdir(f"{ckpt}/model_step_7/diloco_rank_0") and os.path.isdir(f"{ckpt}/model_step_7/diloco_rank_1")
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--ckpt.path", ckpt, "--ckpt.resume", f"{ckpt}/model_step_7", "--project", log2])
    a, b = _load(log1), _load(log2)
    common_steps = set(a) & set(b)
    assert common_steps == set(range(8, 17))
    for s in common_steps:
        assert np.allclose(a[s][0], b[s][0], atol=1e-2), f"Loss at step {s} is different: {a[s][0]} vs {b[s][0]}"
        assert a[s][1] == b[s][1]


def test_resume_latest_and_topk(tmp_path):
    ckpt = f"{tmp_path}/ckpt"
    args = BASE + ["--max_steps", "6", "--ckpt.path", ckpt, "--ckpt.interval", "2", "--ckpt.topk", "2", "--project", f"{tmp_path}/l.pkl"]
    torchrun(1, "opendiloco_b200.train_fsdp", args)
    assert sorted(os.listdir(ckpt)) == ["model_step_4", "model_step_6"]
    torchrun(1, "opendiloco_b200.train_fsdp", BASE + ["--max_steps", "8", "--ckpt.path", ckpt, "--ckpt.resume", "--project", f"{tmp_path}/l2.pkl"])
    assert min(_load(f"{tmp_path}/l2.pkl")) == 7


def test_train_diloco_torch_two_workers_gloo(tmp_path):
    """BASELINE.json config #1 in miniature: train_diloco_torch, 2 workers, local_steps=3, CPU/gloo."""
    log = f"{tmp_path}/log.pkl"
    torchrun(2, "opendiloco_b200.train_diloco_torch",
             ["--model-name-or-path", "2m", "--fake-data", "--batch-size", "8", "--per-device-train-batch-size", "4", "--seq-length", "64",
              "--local-steps", "3", "--max-steps", "7", "--lr", "1e-2", "--warmup-steps", "2", "--total-steps", "50",
              "--metric-logger-type", "dummy", "--project", log, "--checkpoint-interval", "6", "--checkpoint-path", f"{tmp_path}/out",
              "--eval-steps", "4", "--log-activations-steps", "5"])
    m = pickle.load(open(log, "rb"))
    assert [d["step"] for d in m] == list(range(1, 8))
    assert m[-1]["effective_step"] == 14 and "eval_loss" in m[3] and any(k.startswith("activation/") for k in m[4])
    assert all(np.isfinite(d["Loss"]) for d in m)


def test_no_wait_strategy_through_the_cli(tmp_path):
    """2 DiLoCo workers with --hv.all_reduce_strategy NO_WAIT: rounds are formed through the board; with both workers
    punctual every round is a full one, so the losses equal the WAIT_FOR_ALL run step by step."""
    la, lb = f"{tmp_path}/wait.pkl", f"{tmp_path}/nowait.pkl"
    hv = ["--hv.local_steps", "3", "--hv.galaxy_size", "2", "--hv.skip_load_from_peers", "--total_batch_size", "8", "--max_steps", "7"]
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--project", la])
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--hv.all_reduce_strategy", "NO_WAIT", "--hv.matchmaking_time", "20",
                                                          "--project", lb])
    a, b = _load(la), _load(lb)
    assert set(a) == set(b) == set(range(1, 8))
    for s in a:
        assert np.allclose(a[s][0], b[s][0], atol=1e-4), f"step {s}: {a[s][0]} vs {b[s][0]}"


def test_training_on_pretokenised_shards(tmp_path):
    """scripts/tokenize_corpus.py (byte-level fallback tokenizer) -> shards -> train_fsdp with --dataset_name_or_path tokens:...:
    the native mmap / prefetch loader feeds the driver, 2 data-parallel ranks read disjoint windows, and the loss falls on
    (highly repetitive) real text."""
    src = tmp_path / "corpus.txt"
    src.write_text("".join(f"the quick brown fox number {i % 7} jumps over the lazy dog again and again.\n" for i in range(600)))
    res = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "tokenize_corpus.py"), "--input", str(src), "--output-dir",
                          str(tmp_path / "tok"), "--tokenizer", "byte", "--shard-tokens", "20000"],
                         env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    assert len(os.listdir(tmp_path / "tok")) >= 2
    log = f"{tmp_path}/tok.pkl"
    args = [a for a in BASE if a != "--fake_data"] + ["--dataset_name_or_path", f"tokens:{tmp_path}/tok/*.tok", "--max_steps", "10",
                                                      "--total_batch_size", "8", "--project", log]
    torchrun(2, "opendiloco_b200.train_fsdp", args)
    losses = _load(log)
    assert set(losses) == set(range(1, 11))
    assert losses[10][0] < losses[1][0] - 1.0


@pytest.mark.parametrize("saved,resumed", [("SHARD_GRAD_OP", "NO_SHARD")])
def test_checkpoint_is_resharded_on_load(tmp_path, saved, resumed):
    """Checkpoints hold flat [lo, hi) slices of the parameter / optimizer arenas, so a run saved under one sharding strategy
    resumes under another (the reference's DCP checkpoints are tied to the FSDP wrapping they were written with)."""
    ckpt = f"{tmp_path}/ckpt"
    log1, log2 = f"{tmp_path}/log1.pkl", f"{tmp_path}/log2.pkl"
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + ["--max_steps", "8", "--sharding_strategy", saved, "--ckpt.path", ckpt,
                                                      "--ckpt.interval", "4", "--project", log1])
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + ["--max_steps", "8", "--sharding_strategy", resumed, "--ckpt.path", ckpt,
                                                      "--ckpt.resume", f"{ckpt}/model_step_4", "--project", log2])
    a, b = _load(log1), _load(log2)
    assert set(a) & set(b) == {5, 6, 7, 8}
    for s in (5, 6, 7, 8):
        assert np.allclose(a[s][0], b[s][0], atol=1e-3), f"Loss at step {s} is different: {a[s][0]} vs {b[s][0]}"
        assert a[s][1] == b[s][1]


@pytest.mark.parametrize("precision", ["fp16-mixed"])
def test_other_precision_modes_run(tmp_path, precision):
    """fp16-mixed drives the GradScaler path (train_fsdp.py:383-405: unscale -> clip -> scaler.step -> update); bf16-mixed is
    what every other CLI test uses and 32-true is covered by the fp32 model tests."""
    log = f"{tmp_path}/p.pkl"
    args = [a for a in BASE]
    args[args.index("--precision") + 1] = precision
    torchrun(1, "opendiloco_b200.train_fsdp", args + ["--max_steps", "4", "--total_batch_size", "8", "--project", log])
    losses = _load(log)
    assert set(losses) == {1, 2, 3, 4} and all(np.isfinite(v[0]) for v in losses.values())


def test_swarm_runs_on_the_native_board(tmp_path):
    """2 DiLoCo workers with ODB_BOARD pointing at the native membership board hosted by this test process: progress records
    and the outer-step handshake go through it (not the c10d store), the run finishes and the board holds the traces."""
    from opendiloco_b200.parallel import rendezvous as rdv

    if not rdv.available():
        pytest.skip("libodbhost.so not built")
    server = rdv.RendezvousServer(0)
    try:
        log = f"{tmp_path}/board.pkl"
        hv = ["--hv.local_steps", "2", "--hv.galaxy_size", "2", "--hv.skip_load_from_peers", "--hv.timeout_waiting_for_peers", "60",
              "--total_batch_size", "8", "--max_steps", "5"]
        torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--project", log], extra_env={"ODB_BOARD": f"odb://127.0.0.1:{server.port}"})
        assert set(_load(log)) == set(range(1, 6))
        board = rdv.RendezvousClient("127.0.0.1", server.port)
        for r in (0, 1):
            rec = board.get(f"llama_progress/worker-{r}")          # tracker prefix = run_id ("llama", train_fsdp.py:300)
            assert rec is not None and rec.decode().count(",") == 3
        assert server.num_keys() >= 4            # progress records + the arrival keys of two outer steps
        board.close()
    finally:
        server.stop()


def test_run_training_sh_launches_two_workers(tmp_path):
    """The launcher contract of the reference (open_diloco/run_training.sh:28-36): ``./run_training.sh <N> <gpus per worker>
    <initial_peer|auto> [train_fsdp flags]`` starts N separate torchrun jobs that meet on one rendezvous address, each logging
    to logs/log<i>.  Two CPU workers, 4 steps, one outer step."""
    # The launcher gives worker i the GPU slice "i"; with one GPU that puts worker 0 on NCCL and worker 1, which sees no GPU,
    # on gloo, and the two never meet.  A ``torchrun`` first on PATH records the slice and hides the GPUs from the workers.
    shim = tmp_path / "bin" / "torchrun"
    shim.parent.mkdir()
    shim.write_text('#!/bin/sh\necho "launcher slice: CUDA_VISIBLE_DEVICES=$CUDA_VISIBLE_DEVICES"\n'
                    f'export CUDA_VISIBLE_DEVICES=\nexec "{sys.executable}" -m torch.distributed.run "$@"\n')
    shim.chmod(0o755)
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="2", WANDB_MODE="disabled", DILOCO_WAIT="1",
               DILOCO_PORT=str(free_port()), PATH=f"{shim.parent}{os.pathsep}{os.environ.get('PATH', '')}")
    args = [a for a in BASE if a != "16"]          # drop the DP total batch; DiLoCo: per-worker batch
    args[args.index("--total_batch_size"):args.index("--total_batch_size") + 1] = ["--total_batch_size", "4"]
    cmd = ["bash", os.path.join(ROOT, "run_training.sh"), "2", "1", "auto", *args, "--hv.local_steps", "2", "--max_steps", "4",
           "--hv.skip_load_from_peers", "--hv.matchmaking_time", "1", "--project", f"{tmp_path}/log.pkl"]
    res = subprocess.run(cmd, env=env, cwd=tmp_path, capture_output=True, text=True, timeout=240)
    logs = {i: open(f"{tmp_path}/logs/log{i}").read() for i in (0, 1)}
    assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-1500:] + logs[0][-2000:] + logs[1][-1500:]
    assert "Training completed." in logs[0] and "Training completed." in logs[1]
    assert all(f"launcher slice: CUDA_VISIBLE_DEVICES={i}\n" in logs[i] for i in (0, 1))
    assert "DiLoCo enabled: 2 workers x 1 GPU(s)" in logs[0]
    assert set(_load(f"{tmp_path}/log.pkl")) == {1, 2, 3, 4}


def test_checkpoint_interchange_with_the_dcp_format(tmp_path):
    """Our flat-shard checkpoint -> the reference's DCP layout (ckpt_utils.py:48-100: dcp.save of {"model", "optimizer"} +
    global_state_dict.pt) -> back: weights, Adam moments, step, outer momentum survive the round trip, and the DCP directory
    loads with plain ``dcp.load`` into HF-named tensors."""
    import torch
    import torch.distributed.checkpoint as dcp

    from opendiloco_b200.models.config import LlamaConfig
    from opendiloco_b200.utils.ckpt import _load
    from opendiloco_b200.utils.dcp_interop import export_dcp, import_dcp

    ckpt = f"{tmp_path}/ckpt"
    hv = ["--hv.local_steps", "2", "--hv.galaxy_size", "2", "--hv.skip_load_from_peers", "--hv.matchmaking_time", "1",
          "--total_batch_size", "8", "--max_steps", "4"]
    torchrun(2, "opendiloco_b200.train_fsdp", BASE + hv + ["--ckpt.path", ckpt, "--ckpt.interval", "4", "--project", f"{tmp_path}/l.pkl"])
    src = f"{ckpt}/model_step_4/diloco_rank_0"
    export_dcp(src, f"{tmp_path}/dcp")
    assert os.path.isfile(f"{tmp_path}/dcp/.metadata") and os.path.isfile(f"{tmp_path}/dcp/global_state_dict.pt")
    cfg = LlamaConfig.from_pretrained("2m")
    name = "model.layers.1.mlp.down_proj.weight"
    probe = {"model": {name: torch.zeros(cfg.hidden_size, cfg.intermediate_size)}}
    dcp.load(probe, checkpoint_id=f"{tmp_path}/dcp", no_dist=True)
    assert probe["model"][name].abs().sum() > 0
    g = _load(f"{tmp_path}/dcp/global_state_dict.pt")
    assert g["outer_optimizer"]["state"][0]["momentum_buffer"].shape == (cfg.vocab_size, cfg.hidden_size)
    import_dcp(f"{tmp_path}/dcp", f"{tmp_path}/back", cfg)
    a, b = _load(f"{src}/__0_0.distcp"), _load(f"{tmp_path}/back/__0_0.distcp")
    for key in ("model", "exp_avg", "exp_avg_sq", "outer_momentum"):
        assert torch.equal(a[key].float(), b[key].float()), key
    assert a["step"] == b["step"] == 4
