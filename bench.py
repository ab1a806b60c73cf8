#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): DiLoCo training throughput of Llama-150M, 1 worker per GPU, bf16, synthetic
tokens, random-init weights.

    python bench.py --gpus 1 --steps 8 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
        bench.py --gpus 8 --steps 8 --warmup 3
    python bench.py --impl reference ...        # the UNMODIFIED reference (baseline/_ref) on the same config
    python bench.py --steps 8 --dump-outputs out/  # also write what the last timed step computed (out/*.npy)

A "step" is one inner optimizer step of every worker: ``batch`` sequences x ``seq`` tokens per worker processed as
``batch / micro_batch`` gradient-accumulated micro-batches, global-norm clip, AdamW, LR schedule; the DiLoCo outer step
(pseudo-gradient all-reduce + Nesterov) falls due on the LAST timed step (local_steps = warmup + steps), so the timed
window contains the whole algorithm.  ``value`` = whole-job tokens/s over exactly K steps, timed on the device with
CUDA events between barriers, max over ranks.  ``e2e`` = the same through the public ``DiLoCoTrainer.train_step`` API
with, every micro-batch, the pinned host->device copy of the inputs and, every step, a device->host read of the loss.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-fsdp"],
                    help="ours | reference (unmodified train_diloco_torch.py, eager: the DiLoCo oracle) | reference-fsdp "
                         "(unmodified train_fsdp.py, FSDP NO_SHARD + torch.compile: the stronger inner-step baseline)")
    ap.add_argument("--model", default="150m")
    ap.add_argument("--seq", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=512, help="sequences per worker per optimizer step (reference --batch-size)")
    ap.add_argument("--micro-batch", type=int, default=32, help="per-device micro-batch (reference --per-device-train-batch-size)")
    ap.add_argument("--local-steps", type=int, default=None, help="H; default warmup+steps (one outer step, on the last timed step)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--compression", default=None)
    ap.add_argument("--no-fused-collective", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss of the last timed step and a fixed sample of the fp32 master "
                         "weights it left behind as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


# --------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md 'clocks' line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_PARAM_SAMPLE = 1 << 23          # 32 MB of fp32 weights


def dump_outputs(out_dir: str, loss, master) -> None:
    """What a caller of ``train_step`` holds after the last timed step: the loss it returned and the parameters it left.
    Models larger than DUMP_PARAM_SAMPLE parameters are sampled at fixed (seed 0) positions of the flat master vector."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n = master.numel()
    if n > DUMP_PARAM_SAMPLE:
        idx = torch.randint(n, (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        master = master[idx.to(master.device)]
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())
    np.save(os.path.join(out_dir, "master_params.npy"), master.detach().float().cpu().numpy())


def baseline_number():
    """BASELINE.md publishes no throughput for the reference (published = {}), so vs_baseline is null."""
    try:
        pub = json.load(open(os.path.join(ROOT, "BASELINE.json"))).get("published") or {}
        v = pub.get("tokens_per_sec")
        return float(v) if v else None
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------- our arm
def run_ours(a) -> dict:
    import torch
    import torch.distributed as dist

    from opendiloco_b200 import _lib
    from opendiloco_b200.models.config import LlamaConfig
    from opendiloco_b200.models.llama import LlamaForCausalLM
    from opendiloco_b200.parallel import comm
    from opendiloco_b200.trainer import DiLoCoTrainer, TrainerConfig
    from opendiloco_b200.utils.data import NativeTokenLoader, SyntheticTokenLoader

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {a.gpus}"
    torch.cuda.set_device(local_rank)
    if world > 1:
        comm.init_distributed("nccl")
    dev = torch.device("cuda", local_rank)
    cfg = LlamaConfig.from_pretrained(a.model)
    model = LlamaForCausalLM(cfg, device=dev, precision="bf16-mixed", seed=0)
    accum = a.batch // a.micro_batch
    H = a.local_steps if a.local_steps is not None else a.warmup + a.steps
    compression = None
    if a.compression:
        from opendiloco_b200.parallel.compression import get_compression

        compression = get_compression(a.compression)
    topo = comm.build_topology(galaxy_size=world, gpus_per_worker=1)
    tr = DiLoCoTrainer(model, TrainerConfig(grad_accum=accum, local_steps=H, samples_per_step=a.batch, warmup_steps=1000,
                                            total_steps=88_000, compression=compression,
                                            fused_collective=False if a.no_fused_collective else None), topo)
    tr.broadcast_initial_weights()
    try:      # C++ prefetcher filling pinned buffers (csrc/host/tokengen.cc)
        loader = NativeTokenLoader(a.micro_batch, a.seq, vocab_size=cfg.vocab_size, seed=1234, rank=rank)
    except RuntimeError:
        loader = SyntheticTokenLoader(a.micro_batch, a.seq, vocab_size=cfg.vocab_size, seed=1234, rank=rank, with_mask=False)
    tokens_per_step = a.batch * a.seq * world

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-timed arm: inputs pre-staged in HBM, CUDA events around exactly K steps
    staged = [{k: v.to(dev) for k, v in next(loader).items()} for _ in range(accum)]
    for b in staged:
        b["labels"] = b["input_ids"]

    def staged_iter():
        while True:
            yield from staged

    it = staged_iter()
    for _ in range(a.warmup):
        tr.train_step(it)
    sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    _lib.reset_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.steps):
        loss = tr.train_step(it)
    ev1.record()
    sync()
    my_ms = ev0.elapsed_time(ev1)
    dev_ms = max_over_ranks(my_ms)
    per_rank_ms = [my_ms / a.steps]
    if world > 1:       # who is the slowest board?  (names the limiter of the 1 -> N curve)
        t = torch.tensor([my_ms / a.steps], dtype=torch.float64, device=dev)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [round(float(x.item()), 3) for x in allt]
    launches = _lib.launch_count()
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:        # before the outer-sync timing and the e2e arm move the weights on
        dump_outputs(a.dump_outputs, loss, model.arena.master)
    outer_in_window = sum(1 for s in range(a.warmup + 1, a.warmup + a.steps + 1) if s % H == 0)
    value = tokens_per_step * a.steps / (dev_ms / 1e3)

    # ---------------- separate measurement of the outer sync alone (ms, effective GB/s over the fp32 parameter vector)
    # ``outer_sync_ms``: device time of the sync itself (pseudo-gradient -> all-reduce -> Nesterov -> weights), membership
    # handshake switched off.  ``outer_sync_with_handshake_ms``: the whole ``_update_global_epoch`` including the board
    # round trips of the arrival handshake; in training the host reaches that point while the GPU still works through the
    # queued micro-batches, so those round trips are hidden - here the queue is empty and they show up on the events.
    outer_ms = outer_hs_ms = None
    if tr.is_diloco:
        opt = tr.optimizer

        def time_outer():
            times = []
            for _ in range(4):
                sync()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                opt._update_global_epoch()
                e1.record()
                sync()
                times.append(max_over_ranks(e0.elapsed_time(e1)))
            return min(times[1:])

        outer_hs_ms = time_outer()
        saved = opt.timeout_waiting_for_peers
        opt.timeout_waiting_for_peers = None
        outer_ms = time_outer()
        opt.timeout_waiting_for_peers = saved
    nparam = model.arena.numel
    # after an outer step every worker must hold bit-identical parameters: wrap-around integer checksum, min == max
    params_equal = None
    if world > 1 and tr.is_diloco:
        fp = model.arena.master.view(torch.int32).sum(dtype=torch.int64)
        pair = torch.stack([fp, -fp])
        dist.all_reduce(pair, op=dist.ReduceOp.MAX)
        params_equal = bool(int(pair[0]) == -int(pair[1]))
        assert params_equal, "workers hold different parameters after the outer step"

    # ---------------- end-to-end arm: public API, pinned H2D every micro-batch, D2H loss read every step
    e2e = None
    if not a.no_e2e:
        h2d = a.micro_batch * a.seq * 8 * accum          # int64 input ids (labels alias the ids on the host)
        d2h = 4
        for _ in range(a.warmup):
            float(tr.train_step(loader).item())
        sync()
        t0 = time.perf_counter()
        last = 0.0
        for _ in range(a.steps):
            last = float(tr.train_step(loader).item())
        sync()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": tokens_per_step * a.steps / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3 / a.steps, "last_loss": last}

    flops_tok = cfg.flops_per_token(a.seq)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sustained = peaks.get("bf16_tflops_sustained", 1400.0)
    out = {
        "metric": "tokens_per_sec (DiLoCo inner steps incl. one outer sync in the timed window)",
        "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": (value / baseline_number()) if baseline_number() else None,
        "dtype": "bf16", "data": "synthetic tokens (uniform over vocab), random-init weights",
        "impl": "ours",
        "config": {"model": f"llama-{a.model}", "global_batch": a.batch * world, "per_worker_batch": a.batch,
                   "micro_batch": a.micro_batch, "grad_accum": accum, "seq_len": a.seq, "parallelism": f"diloco{world}x1",
                   "local_steps": H, "outer_steps_in_timed_window": outer_in_window},
        "notes": {"l2": "per-step working set (>10 GB activations + 3.4 GB optimizer state) >> 126 MB L2; no flush needed",
                  "inner_opt": "AdamW lr4e-4 wd0.1 b(0.9,0.95) clip1.0 cosine(1000,88000)", "outer_opt": "SGD lr0.7 m0.9 nesterov",
                  "entry": "opendiloco_b200.trainer.DiLoCoTrainer.train_step"},
        "per_rank_ms_per_step": per_rank_ms, "params_equal_across_ranks": params_equal,
        "tokens_per_sec_per_gpu": value / world,
        "mfu_vs_measured_sustained": (value / world) * flops_tok / (sustained * 1e12),
        "outer_sync_ms": outer_ms, "outer_sync_with_handshake_ms": outer_hs_ms,
        "outer_sync_eff_GBps": (nparam * 4 / (outer_ms / 1e3) / 1e9) if outer_ms else None,
        "outer_fused_collective": bool(getattr(tr.optimizer, "_fused", None)) if tr.is_diloco else None,
        "outer_kernel": (("sharded in-place (ZeRO-1 outer optimizer over NVLS)" if tr.optimizer._fused.sharded else "replicated update")
                         if tr.is_diloco and getattr(tr.optimizer, "_fused", None) else None),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
    }
    if world > 1:
        dist.destroy_process_group()
    return out if rank == 0 else {}


# --------------------------------------------------------------------------------------------------- reference arm
def run_reference(a) -> dict:
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "open_diloco")):
        return {"impl": a.impl, "unavailable": "baseline/_ref/open_diloco missing (pip --target install not present)"}
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        if a.impl == "reference-fsdp":
            from run_reference_fsdp import run as run_ref
        else:
            from run_reference import run as run_ref
    except Exception as e:  # pragma: no cover
        return {"impl": a.impl, "unavailable": f"reference shims failed to import: {type(e).__name__}: {e}"}
    try:
        return run_ref(a, ClockSampler)
    except Exception as e:
        import traceback

        traceback.print_exc()
        return {"impl": a.impl, "unavailable": f"{type(e).__name__}: {str(e)[:200]}"}


def main():
    a = parse_args()
    out = run_ours(a) if a.impl == "ours" else run_reference(a)
    if out:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
