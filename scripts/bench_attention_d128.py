"""Head size 128 on the tcgen05 attention kernels against the library paths they replace (not part of bench.py).

    python scripts/bench_attention_d128.py [--out profiles/r4_attention_d128.jsonl] [--iters 10]

1. Kernel level, T = B*S = 32768 tokens, S in {1024, 2048, 4096}, (Hq, Hkv) in {(16, 16), (32, 8)}, head size 128.  CUDA
   events around `iters` launches after warm-up, forward and backward timed separately:
     * unmasked: our kernels ("tc") against cuDNN through aten (the head_dim-128 route before this change; its backward
       hands back three dense gradients, as the engine asks for);
     * masked, on a right-padded batch (lengths uniform in [S/4, S]) and on packed EOS-terminated documents (lengths
       uniform in [32, 512]): our MASKED kernels against torch SDPA with the equivalent dense boolean mask differentiated
       by autograd (the route masked head_dim-128 batches took before).
   TF/s use the causal-half FLOP count: forward 2 GEMMs, backward 5, each 2*S*S*D/2 per (batch, head).  Masked cases use
   the same count (their work is smaller: `allowed_pairs_vs_causal`).  q|k|v of every shape (>= 128 MB) exceeds the L2.
2. Micro-step of a head_dim-128 model (hidden 2048, 16 heads, 4 KV heads, intermediate 5632, 8 layers, V 32000, B16
   S1024; CUDA-graph replay) through LlamaForCausalLM.forward_backward, ODB_ATTN_LIB tc vs cudnn, unmasked and packed
   documents; the four arms alternate within this one process, the median of `rounds` windows is reported.

Prints and writes one JSON object per measurement, preceded by the card name, power limit and max SM clock read in the
same run.
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from opendiloco_b200 import LlamaConfig, LlamaForCausalLM  # noqa: E402
from opendiloco_b200.ops import attention as A  # noqa: E402
from opendiloco_b200.ops import kernels as K  # noqa: E402

EOS = 2
D = 128
T_TOKENS = 32768


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def batch(kind: str, B: int, S: int, seed: int):
    """(ids, mask or None, document_mask) of one case."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(3, 32000, (B, S), generator=g)
    if kind == "right_pad":
        mask = torch.zeros(B, S, dtype=torch.int64)
        for b in range(B):
            mask[b, :int(torch.randint(S // 4, S + 1, (1,), generator=g))] = 1
        return ids, mask, False
    if kind == "packed_docs":
        for b in range(B):
            p = -1
            while True:
                p += int(torch.randint(32, 513, (1,), generator=g))
                if p >= S:
                    break
                ids[b, p] = EOS
        return ids, None, True
    return ids, None, False


def timed(fn, iters: int) -> float:
    """Mean milliseconds of fn() over iters launches (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def causal_flops(B: int, S: int, Hq: int, gemms: int) -> float:
    return gemms * 2.0 * S * S * D / 2 * B * Hq


def kernel_cases(S: int, Hq: int, Hkv: int, iters: int):
    dev, B = "cuda", T_TOKENS // S
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=dev).to(torch.bfloat16)
    dout = torch.randn(B * S, Hq * D, device=dev).to(torch.bfloat16)
    dqkv = torch.empty_like(qkv)
    cos, sin = K.rope_tables(S, D, 10000.0, dev)
    fwd_f, bwd_f = causal_flops(B, S, Hq, 2), causal_flops(B, S, Hq, 5)
    base = {"bench": "attention_d128", "B": B, "S": S, "Hq": Hq, "Hkv": Hkv}

    def row(case, path, fwd_ms, bwd_ms, frac=1.0):
        return {**base, "case": case, "path": path, "fwd_ms": round(fwd_ms, 4), "bwd_ms": round(bwd_ms, 4),
                "fwd_tflops": round(fwd_f / fwd_ms / 1e9, 1), "bwd_tflops": round(bwd_f / bwd_ms / 1e9, 1),
                "allowed_pairs_vs_causal": round(frac, 4)}

    def tc(desc):
        out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc)
        f = timed(lambda: A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc), iters)
        b = timed(lambda: A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D, dqkv=dqkv, cos=cos, sin=sin, mask=desc), iters)
        return f, b

    def cudnn():
        saved = A._LIB
        A._LIB = "cudnn"
        try:
            out, aux = A.attention_fwd(qkv, B, S, Hq, Hkv, D)
            assert aux[0] == "cudnn"
            f = timed(lambda: A.attention_fwd(qkv, B, S, Hq, Hkv, D), iters)
            b = timed(lambda: A.attention_bwd(dout, qkv, out, aux, dqkv, B, S, Hq, Hkv, D, want_parts=True), iters)
        finally:
            A._LIB = saved
        return f, b

    def sdpa(desc):
        out, aux = A._sdpa_masked_fwd(qkv, desc, B, S, Hq, Hkv, D)
        f = timed(lambda: A._sdpa_masked_fwd(qkv, desc, B, S, Hq, Hkv, D), iters)
        # backward alone: re-running autograd on one retained graph
        b = timed(lambda: torch.autograd.grad(aux[1], aux[2], dout, retain_graph=True), iters)
        return f, b

    yield row("causal", "tc", *tc(None))
    yield row("causal", "cudnn", *cudnn())
    for kind, seed in (("right_pad", 1), ("packed_docs", 2)):
        ids, mask, doc = batch(kind, B, S, seed)
        desc = A.MaskDesc.empty(B, S, dev).build(ids.to(dev), mask.to(dev) if mask is not None else None, EOS if doc else -1)
        frac = float(A.dense_mask(desc, B, S).sum()) / float(B * S * (S + 1) // 2)
        yield row(kind, "tc_masked", *tc(desc), frac)
        yield row(kind, "sdpa_dense_mask", *sdpa(desc), frac)
        torch.cuda.empty_cache()


def micro_step(iters: int, rounds: int):
    cfg = LlamaConfig(hidden_size=2048, intermediate_size=5632, num_hidden_layers=8, num_attention_heads=16,
                      num_key_value_heads=4, vocab_size=32000)
    assert cfg.head_dim == D
    B, S = 16, 1024
    models = {}
    for lib in ("tc", "cudnn"):
        A._LIB = lib                               # each model keeps its own CUDA graphs, captured under its back-end
        models[lib] = LlamaForCausalLM(cfg, device="cuda", precision="bf16-mixed", seed=0)
    inputs = {}
    for kind in ("causal", "packed_docs"):
        ids, mask, doc = batch(kind, B, S, 3)
        inputs[kind] = (ids.cuda(), ids.cuda().clone(), doc)
    arms = [(lib, kind) for kind in inputs for lib in models]
    times = {arm: [] for arm in arms}
    for _ in range(rounds):
        for lib, kind in arms:
            A._LIB = lib
            ids, labels, doc = inputs[kind]
            times[(lib, kind)].append(timed(lambda: models[lib].forward_backward(ids, labels, 1.0, None, document_mask=doc), iters))
    A._LIB = "tc"
    for (lib, kind), ms in times.items():
        med = statistics.median(ms)
        yield {"bench": "llama_d128_micro_step", "attn_lib": lib, "case": kind, "B": B, "S": S, "ms_median": round(med, 3),
               "ms_all": [round(m, 3) for m in ms], "tokens_per_s": round(B * S / med * 1e3)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attention_d128.py needs a GPU")
    rows = [card()]
    print(json.dumps(rows[0]), flush=True)
    gen = [kernel_cases(S, Hq, Hkv, a.iters) for S in (1024, 2048, 4096) for Hq, Hkv in ((16, 16), (32, 8))]
    for r in itertools.chain(*gen, micro_step(a.iters, a.rounds)):
        print(json.dumps(r), flush=True)
        rows.append(r)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()
