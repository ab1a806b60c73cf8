"""Cost of padded / document-masked batches on the tcgen05 attention kernels (not part of bench.py).

    python scripts/bench_masked_attention.py [--out FILE] [--iters 20]

1. Attention forward+backward kernel time (CUDA events, after warm-up) at the Llama-150M shape (B32 S1024, 16 heads of 64)
   and a Llama-1B GQA shape (B16 S1024, 32:4 heads), for: the causal kernels; the MASKED kernels on an all-ones
   description; a right-padded batch (seeded lengths uniform in [S/4, S]); packed documents (seeded lengths uniform in
   [32, 512], EOS-terminated) with document masking; and torch SDPA with the equivalent dense boolean mask, differentiated
   by autograd (the route padded batches took before the masked kernels).  Both shapes' q|k|v (>= 200 MB) exceed the L2.
2. The Llama-150M training micro-step (B32 S1024, CUDA-graph replay) through LlamaForCausalLM.forward_backward: no mask,
   a right-padded batch, packed documents.

Prints and writes one JSON object per measurement, preceded by the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from opendiloco_b200 import LlamaConfig, LlamaForCausalLM  # noqa: E402
from opendiloco_b200.ops import attention as A  # noqa: E402

EOS = 2


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


def attention_cases(B: int, S: int, Hq: int, Hkv: int, iters: int):
    dev = "cuda"
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * 64, device=dev).to(torch.bfloat16)
    dout = torch.randn(B * S, Hq * 64, device=dev).to(torch.bfloat16)

    def tc(desc):
        def run():
            out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, mask=desc)
            A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, mask=desc)
        return run

    def sdpa(desc):
        def run():
            out, aux = A._sdpa_masked_fwd(qkv, desc, B, S, Hq, Hkv, 64)
            torch.autograd.grad(aux[1], aux[2], dout)
        return run

    ids, _, _ = batch("causal", B, S, 0)
    ones = A.MaskDesc.empty(B, S, dev).build(ids.to(dev), None, -1)
    ids_p, mask_p, _ = batch("right_pad", B, S, 1)
    pad = A.MaskDesc.empty(B, S, dev).build(ids_p.to(dev), mask_p.to(dev), -1)
    ids_d, _, _ = batch("packed_docs", B, S, 2)
    docs = A.MaskDesc.empty(B, S, dev).build(ids_d.to(dev), None, EOS)
    kept = lambda d: float(A.dense_mask(d, B, S).sum()) / float(B * S * (S + 1) // 2)  # noqa: E731
    cases = [("causal", tc(None), 1.0), ("masked_all_ones", tc(ones), kept(ones)), ("right_pad", tc(pad), kept(pad)),
             ("packed_docs", tc(docs), kept(docs)), ("sdpa_dense_right_pad", sdpa(pad), kept(pad))]
    for name, fn, frac in cases:
        ms = timed(fn, iters)
        yield {"bench": "attention_fwd_bwd", "B": B, "S": S, "Hq": Hq, "Hkv": Hkv, "case": name, "ms": round(ms, 4),
               "allowed_pairs_vs_causal": round(frac, 4)}


def micro_step(iters: int):
    cfg = LlamaConfig.from_pretrained("150m")
    B, S = 32, 1024
    for kind in ("causal", "right_pad", "packed_docs"):
        model = LlamaForCausalLM(cfg, device="cuda", precision="bf16-mixed", seed=0)
        ids, mask, doc = batch(kind, B, S, 3)
        ids = ids.cuda()
        labels = ids.clone()
        if mask is not None:
            labels[mask.cuda() == 0] = -100
        ms = timed(lambda: model.forward_backward(ids, labels, 1.0, mask, document_mask=doc), iters)
        yield {"bench": "llama150m_micro_step", "B": B, "S": S, "case": kind, "ms": round(ms, 3),
               "tokens_per_s": round(B * S / ms * 1e3)}
        del model
        torch.cuda.empty_cache()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_masked_attention.py needs a GPU")
    rows = [card()]
    print(json.dumps(rows[0]), flush=True)
    for r in [*attention_cases(32, 1024, 16, 16, a.iters), *attention_cases(16, 1024, 32, 4, a.iters), *micro_step(a.iters)]:
        print(json.dumps(r), flush=True)
        rows.append(r)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()
