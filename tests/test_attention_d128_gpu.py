"""Head size 128 on a B200: the tcgen05 attention kernels (causal and MASKED) against fp32 references, their determinism and
dispatch, and a D = 128 model's engine step on them (bf16 vs fp32, tc vs cuDNN, CUDA graph vs eager, no library attention
kernel in the trace)."""
import math

import pytest
import torch

from opendiloco_b200 import LlamaConfig, LlamaForCausalLM
from opendiloco_b200.ops import attention as A
from opendiloco_b200.ops import kernels as K

pytestmark = pytest.mark.gpu

DEV = "cuda"
BF = torch.bfloat16
D = 128
EOS = 2
FAMILIES = ["right_pad", "left_pad", "hole", "eos_127_128", "eos_consecutive", "eos_pad", "packed_docs"]
SHAPES = [(1, 128, 8, 8), (2, 384, 8, 8), (2, 1024, 16, 16), (2, 2048, 32, 8), (3, 1024, 16, 2)]


def rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-12)).item()


def make_batch(family: str, B: int, S: int, seed: int = 0):
    """(ids [B, S] int64, mask [B, S] int64 or None, eos) of one mask family; every row differs."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(3, 1000, (B, S), generator=g)
    mask, eos = None, -1
    lengths = [1 + int(torch.randint(0, S, (1,), generator=g)) for _ in range(B)]
    lengths[0] = 1                                               # a row with a single real token
    if family in ("right_pad", "eos_pad"):
        mask = torch.zeros(B, S, dtype=torch.int64)
        for b, n in enumerate(lengths):
            mask[b, :n] = 1
    elif family == "left_pad":
        mask = torch.zeros(B, S, dtype=torch.int64)
        for b, n in enumerate(lengths):
            mask[b, S - n:] = 1
    elif family == "hole":
        mask = torch.ones(B, S, dtype=torch.int64)
        for b in range(B):
            a = int(torch.randint(0, S // 2, (1,), generator=g))
            mask[b, a:a + 1 + (S // 16) * (b + 1)] = 0
    if family.startswith("eos") or family == "packed_docs":
        eos = EOS
    if family == "eos_127_128":
        ids[:, 127] = EOS
        ids[:, 128] = EOS
        ids[1:, S - 300] = EOS
    elif family == "eos_consecutive":
        for b in range(B):
            a = 200 + 97 * b
            ids[b, a:a + 4] = EOS
    elif family == "eos_pad":
        for b, n in enumerate(lengths):
            for p in (n // 3, n // 2, n + 5):
                if p < S:
                    ids[b, p] = EOS
    elif family == "packed_docs":
        for b in range(B):
            p = 0
            while True:
                p += 1 + int(torch.randint(0, 400, (1,), generator=g))
                if p >= S:
                    break
                ids[b, p] = EOS
    return ids, mask, eos


def describe(ids, mask, eos):
    B, S = ids.shape
    return A.MaskDesc.empty(B, S, DEV).build(ids.to(DEV), mask.to(DEV) if mask is not None else None, eos)


def reference(qkv, dout, desc, B, S, Hq, Hkv):
    """fp32 attention at head size 128, causal (desc None) or with the dense mask of a description: (out, lse, dqkv)."""
    x = qkv.float().detach().requires_grad_(True)
    q, k, v = (t.permute(0, 2, 1, 3) for t in A.split_qkv(x, B, S, Hq, Hkv, D))
    k, v = k.repeat_interleave(Hq // Hkv, dim=1), v.repeat_interleave(Hq // Hkv, dim=1)
    att = (q @ k.transpose(-1, -2)) / math.sqrt(D)
    allowed = torch.ones(S, S, dtype=torch.bool, device=DEV).tril() if desc is None else A.dense_mask(desc, B, S)
    att = att.masked_fill(~allowed, float("-inf"))
    lse = torch.logsumexp(att, dim=-1)
    out = (torch.softmax(att, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * S, Hq * D)
    out.backward(dout.float())
    return out.detach(), lse.detach(), x.grad


def _check_grads(grads, dref, Hq, Hkv, tol=1e-2):
    dq, dk, dv = grads
    q_dim, kv_dim = Hq * D, Hkv * D
    assert rel(dq, dref[:, :q_dim]) < tol
    assert rel(dk, dref[:, q_dim:q_dim + kv_dim]) < tol
    assert rel(dv, dref[:, q_dim + kv_dim:]) < tol


@pytest.mark.parametrize("B,S,Hq,Hkv", SHAPES)
def test_causal_kernels_against_fp32(B, S, Hq, Hkv):
    torch.manual_seed(0)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D)
    dout = torch.randn_like(out)
    grads = A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D)
    for t in (out, lse, *grads):
        assert torch.isfinite(t.float()).all()
    ref_out, ref_lse, dref = reference(qkv, dout, None, B, S, Hq, Hkv)
    assert rel(out, ref_out) < 5e-3
    assert (lse - ref_lse).abs().max().item() < 1e-3
    _check_grads(grads, dref, Hq, Hkv)


@pytest.mark.parametrize("B,S,Hq,Hkv", [(2, 1024, 16, 16), (3, 1024, 16, 2)])
def test_packed_rope_transpose(B, S, Hq, Hkv):
    """Packed dq|dk|dv with the RoPE transpose in the kernels == dense gradients rotated afterwards by rope_(backward=True)."""
    torch.manual_seed(2)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    cos, sin = K.rope_tables(S, D, 10000.0, DEV)
    out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D)
    dout = torch.randn_like(out)
    packed = A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D, dqkv=torch.empty_like(qkv), cos=cos, sin=sin)
    dense = torch.cat(A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D), dim=1)
    K.rope_(dense, cos, sin, S, Hq + Hkv, D, backward=True)
    assert rel(packed, dense) < 6e-3


@pytest.mark.parametrize("B,S,Hq,Hkv", [(2, 1024, 16, 16), (3, 2048, 16, 4)])
@pytest.mark.parametrize("family", FAMILIES)
def test_masked_kernels_against_fp32(family, B, S, Hq, Hkv):
    torch.manual_seed(0)
    ids, mask, eos = make_batch(family, B, S, seed=B * S + Hq)
    desc = describe(ids, mask, eos)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc)
    dout = torch.randn_like(out)
    grads = A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D, mask=desc)
    for t in (out, lse, *grads):
        assert torch.isfinite(t.float()).all()
    ref_out, ref_lse, dref = reference(qkv, dout, desc, B, S, Hq, Hkv)
    assert rel(out, ref_out) < 5e-3
    assert (lse - ref_lse).abs().max().item() < 1e-3
    _check_grads(grads, dref, Hq, Hkv)


@pytest.mark.parametrize("B,S,Hq,Hkv", [(2, 1024, 16, 16), (3, 2048, 32, 4)])
def test_all_ones_description_matches_causal(B, S, Hq, Hkv):
    torch.manual_seed(1)
    desc = describe(torch.randint(3, 1000, (B, S)), None, -1)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    out_c, lse_c = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D)
    out_m, lse_m = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc)
    assert rel(out_m, out_c) < 1e-5 and rel(lse_m, lse_c) < 1e-5
    dout = torch.randn_like(out_c)
    gc = A.tc_attention_bwd(dout, qkv, out_c, lse_c, B, S, Hq, Hkv, D)
    gm = A.tc_attention_bwd(dout, qkv, out_m, lse_m, B, S, Hq, Hkv, D, mask=desc)
    for a, b in zip(gc, gm):
        assert rel(b, a) < 1e-5


def test_backward_is_deterministic():
    B, S, Hq, Hkv = 2, 2048, 32, 8
    torch.manual_seed(3)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    out, lse = A.tc_attention_fwd(qkv, B, S, Hq, Hkv, D)
    dout = torch.randn_like(out)
    first = A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D, dqkv=torch.empty_like(qkv)).clone()
    second = A.tc_attention_bwd(dout, qkv, out, lse, B, S, Hq, Hkv, D, dqkv=torch.empty_like(qkv))
    assert torch.equal(first, second)


def test_dispatch_takes_tc():
    B, S, Hq, Hkv = 2, 1024, 8, 4
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device=DEV).to(BF)
    assert A.attention_fwd(qkv, B, S, Hq, Hkv, D)[1][0] == "tc"
    ids, mask, eos = make_batch("packed_docs", B, S, seed=9)
    assert A.attention_fwd(qkv, B, S, Hq, Hkv, D, mask=describe(ids, mask, eos))[1][0] == "tc"


def _cfg():
    return LlamaConfig(hidden_size=1024, intermediate_size=2816, num_hidden_layers=2, num_attention_heads=8,
                       num_key_value_heads=4, vocab_size=32000)


def _labels(ids, mask):
    lab = ids.clone()
    if mask is not None:
        lab[mask == 0] = -100
    return lab


def _worst(a, b):
    errs = {n: ((a.arena.g(n) - b.arena.g(n)).norm() / (b.arena.g(n).norm() + 1e-12)).item() for n in a.arena.slots}
    return max(errs.items(), key=lambda kv: kv[1])


@pytest.mark.parametrize("document_mask", [False, True])
def test_engine_bf16_against_fp32(document_mask):
    cfg = _cfg()
    assert cfg.head_dim == D
    ref = LlamaForCausalLM(cfg, device=DEV, precision="32-true", seed=2)
    gpu = LlamaForCausalLM(cfg, device=DEV, precision="bf16-mixed", seed=2)
    ids, _, _ = make_batch("packed_docs", 2, 1024, seed=5)
    ids = ids.to(DEV)
    lr = ref.forward_backward(ids, ids, 1.0, document_mask=document_mask)
    lg = gpu.forward_backward(ids, ids, 1.0, document_mask=document_mask)
    assert torch.isfinite(lg) and abs(lr.item() - lg.item()) / lr.item() < 2e-3, (lr.item(), lg.item())
    worst = _worst(gpu, ref)
    print("document_mask", document_mask, "worst per-tensor rel err vs fp32:", worst)
    assert worst[1] < 2e-2


@pytest.mark.parametrize("family", [None, "right_pad", "packed_docs"])
def test_engine_tc_against_cudnn(family, monkeypatch):
    cfg = _cfg()
    ids, mask, eos = make_batch(family or "right_pad", 2, 1024, seed=6)
    mask = mask if family == "right_pad" else None
    doc = family == "packed_docs"
    ids, lab = ids.to(DEV), _labels(ids, mask).to(DEV)
    dm = mask.to(DEV) if mask is not None else None
    losses, models = {}, {}
    for lib in ("tc", "cudnn"):
        monkeypatch.setattr(A, "_LIB", lib)
        models[lib] = LlamaForCausalLM(cfg, device=DEV, precision="bf16-mixed", seed=3)
        losses[lib] = models[lib].forward_backward(ids, lab, 1.0, dm, document_mask=doc).item()
    assert abs(losses["tc"] - losses["cudnn"]) / losses["cudnn"] < 1e-3, losses
    worst = _worst(models["tc"], models["cudnn"])
    print(family, "worst per-tensor rel err tc vs cudnn:", worst)
    assert worst[1] < 2e-2


@pytest.mark.parametrize("document_mask", [False, True])
def test_graphed_masked_steps_match_eager(document_mask, monkeypatch):
    """Five micro-steps, a different mask on each: the CUDA-graph replay (captured on the third) equals eager execution."""
    cfg = _cfg()
    models = {k: LlamaForCausalLM(cfg, device=DEV, precision="bf16-mixed", seed=7) for k in ("graph", "eager", "eager2")}
    for step in range(5):
        ids, mask, _ = make_batch("packed_docs" if document_mask else "right_pad", 2, 1024, seed=100 + step)
        if document_mask and step % 2:
            mask = make_batch("hole", 2, 1024, seed=200 + step)[1]          # document and padding mask together
        ids, lab = ids.to(DEV), _labels(ids, mask).to(DEV)
        dm = mask.to(DEV) if mask is not None else None
        losses = {}
        for k, m in models.items():
            monkeypatch.setenv("ODB_CUDA_GRAPH", "1" if k == "graph" else "0")
            losses[k] = m.forward_backward(ids, lab, 0.5, dm, document_mask=document_mask).clone()
        torch.cuda.synchronize()
        gg, ge, ge2 = (models[k].arena.grad for k in ("graph", "eager", "eager2"))
        if torch.equal(ge, ge2) and torch.equal(losses["eager"], losses["eager2"]):
            assert torch.equal(losses["graph"], losses["eager"]), step
            assert torch.equal(gg, ge), step
        else:   # reductions elsewhere in the step whose order is not fixed: eager itself is not reproducible
            assert rel(gg, ge) <= max(10 * rel(ge2, ge), 1e-6), step
    assert any(k[4] for k in models["graph"].engine._graphs), "no masked micro-step was captured"


def test_no_library_attention_kernel_in_masked_step(monkeypatch):
    monkeypatch.setenv("ODB_CUDA_GRAPH", "0")
    model = LlamaForCausalLM(_cfg(), device=DEV, precision="bf16-mixed", seed=8)
    ids, mask, _ = make_batch("packed_docs", 2, 1024, seed=11)
    mask = make_batch("right_pad", 2, 1024, seed=12)[1]
    ids, lab, dm = ids.to(DEV), _labels(ids, mask).to(DEV), mask.to(DEV)
    model.forward_backward(ids, lab, 1.0, dm, document_mask=True)                   # warm-up (prep, workspace)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        model.forward_backward(ids, lab, 1.0, dm, document_mask=True)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    lowered = [n.lower() for n in names]
    library = [n for n, l in zip(names, lowered) if any(s in l for s in ("cudnn", "flash", "fmha", "sdpa", "efficient"))]
    assert not library, library
    for ours in ("attn_fwd_kernel", "attn_bwd_dkv_d128_kernel", "attn_bwd_dq_d128_kernel"):
        assert any(ours in n for n in names), (ours, sorted(names))
