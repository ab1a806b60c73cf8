"""Mask descriptions for padded and document-masked batches (ops/kernels.py::attn_mask_prep reference), the math attention
reference driven by them, document-mask equivalence of the engine, and --document-mask through train_fsdp."""
import math
import os
import pickle
import sys

import pytest
import torch

from opendiloco_b200 import LlamaConfig, LlamaForCausalLM
from opendiloco_b200.ops import attention as A

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_training_cpu import BASE, torchrun  # noqa: E402

EOS = 2


def describe(ids, mask=None, eos=-1):
    ids = torch.as_tensor(ids, dtype=torch.int64)
    ids = ids[None] if ids.dim() == 1 else ids
    if mask is not None:
        mask = torch.as_tensor(mask)
        mask = mask[None] if mask.dim() == 1 else mask
    return A.MaskDesc.empty(*ids.shape, "cpu").build(ids, mask, eos)


def bits(desc, b=0):
    return [(int(w) >> i) & 1 for w in desc.vbits[b].tolist() for i in range(32)]


def row(S, fill=5):
    return [fill] * S


def test_right_padding():
    S = 256
    d = describe(row(S), [1] * 100 + [0] * 156)
    lo = d.lo.tolist()
    assert lo == [0] * S                                     # pad queries keep attending to the real keys (and themselves)
    assert bits(d) == [1] * 100 + [0] * 156
    assert d.kv_lo.tolist() == [[0, 0]] and d.q_hi.tolist() == [[1, 1]] and d.lo_hi.tolist() == [[0, 0]]
    assert int(d.vbits[0, 3]) == (1 << 4) - 1 and int(d.vbits[0, 0]) == -1


def test_left_padding():
    S = 384
    d = describe(row(S), [0] * 200 + [1] * 184)
    assert d.lo.tolist() == list(range(200)) + [200] * 184   # leading pads see only themselves
    assert bits(d) == [0] * 200 + [1] * 184
    assert d.kv_lo.tolist() == [[0, 1, 1]]
    assert d.lo_hi.tolist() == [[127, 200, 200]]
    assert d.q_hi.tolist() == [[0, 2, 2]]


def test_hole_in_the_mask():
    S = 256
    m = [1] * S
    m[10:150] = [0] * 140
    d = describe(row(S), m)
    assert d.lo.tolist() == [0] * S
    assert bits(d) == m
    assert d.kv_lo.tolist() == [[0, 0]] and d.q_hi.tolist() == [[1, 1]]
    # first real key is a pad: queries inside the leading pad run see only themselves
    m2 = [0] * 20 + [1] * 236
    assert describe(row(S), m2).lo.tolist()[:21] == list(range(20)) + [20]


def test_eos_at_127_and_128():
    S = 384
    ids = row(S)
    ids[127] = EOS
    ids[128] = EOS
    d = describe(ids, eos=EOS)
    lo = d.lo.tolist()
    assert lo[:128] == [0] * 128                             # the EOS belongs to the document it ends
    assert lo[128] == 128                                    # a one-token document: the second EOS
    assert lo[129:] == [129] * (S - 129)
    assert d.kv_lo.tolist() == [[0, 1, 1]] and d.lo_hi.tolist() == [[0, 129, 129]]
    assert d.q_hi.tolist() == [[0, 2, 2]]                    # key tile 0 is never seen by query tiles 1, 2
    assert bits(d) == [1] * S
    # without document masking the same ids are plain causal
    assert describe(ids).lo.tolist() == [0] * S


def test_consecutive_eos():
    S = 256
    ids = row(S)
    ids[50:53] = [EOS] * 3
    lo = describe(ids, eos=EOS).lo.tolist()
    assert lo[:51] == [0] * 51 and lo[51] == 51 and lo[52] == 52 and lo[53:] == [53] * (S - 53)


def test_eos_with_padding():
    S = 256
    ids = row(S)
    ids[40] = EOS
    ids[170] = EOS                                           # an EOS inside the right padding
    m = [1] * 150 + [0] * 106
    d = describe(ids, m, eos=EOS)
    lo = d.lo.tolist()
    assert lo[:41] == [0] * 41 and lo[41:171] == [41] * 130
    assert lo[171:] == list(range(171, S))                   # no real key in the document after the pad EOS
    assert d.kv_lo.tolist() == [[0, 0]] and d.lo_hi.tolist() == [[41, 255]] and d.q_hi.tolist() == [[1, 1]]
    # left padding + documents: the first document starts at the first real token
    ids2 = row(S)
    ids2[100] = EOS
    m2 = [0] * 60 + [1] * 196
    lo2 = describe(ids2, m2, eos=EOS).lo.tolist()
    assert lo2[:60] == list(range(60)) and lo2[60:101] == [60] * 41 and lo2[101:] == [101] * (S - 101)


def test_batch_rows_are_independent_and_dtypes_agree():
    torch.manual_seed(0)
    ids = torch.randint(3, 50, (3, 256))
    ids[ids == 7] = EOS
    m = (torch.rand(3, 256) > 0.2).long()
    ref = describe(ids, m, eos=EOS)
    for b in range(3):
        one = describe(ids[b], m[b], eos=EOS)
        assert torch.equal(one.lo, ref.lo.view(3, -1)[b]) and torch.equal(one.q_hi[0], ref.q_hi[b])
    for dt in (torch.bool, torch.int32, torch.uint8):
        alt = describe(ids, m.to(dt), eos=EOS)
        assert all(torch.equal(getattr(alt, n), getattr(ref, n)) for n in ("lo", "vbits", "kv_lo", "q_hi", "lo_hi"))


def test_math_reference_matches_causal_key_mask_or_eye():
    """Document masking off: the description's dense mask is exactly `causal & key_mask | eye`, the semantics of the SDPA
    route padded batches took before; the math reference driven by the description gives that attention."""
    torch.manual_seed(1)
    B, S, Hq, Hkv, D = 3, 256, 4, 2, 64
    for trial in range(4):
        m = (torch.rand(B, S) > [0.1, 0.5, 0.9, 0.3][trial]).long()
        if trial == 3:
            m[0] = 0                                         # an all-pad row
        desc = describe(torch.randint(3, 100, (B, S)), m)
        causal = torch.ones(S, S, dtype=torch.bool).tril()
        legacy = (causal[None, None] & m.bool()[:, None, None, :]) | torch.eye(S, dtype=torch.bool)[None, None]
        assert torch.equal(A.dense_mask(desc, B, S), legacy)
        qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D)
        out, (lse, _) = A.attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc)
        q, k, v = (t.transpose(1, 2) for t in A.split_qkv(qkv, B, S, Hq, Hkv, D))
        ref = torch.nn.functional.scaled_dot_product_attention(q, k, v, attn_mask=legacy, enable_gqa=True)
        assert torch.allclose(out, ref.transpose(1, 2).reshape(B * S, Hq * D), atol=1e-5)
        assert torch.isfinite(lse).all()


def _packed_vs_separate(cfg, S, doc_lens, seed=0):
    g = torch.Generator().manual_seed(seed)
    docs = [torch.cat([torch.randint(3, cfg.vocab_size, (n - 1,), generator=g), torch.tensor([cfg.eos_token_id])]) for n in doc_lens]
    packed = torch.cat(docs)
    assert packed.numel() == S
    plab = packed.clone()
    start = 0
    for n in doc_lens[:-1]:
        start += n
        plab[start] = -100                                   # the EOS does not predict the next document's first token
    sep = torch.zeros(len(docs), S, dtype=torch.int64)
    mask = torch.zeros(len(docs), S, dtype=torch.int64)
    for b, d in enumerate(docs):
        sep[b, :d.numel()] = d
        mask[b, :d.numel()] = 1
    slab = sep.masked_fill(mask == 0, -100)
    return packed[None], plab[None], sep, slab, mask


def test_document_mask_matches_separate_rows_fp32():
    """A packed row [A EOS B EOS C ...] with document_mask=True == the same documents as separate right-padded rows: loss and
    every parameter gradient (RoPE positions differ, but scores depend only on s - t)."""
    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, vocab_size=512)
    packed, plab, sep, slab, mask = _packed_vs_separate(cfg, 192, [70, 1, 57, 64])
    a = LlamaForCausalLM(cfg, device="cpu", precision="32-true", seed=3)
    b = LlamaForCausalLM(cfg, device="cpu", precision="32-true", seed=3)
    la = a.forward_backward(packed, plab, 1.0, document_mask=True)
    lb = b.forward_backward(sep, slab, 1.0, mask)
    assert math.isclose(la.item(), lb.item(), rel_tol=1e-5)
    for n in a.arena.slots:
        ga, gb = a.arena.g(n), b.arena.g(n)
        assert torch.allclose(ga, gb, rtol=1e-5, atol=1e-5 * gb.abs().max().item()), n
    # without document masking the packed row attends across documents and the loss differs
    c = LlamaForCausalLM(cfg, device="cpu", precision="32-true", seed=3)
    assert not math.isclose(c.forward_backward(packed, plab, 1.0).item(), lb.item(), rel_tol=1e-4)
    # the autograd facade takes the same flag
    d = LlamaForCausalLM(cfg, device="cpu", precision="32-true", seed=3)
    d.train()
    loss = d(input_ids=packed, labels=plab, document_mask=True).loss
    loss.backward()
    assert math.isclose(loss.item(), lb.item(), rel_tol=1e-5)
    assert torch.allclose(d.arena.grad, b.arena.grad, rtol=1e-4, atol=1e-6)


def test_mask_shape_is_checked():
    cfg = LlamaConfig(hidden_size=128, intermediate_size=256, num_hidden_layers=1, num_attention_heads=2, vocab_size=512)
    model = LlamaForCausalLM(cfg, device="cpu", precision="32-true", seed=0)
    ids = torch.randint(3, 512, (2, 64))
    with pytest.raises(ValueError):
        model.forward_backward(ids, ids, 1.0, torch.zeros(2, 1, 1, 64))
    with pytest.raises(ValueError):
        model.forward_backward(ids, ids, 1.0, torch.zeros(2, 32))


def test_train_fsdp_document_mask_on_token_shard(tmp_path):
    """--document-mask on a pre-tokenised shard (EOS-separated documents): two optimizer steps on gloo, finite loss."""
    from opendiloco_b200.utils.data import write_token_shard

    g = torch.Generator().manual_seed(0)
    toks = torch.randint(3, 250, (40_000,), generator=g)
    toks[torch.randint(0, toks.numel(), (600,), generator=g)] = EOS
    os.makedirs(tmp_path / "tok")
    write_token_shard(str(tmp_path / "tok" / "shard_0.tok"), toks)
    log = f"{tmp_path}/doc.pkl"
    args = [a for a in BASE if a != "--fake_data"] + ["--dataset_name_or_path", f"tokens:{tmp_path}/tok/*.tok", "--document-mask",
                                                      "--max_steps", "2", "--total_batch_size", "8", "--project", log]
    torchrun(2, "opendiloco_b200.train_fsdp", args)
    with open(log, "rb") as f:
        losses = {d["step"]: d["Loss"] for d in pickle.load(f)}
    assert set(losses) == {1, 2} and all(math.isfinite(v) for v in losses.values())
