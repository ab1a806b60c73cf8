"""Head size 128 without a GPU: the config's head_dim key, the tcgen05 dispatch predicate per head size, and the fp32
math reference at D = 128."""
import json

import pytest
import torch

from opendiloco_b200 import LlamaConfig
from opendiloco_b200.ops import attention as A


def _d128_dict(**extra):
    d = dict(hidden_size=1024, intermediate_size=2816, num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=4,
             vocab_size=32000)
    d.update(extra)
    return d


def test_head_dim_accepted_when_it_matches(tmp_path):
    assert LlamaConfig.from_dict(_d128_dict(head_dim=128)).head_dim == 128
    assert LlamaConfig.from_dict(_d128_dict(head_dim=None)).head_dim == 128      # HF writes null for "derived"
    assert LlamaConfig.from_dict(_d128_dict()).head_dim == 128
    p = tmp_path / "config.json"
    p.write_text(json.dumps(_d128_dict(head_dim=128)))
    assert LlamaConfig.from_pretrained(str(p)).head_dim == 128
    for preset in ("2m", "14m", "60m", "150m", "1b"):                            # every preset carries a matching key
        LlamaConfig.from_pretrained(preset)


def test_head_dim_rejected_when_it_differs(tmp_path):
    with pytest.raises(ValueError, match=r"head_dim 64 .*1024 / 8 = 128"):
        LlamaConfig.from_dict(_d128_dict(head_dim=64))
    p = tmp_path / "config.json"
    p.write_text(json.dumps(_d128_dict(head_dim=256)))
    with pytest.raises(ValueError, match="head_dim 256"):
        LlamaConfig.from_pretrained(str(p))


D64_SYMBOLS = {"odb_attn_fwd", "odb_attn_bwd", "odb_attn_fwd_masked", "odb_attn_bwd_masked"}
D128_SYMBOLS = {"odb_attn_fwd_d128", "odb_attn_bwd_d128", "odb_attn_fwd_d128_masked", "odb_attn_bwd_d128_masked"}


@pytest.mark.parametrize("library,usable", [
    (D64_SYMBOLS | D128_SYMBOLS, {32: False, 64: True, 96: False, 128: True}),
    (D64_SYMBOLS, {32: False, 64: True, 96: False, 128: False}),                  # built before the D = 128 kernels
    (D64_SYMBOLS | D128_SYMBOLS - {"odb_attn_bwd_d128_masked"}, {32: False, 64: True, 96: False, 128: False}),
    (set(), {32: False, 64: False, 96: False, 128: False}),
])
def test_tc_usable_per_head_size(library, usable, monkeypatch):
    monkeypatch.setattr(A._lib, "has_symbol", lambda name: name in library)
    S, Hq, Hkv = 256, 8, 4
    for D, want in usable.items():
        qkv = torch.empty(2 * S, (Hq + 2 * Hkv) * D, dtype=torch.bfloat16)
        assert A._tc_usable(qkv, S, Hq, Hkv, D) == want, D
    qkv = torch.empty(2 * S, (Hq + 2 * Hkv) * 128, dtype=torch.bfloat16)
    assert not A._tc_usable(qkv, 200, Hq, Hkv, 128)                               # S % 128 != 0
    assert not A._tc_usable(qkv.float(), S, Hq, Hkv, 128)                         # bf16 only


@pytest.mark.parametrize("Hq,Hkv", [(4, 4), (4, 2)])
def test_math_reference_all_ones_description_is_causal(Hq, Hkv):
    B, S, D = 2, 256, 128
    torch.manual_seed(0)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D)
    desc = A.MaskDesc.empty(B, S, "cpu").build(torch.randint(3, 1000, (B, S)), None, -1)
    out_c, aux_c = A.attention_fwd(qkv, B, S, Hq, Hkv, D)
    out_m, aux_m = A.attention_fwd(qkv, B, S, Hq, Hkv, D, mask=desc)
    assert torch.equal(out_c, out_m) and torch.equal(aux_c[0], aux_m[0])
    dout = torch.randn_like(out_c)
    gc = A.attention_bwd(dout, qkv, out_c, aux_c, torch.empty_like(qkv), B, S, Hq, Hkv, D)
    gm = A.attention_bwd(dout, qkv, out_m, aux_m, torch.empty_like(qkv), B, S, Hq, Hkv, D, mask=desc)
    assert torch.equal(gc, gm)
    # and the causal reference is the plain softmax attention of q . k / sqrt(128)
    q, k, v = (t.permute(0, 2, 1, 3) for t in A.split_qkv(qkv, B, S, Hq, Hkv, D))
    k, v = k.repeat_interleave(Hq // Hkv, dim=1), v.repeat_interleave(Hq // Hkv, dim=1)
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True)
    assert torch.allclose(out_c, ref.permute(0, 2, 1, 3).reshape(B * S, Hq * D), atol=1e-5)
