"""Causal self-attention over the packed qkv buffer (SURVEY.md §2.5 K5).

Layout contract (chosen so that no transpose is ever materialised): the fused QKV GEMM writes
``qkv[T, (Hq + 2*Hkv) * D]`` with token-major rows; q/k/v are strided *views* ``[B, S, H, D]`` of it and the
attention output is written token-major ``[T, Hq*D]`` so it feeds the o-proj GEMM directly.

Back-ends:
  * ``tc``     - our tcgen05 kernel (``csrc/attn_sm100.cu``), used when built and the shape qualifies
  * ``cudnn``  - cuDNN fused attention through aten (sm_100 kernels; measured 495/444 TF/s fwd/bwd at B32 S1024 H16 D64)
  * ``flash``  - flash-attn 2.8 library kernels (sm_80 mma.sync code: 266/196 TF/s on B200), ODB_ATTN_LIB=flash
  * ``math``   - fp32 PyTorch reference (CPU, tests)
The reference framework itself calls a library here (torch SDPA / flash-attn: train_fsdp.py:107,173).

Padding and per-document masks travel as a ``MaskDesc`` (``kernels.attn_mask_prep``): the ``tc`` back-end runs the
MASKED instantiations of its kernels on it; every other case expands it with ``dense_mask`` - the math reference on the
CPU, torch SDPA with that boolean mask on CUDA.
"""
from __future__ import annotations

import math
import os

import torch

import ctypes
from dataclasses import dataclass

from .. import _lib
from . import kernels as K

_FLASH = None
# Back-end of the bf16 CUDA path: "tc" = our tcgen05 kernels (csrc/attn_sm100.cu, attn_bwd_sm100.cu,
# attn_bwd_d128_sm100.cu; head_dim 64 or 128, S % 128 == 0), "cudnn" / "flash" = the library kernels (kept as comparison
# baselines and for other head sizes).
_LIB = os.environ.get("ODB_ATTN_LIB", "tc")

# Entry points the tcgen05 back-end needs per head size.  A library built before the head_dim-128 kernels existed lacks
# the second set, and such models keep the library path instead of failing.
_TC_SYMBOLS = {
    64: ("odb_attn_fwd", "odb_attn_bwd"),
    128: ("odb_attn_fwd_d128", "odb_attn_bwd_d128", "odb_attn_fwd_d128_masked", "odb_attn_bwd_d128_masked"),
}


def _tc_usable(qkv: torch.Tensor, S: int, Hq: int, Hkv: int, D: int) -> bool:
    return (D in _TC_SYMBOLS and S % 128 == 0 and Hq % Hkv == 0 and qkv.dtype == torch.bfloat16 and qkv.stride(1) == 1
            and qkv.stride(0) % 8 == 0 and all(_lib.has_symbol(n) for n in _TC_SYMBOLS[D]))


def bwd_applies_rope(aux) -> bool:
    """True when ``attention_bwd`` given ``rope=`` already undid the RoPE rotation of dq / dk (our kernels' post-pass)."""
    return isinstance(aux[0], str) and aux[0] == "tc"

_lib.register_optional("odb_attn_fwd", [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p])


_lib.register_optional("odb_attn_bwd", [ctypes.c_void_p] * 11 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 4 + [ctypes.c_float, ctypes.c_void_p])
_lib.register_optional("odb_attn_fwd_masked", [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 2
                       + [ctypes.c_float] + [ctypes.c_void_p] * 4)
_lib.register_optional("odb_attn_bwd_masked", [ctypes.c_void_p] * 11 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 4
                       + [ctypes.c_float] + [ctypes.c_void_p] * 5)
# head_dim 128: the forward takes the same arguments; the backward has no dQ accumulator argument and its masked form
# also takes kv_lo (the dQ kernel walks key tiles like the forward)
_lib.register_optional("odb_attn_fwd_d128", [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_float,
                                             ctypes.c_void_p, ctypes.c_void_p])
_lib.register_optional("odb_attn_fwd_d128_masked", [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 2
                       + [ctypes.c_float] + [ctypes.c_void_p] * 4)
_lib.register_optional("odb_attn_bwd_d128", [ctypes.c_void_p] * 10 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 4
                       + [ctypes.c_float, ctypes.c_void_p])
_lib.register_optional("odb_attn_bwd_d128_masked", [ctypes.c_void_p] * 10 + [ctypes.c_int] * 4 + [ctypes.c_longlong] * 4
                       + [ctypes.c_float] + [ctypes.c_void_p] * 6)
_SCRATCH: dict = {}


@dataclass
class MaskDesc:
    """Per-batch description of a padding and/or per-document causal mask (int32 tensors written by
    ``kernels.attn_mask_prep``, which documents the semantics): lo [B*S], vbits [B, ceil(S/32)], kv_lo / q_hi / lo_hi
    [B, ceil(S/128)]."""
    lo: torch.Tensor
    vbits: torch.Tensor
    kv_lo: torch.Tensor
    q_hi: torch.Tensor
    lo_hi: torch.Tensor

    @classmethod
    def empty(cls, B: int, S: int, device) -> "MaskDesc":
        i32 = dict(dtype=torch.int32, device=device)
        nq = (S + 127) // 128
        return cls(torch.empty(B * S, **i32), torch.empty(B, (S + 31) // 32, **i32), torch.empty(B, nq, **i32),
                   torch.empty(B, nq, **i32), torch.empty(B, nq, **i32))

    def build(self, ids: torch.Tensor, mask: torch.Tensor | None, eos: int) -> "MaskDesc":
        """Describe ``mask`` ([B, S], nonzero = real token; None = all ones) and, with ``eos >= 0``, the documents of ``ids``."""
        K.attn_mask_prep(ids, mask, eos, self.lo, self.vbits, self.kv_lo, self.q_hi, self.lo_hi)
        return self


def dense_mask(desc: MaskDesc, B: int, S: int) -> torch.Tensor:
    """Boolean [B, 1, S, S] mask (True = attend) of a description: ``t == s or (lo[s] <= t < s and valid[t])``."""
    dev = desc.lo.device
    t = torch.arange(S, device=dev)
    valid = ((desc.vbits.long()[:, t // 32] >> (t % 32)) & 1).bool()
    lo = desc.lo.view(B, S).long()
    allowed = (lo[:, :, None] <= t) & (t < t[:, None]) & valid[:, None, :]
    return (allowed | torch.eye(S, dtype=torch.bool, device=dev))[:, None]


def _bwd_scratch(dev, T: int, Hq: int, D: int, masked: bool = False):
    """fp32 dQ accumulator + per-query statistics of the backward kernel (reused across layers / steps: every call
    rewrites them completely before reading).  The masked kernel keeps a third statistics row.  The head_dim-128
    backward writes dQ once, in bf16, and needs no accumulator (None)."""
    key = (dev, T, Hq, D) if not masked else (dev, T, Hq, D, True)
    sc = _SCRATCH.get(key)
    if sc is None:
        sc = (torch.empty(T, Hq * D, dtype=torch.float32, device=dev) if D == 64 else None,
              torch.empty((3 if masked else 2) * T * Hq, dtype=torch.float32, device=dev))
        _SCRATCH[key] = sc
    return sc


def tc_attention_bwd(dout: torch.Tensor, qkv: torch.Tensor, out: torch.Tensor, lse: torch.Tensor, B: int, S: int, Hq: int, Hkv: int,
                     D: int = 64, dqkv: torch.Tensor | None = None, cos: torch.Tensor | None = None, sin: torch.Tensor | None = None,
                     mask: MaskDesc | None = None):
    """Our tcgen05 attention backward.  D = 64 (csrc/attn_bwd_sm100.cu): pre-pass (row statistics, zero dQ accumulator),
    main kernel, post-pass (dQ fp32 -> bf16).  D = 128 (csrc/attn_bwd_d128_sm100.cu): pre-pass, dK/dV kernel, dQ kernel.
    With ``dqkv`` the three gradients land in the column blocks of that packed [T, (Hq+2*Hkv)*D] buffer (returned);
    otherwise returns dense (dq, dk, dv).  With ``cos``/``sin`` dq and dk also leave with the RoPE rotation undone (the
    backward of the fused QKV+RoPE projection epilogue).  ``mask``: the MASKED kernel instantiation."""
    assert D in (64, 128) and S % 128 == 0 and dout.is_contiguous() and out.is_contiguous()
    T = B * S
    dev = qkv.device
    dq_acc, stats = _bwd_scratch(dev, T, Hq, D, masked=mask is not None)
    if dqkv is not None:
        dq, dk, dv = dqkv[:, : Hq * D], dqkv[:, Hq * D:(Hq + Hkv) * D], dqkv[:, (Hq + Hkv) * D:]
    else:
        dq = torch.empty(T, Hq * D, dtype=qkv.dtype, device=dev)
        dk = torch.empty(T, Hkv * D, dtype=qkv.dtype, device=dev)
        dv = torch.empty(T, Hkv * D, dtype=qkv.dtype, device=dev)
    assert dk.stride(0) == dv.stride(0)
    if D == 128:
        args = (qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), stats.data_ptr(), dq.data_ptr(), dk.data_ptr(),
                dv.data_ptr(), cos.data_ptr() if cos is not None else None, sin.data_ptr() if sin is not None else None,
                B, S, Hq, Hkv, qkv.stride(0), out.stride(0), dq.stride(0), dk.stride(0), 1.0 / math.sqrt(D))
        if mask is None:
            _lib.check(_lib.cuda_lib().odb_attn_bwd_d128(*args, _lib.stream_ptr(qkv)), "attn_bwd_d128")
        else:
            _lib.check(_lib.cuda_lib().odb_attn_bwd_d128_masked(*args, mask.lo.data_ptr(), mask.vbits.data_ptr(),
                                                                mask.kv_lo.data_ptr(), mask.q_hi.data_ptr(),
                                                                mask.lo_hi.data_ptr(), _lib.stream_ptr(qkv)),
                       "attn_bwd_d128_masked")
        _lib.count_launch(3)
        return dqkv if dqkv is not None else (dq, dk, dv)
    args = (qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), stats.data_ptr(), dq_acc.data_ptr(), dq.data_ptr(),
            dk.data_ptr(), dv.data_ptr(), cos.data_ptr() if cos is not None else None, sin.data_ptr() if sin is not None else None,
            B, S, Hq, Hkv, qkv.stride(0), out.stride(0), dq.stride(0), dk.stride(0), 1.0 / math.sqrt(D))
    if mask is None:
        _lib.check(_lib.cuda_lib().odb_attn_bwd(*args, _lib.stream_ptr(qkv)), "attn_bwd")
    else:
        _lib.check(_lib.cuda_lib().odb_attn_bwd_masked(*args, mask.lo.data_ptr(), mask.vbits.data_ptr(), mask.q_hi.data_ptr(),
                                                       mask.lo_hi.data_ptr(), _lib.stream_ptr(qkv)), "attn_bwd_masked")
    _lib.count_launch(3)
    return dqkv if dqkv is not None else (dq, dk, dv)


def tc_attention_fwd(qkv: torch.Tensor, B: int, S: int, Hq: int, Hkv: int, D: int = 64, dbg: torch.Tensor | None = None,
                     mask: MaskDesc | None = None):
    """Our tcgen05 causal attention forward.  Returns (out [T, Hq*D] bf16, lse [B, Hq, S] fp32, natural log).
    ``mask``: the MASKED kernel instantiation."""
    assert D in (64, 128) and S % 128 == 0 and qkv.dtype == torch.bfloat16 and qkv.stride(1) == 1
    out = torch.empty(B * S, Hq * D, dtype=qkv.dtype, device=qkv.device)
    lse = torch.empty(B, Hq, S, dtype=torch.float32, device=qkv.device)
    lib = _lib.cuda_lib()
    fwd, fwd_masked = (lib.odb_attn_fwd, lib.odb_attn_fwd_masked) if D == 64 else (lib.odb_attn_fwd_d128, lib.odb_attn_fwd_d128_masked)
    if mask is not None:
        _lib.check(fwd_masked(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, S, Hq, Hkv, qkv.stride(0), out.stride(0),
                              1.0 / math.sqrt(D), mask.lo.data_ptr(), mask.vbits.data_ptr(), mask.kv_lo.data_ptr(),
                              _lib.stream_ptr(qkv)), "attn_fwd_masked")
        _lib.count_launch()
        return out, lse
    _lib.check(fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, S, Hq, Hkv, qkv.stride(0),
                                            out.stride(0), 1.0 / math.sqrt(D), dbg.data_ptr() if dbg is not None else None,
                                            _lib.stream_ptr(qkv)), "attn_fwd")
    _lib.count_launch()
    return out, lse


def _flash():
    global _FLASH
    if _FLASH is None:
        import flash_attn.flash_attn_interface as fi

        _FLASH = fi
    return _FLASH


def split_qkv(qkv: torch.Tensor, B: int, S: int, Hq: int, Hkv: int, D: int):
    """Strided [B,S,H,D] views of the packed buffer (no copies)."""
    row = qkv.shape[1]
    base = qkv.view(B, S, row)
    q = base[:, :, : Hq * D].unflatten(-1, (Hq, D))
    k = base[:, :, Hq * D:(Hq + Hkv) * D].unflatten(-1, (Hkv, D))
    v = base[:, :, (Hq + Hkv) * D:].unflatten(-1, (Hkv, D))
    return q, k, v


def _sdpa_masked_fwd(qkv, mask: MaskDesc, B, S, Hq, Hkv, D):
    """CUDA fallback of the masked cases the tcgen05 kernels do not take: torch SDPA with the dense mask, differentiated
    by autograd in ``attention_bwd``."""
    q, k, v = split_qkv(qkv, B, S, Hq, Hkv, D)
    leaves = [t.detach().transpose(1, 2).requires_grad_(True) for t in (q, k, v)]
    with torch.enable_grad():
        o = torch.nn.functional.scaled_dot_product_attention(leaves[0], leaves[1], leaves[2], attn_mask=dense_mask(mask, B, S),
                                                             enable_gqa=(Hq != Hkv))
        out = o.transpose(1, 2).reshape(B * S, Hq * D)
    return out.detach(), ("sdpa", out, leaves)


def attention_fwd(qkv: torch.Tensor, B: int, S: int, Hq: int, Hkv: int, D: int, mask: MaskDesc | None = None):
    """Returns (out [T, Hq*D], aux).  Causal, scale 1/sqrt(D); ``mask`` restricts it further (see ``MaskDesc``)."""
    q, k, v = split_qkv(qkv, B, S, Hq, Hkv, D)
    scale = 1.0 / math.sqrt(D)
    if mask is not None and qkv.is_cuda:
        if _LIB == "tc" and _tc_usable(qkv, S, Hq, Hkv, D):
            if not (_lib.has_symbol("odb_attn_fwd_masked") and _lib.has_symbol("odb_attn_bwd_masked")):
                raise _lib.NativeLibraryMissing("libodb200.so lacks the masked attention kernels: rebuild it")
            out, lse = tc_attention_fwd(qkv, B, S, Hq, Hkv, D, mask=mask)
            return out, ("tc", lse)
        return _sdpa_masked_fwd(qkv, mask, B, S, Hq, Hkv, D)
    if qkv.is_cuda and qkv.dtype in (torch.bfloat16, torch.float16):
        if _LIB == "tc" and _tc_usable(qkv, S, Hq, Hkv, D):
            out, lse = tc_attention_fwd(qkv, B, S, Hq, Hkv, D)
            return out, ("tc", lse)
        if _LIB != "flash":
            r = torch.ops.aten._scaled_dot_product_cudnn_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), None,
                                                                   True, 0.0, True, False, scale=scale)
            out = r[0].transpose(1, 2)          # cuDNN keeps the [B,S,H,D] memory layout of q
            if not out.is_contiguous():
                out = out.contiguous()
            return out.view(B * S, Hq * D), ("cudnn", r)
        out, lse, _, rng = _flash()._flash_attn_forward(q, k, v, 0.0, scale, True, -1, -1, 0.0, None, False)
        return out.view(B * S, Hq * D), (lse, rng)
    # fp32 math reference
    qf, kf, vf = (t.float().permute(0, 2, 1, 3) for t in (q, k, v))
    if Hkv != Hq:
        rep = Hq // Hkv
        kf, vf = kf.repeat_interleave(rep, dim=1), vf.repeat_interleave(rep, dim=1)
    att = (qf @ kf.transpose(-1, -2)) * scale
    allowed = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril() if mask is None else dense_mask(mask, B, S)
    att = att.masked_fill(~allowed, float("-inf"))
    lse = torch.logsumexp(att, dim=-1)
    p = torch.softmax(att, dim=-1)
    out = (p @ vf).permute(0, 2, 1, 3).reshape(B * S, Hq * D).to(qkv.dtype)
    return out, (lse, None)


def attention_bwd(dout: torch.Tensor, qkv: torch.Tensor, out: torch.Tensor, aux, dqkv: torch.Tensor, B: int, S: int,
                  Hq: int, Hkv: int, D: int, want_parts: bool = False, rope=None, mask: MaskDesc | None = None):
    """Writes dq|dk|dv into the packed ``dqkv`` buffer (same layout as qkv) and returns it - or, with ``want_parts`` and a
    back-end that produces separate dense gradients, returns the tuple (dq [T,Hq*D], dk [T,Hkv*D], dv [T,Hkv*D]).
    ``rope=(cos, sin)``: a back-end for which ``bwd_applies_rope(aux)`` holds also undoes the rotation of dq / dk.
    ``mask``: the description the forward ran with."""
    if isinstance(aux[0], str) and aux[0] == "tc":
        cos, sin = rope if rope is not None else (None, None)
        return tc_attention_bwd(dout, qkv, out, aux[1], B, S, Hq, Hkv, D, dqkv=dqkv, cos=cos, sin=sin, mask=mask)
    if isinstance(aux[0], str) and aux[0] == "sdpa":
        gq, gk, gv = torch.autograd.grad(aux[1], aux[2], dout)
        dq, dk, dv = split_qkv(dqkv, B, S, Hq, Hkv, D)
        dq.copy_(gq.transpose(1, 2))
        dk.copy_(gk.transpose(1, 2))
        dv.copy_(gv.transpose(1, 2))
        return dqkv
    q, k, v = split_qkv(qkv, B, S, Hq, Hkv, D)
    dq, dk, dv = split_qkv(dqkv, B, S, Hq, Hkv, D)
    scale = 1.0 / math.sqrt(D)
    lse, rng = aux
    if isinstance(lse, str) and lse == "cudnn":
        r = rng
        g = torch.ops.aten._scaled_dot_product_cudnn_attention_backward(
            dout.view(B, S, Hq, D).transpose(1, 2), q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), r[0], r[1], r[6],
            r[7], None, r[2], r[3], r[4], r[5], 0.0, True, scale=scale)
        if want_parts:
            # cuDNN hands back three dense [B,S,H,D] tensors: give them to the caller as [T, H*D] matrices instead of
            # spending three strided copies on packing them (the dgrad GEMM reads its A operand from three tensors)
            parts = [t.transpose(1, 2) for t in g[:3]]
            if all(t.is_contiguous() for t in parts):
                return parts[0].reshape(B * S, Hq * D), parts[1].reshape(B * S, Hkv * D), parts[2].reshape(B * S, Hkv * D)
        dq.copy_(g[0].transpose(1, 2))
        dk.copy_(g[1].transpose(1, 2))
        dv.copy_(g[2].transpose(1, 2))
        return dqkv
    if qkv.is_cuda and qkv.dtype in (torch.bfloat16, torch.float16):
        _flash()._flash_attn_backward(dout.view(B, S, Hq, D), q, k, v, out.view(B, S, Hq, D), lse, dq, dk, dv, 0.0, scale,
                                      True, -1, -1, 0.0, None, False, rng)
        return dqkv
    qf, kf, vf = (t.float().permute(0, 2, 1, 3) for t in (q, k, v))
    rep = Hq // Hkv
    if rep != 1:
        kf, vf = kf.repeat_interleave(rep, dim=1), vf.repeat_interleave(rep, dim=1)
    att = (qf @ kf.transpose(-1, -2)) * scale
    allowed = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril() if mask is None else dense_mask(mask, B, S)
    att = att.masked_fill(~allowed, float("-inf"))
    p = torch.softmax(att, dim=-1)
    do = dout.float().view(B, S, Hq, D).permute(0, 2, 1, 3)
    dvf = p.transpose(-1, -2) @ do
    dp = do @ vf.transpose(-1, -2)
    ds = p * (dp - (dp * p).sum(-1, keepdim=True))
    dqf = (ds @ kf) * scale
    dkf = (ds.transpose(-1, -2) @ qf) * scale
    if rep != 1:
        dkf = dkf.view(B, Hkv, rep, S, D).sum(2)
        dvf = dvf.view(B, Hkv, rep, S, D).sum(2)
    dq.copy_(dqf.permute(0, 2, 1, 3).to(dqkv.dtype))
    dk.copy_(dkf.permute(0, 2, 1, 3).to(dqkv.dtype))
    dv.copy_(dvf.permute(0, 2, 1, 3).to(dqkv.dtype))
    return dqkv
