"""Python front-end of the sm_100a kernels (``csrc/*.cu``) with a PyTorch reference beside each op.

Dispatch rule (there is exactly one): CUDA tensors -> our kernel (raises if the library is not built);
CPU tensors -> the reference implementation below, written to reproduce the same rounding points
(bf16 storage, fp32 statistics) so the CPU suite is a numerics oracle for the GPU suite.

All ops take pre-allocated outputs where the training engine owns the buffers.
"""
from __future__ import annotations

import math

import torch

from .. import _lib

BF16 = torch.bfloat16


def _p(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _chk_bf16(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None:
            assert t.dtype == BF16 and t.is_contiguous(), (t.dtype, t.stride())


# ------------------------------------------------------------------------------------------------ embedding
def embedding_fwd(ids: torch.Tensor, weight: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """out[t] = weight[ids[t]] ; ids int64 [T], weight bf16 [V, h].  (SURVEY K1; modeling_llama.py:389)"""
    T, h = ids.numel(), weight.shape[1]
    if out is None:
        out = torch.empty(T, h, dtype=weight.dtype, device=weight.device)
    if weight.is_cuda and weight.dtype == BF16:
        _chk_bf16(weight, out)
        assert ids.dtype == torch.int64 and ids.is_contiguous()
        _lib.check(_lib.cuda_lib().odb_embedding_fwd(_p(ids), _p(weight), _p(out), T, h, _lib.stream_ptr(out)), "embedding_fwd")
        _lib.count_launch()
    else:
        torch.index_select(weight, 0, ids.reshape(-1), out=out)
    return out


def embedding_bwd(ids: torch.Tensor, dout: torch.Tensor, dweight: torch.Tensor, scale: float = 1.0) -> None:
    """dweight[ids[t]] += scale * dout[t]  (fp32 accumulate)."""
    T, h = ids.numel(), dweight.shape[1]
    if dweight.is_cuda and dout.dtype == BF16:
        _chk_bf16(dout)
        assert dweight.dtype == torch.float32 and dweight.is_contiguous()
        _lib.check(_lib.cuda_lib().odb_embedding_bwd(_p(ids), _p(dout), _p(dweight), T, h, float(scale), _lib.stream_ptr(dout)),
                   "embedding_bwd")
        _lib.count_launch()
    else:
        dweight.index_add_(0, ids.reshape(-1), dout.reshape(T, h).float(), alpha=scale)


# ------------------------------------------------------------------------------------------------ RMSNorm
def rmsnorm_fwd(x: torch.Tensor, w: torch.Tensor, eps: float, delta: torch.Tensor | None = None,
                out: torch.Tensor | None = None, rstd: torch.Tensor | None = None, x_out: torch.Tensor | None = None):
    """x_new = bf16(x + delta) (stored to x_out, default in place) ; y = w * bf16(x_new * rsqrt(mean(x_new^2)+eps)).

    Returns (y, rstd).  Rounding points follow HF LlamaRMSNorm (modeling_llama.py:62-67): statistics in fp32,
    normalised value cast to the activation dtype before the weight multiply.
    """
    T, h = x.shape
    if out is None:
        out = torch.empty_like(x)
    if rstd is None:
        rstd = torch.empty(T, dtype=torch.float32, device=x.device)
    if x_out is None:
        x_out = x
    if x.is_cuda and x.dtype == BF16:
        _chk_bf16(x, w, out, delta, x_out)
        _lib.check(_lib.cuda_lib().odb_rmsnorm_fwd(_p(x), _p(x_out), _p(delta), _p(w), _p(out), _p(rstd), T, h, float(eps),
                                                   _lib.stream_ptr(x)), "rmsnorm_fwd")
        _lib.count_launch()
    else:
        if delta is not None:
            x_out.copy_((x.float() + delta.float()).to(x.dtype))
            x = x_out
        xf = x.float()
        r = torch.rsqrt(xf.pow(2).mean(-1) + eps)
        rstd.copy_(r)
        out.copy_((w.float() * (xf * r[:, None]).to(x.dtype).float()).to(x.dtype))
    return out, rstd


def rmsnorm_bwd(dy: torch.Tensor, x: torch.Tensor, w: torch.Tensor, rstd: torch.Tensor, dres_in: torch.Tensor | None,
                dres_out: torch.Tensor, dw: torch.Tensor) -> None:
    """dres_out = (dres_in or 0) + dx ; dw += sum_t dy * bf16(xhat)   (dw fp32 [h], accumulated)."""
    T, h = x.shape
    if x.is_cuda and x.dtype == BF16:
        _chk_bf16(dy, x, w, dres_in, dres_out)
        assert dw.dtype == torch.float32
        _lib.check(_lib.cuda_lib().odb_rmsnorm_bwd(_p(dy), _p(x), _p(w), _p(rstd), _p(dres_in), _p(dres_out), _p(dw), T, h,
                                                   _lib.stream_ptr(x)), "rmsnorm_bwd")
        _lib.count_launch()
    else:
        xf, dyf = x.float(), dy.float()
        xh = xf * rstd[:, None]
        g = dyf * w.float()
        dot = (g * xh).mean(-1, keepdim=True)
        dx = rstd[:, None] * (g - xh * dot)
        if dres_in is not None:
            dx = dx + dres_in.float()
        dw.add_((dyf * xh.to(x.dtype).float()).sum(0))
        dres_out.copy_(dx.to(dres_out.dtype))


# ------------------------------------------------------------------------------------------------ RoPE
def rope_tables(S: int, D: int, theta: float, device) -> tuple[torch.Tensor, torch.Tensor]:
    """fp32 cos/sin tables [S, D/2] (HF LlamaRotaryEmbedding, modeling_llama.py:117-135: inv_freq = theta^(-2i/D))."""
    inv_freq = 1.0 / (theta ** (torch.arange(0, D, 2, dtype=torch.float32, device=device) / D))
    pos = torch.arange(S, dtype=torch.float32, device=device)
    freqs = torch.outer(pos, inv_freq)
    return freqs.cos().contiguous(), freqs.sin().contiguous()


def rope_(qkv: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, S: int, n_rot_heads: int, D: int,
          backward: bool = False) -> torch.Tensor:
    """Rotate, in place, the first n_rot_heads*D columns (q heads then k heads) of qkv [T, row]; position = t % S."""
    T, row = qkv.shape
    if qkv.is_cuda and qkv.dtype == BF16:
        _chk_bf16(qkv)
        _lib.check(_lib.cuda_lib().odb_rope(_p(qkv), _p(cos), _p(sin), T, S, n_rot_heads, D, row, -1.0 if backward else 1.0,
                                            _lib.stream_ptr(qkv)), "rope")
        _lib.count_launch()
    else:
        half = D // 2
        v = qkv[:, : n_rot_heads * D].float().reshape(T // S, S, n_rot_heads, D)
        a, b = v[..., :half], v[..., half:]
        c = cos[None, :, None, :]
        s = sin[None, :, None, :] * (-1.0 if backward else 1.0)
        out = torch.cat([a * c - b * s, b * c + a * s], dim=-1).reshape(T, n_rot_heads * D)
        qkv[:, : n_rot_heads * D] = out.to(qkv.dtype)
    return qkv


# ------------------------------------------------------------------------------------------------ SwiGLU
def swiglu_fwd(gu: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """gu [T, 2I] = [gate | up] -> silu(gate) * up  [T, I]   (modeling_llama.py:182-184)."""
    T, two_i = gu.shape
    I = two_i // 2
    if out is None:
        out = torch.empty(T, I, dtype=gu.dtype, device=gu.device)
    if gu.is_cuda and gu.dtype == BF16:
        _chk_bf16(gu, out)
        _lib.check(_lib.cuda_lib().odb_swiglu_fwd(_p(gu), _p(out), T, I, _lib.stream_ptr(gu)), "swiglu_fwd")
        _lib.count_launch()
    else:
        g, u = gu[:, :I].float(), gu[:, I:].float()
        out.copy_((g * torch.sigmoid(g) * u).to(out.dtype))
    return out


def swiglu_bwd(da: torch.Tensor, gu: torch.Tensor, dgu: torch.Tensor | None = None) -> torch.Tensor:
    """Gradient w.r.t. [gate | up]; dgu may alias gu."""
    T, two_i = gu.shape
    I = two_i // 2
    if dgu is None:
        dgu = torch.empty_like(gu)
    if gu.is_cuda and gu.dtype == BF16:
        _chk_bf16(da, gu, dgu)
        _lib.check(_lib.cuda_lib().odb_swiglu_bwd(_p(da), _p(gu), _p(dgu), T, I, _lib.stream_ptr(gu)), "swiglu_bwd")
        _lib.count_launch()
    else:
        g, u, d = gu[:, :I].float(), gu[:, I:].float(), da.float()
        sg = torch.sigmoid(g)
        dg = d * u * sg * (1 + g * (1 - sg))
        du = d * g * sg
        dgu.copy_(torch.cat([dg, du], dim=1).to(dgu.dtype))
    return dgu


# ------------------------------------------------------------------------------------------------ casts
def cast_to_bf16(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    n = src.numel()
    if src.is_cuda and n % 8 == 0:
        assert src.dtype == torch.float32 and dst.dtype == BF16
        _lib.check(_lib.cuda_lib().odb_cast_f32_bf16(_p(src), _p(dst), n, _lib.stream_ptr(src)), "cast_f32_bf16")
        _lib.count_launch()
    else:
        dst.copy_(src)
    return dst


# ------------------------------------------------------------------------------------------------ cross entropy on a logits tile
def ce_fwd_bwd_(logits: torch.Tensor, labels: torch.Tensor, gscale: torch.Tensor, loss_sum: torch.Tensor,
                sumsq: torch.Tensor | None = None) -> None:
    """In place: logits [R, V] bf16 -> dlogits = (softmax - onehot) * gscale ; loss_sum += sum_r (lse - x_y).

    labels int64 [R] with -100 = ignore ; gscale, loss_sum: fp32 device scalars (shape [1]).
    sumsq (optional) += sum of squared logits (the lm_head activation-norm metric, reference utils.py:35).
    """
    R, V = logits.shape
    if logits.is_cuda and logits.dtype == BF16:
        assert logits.stride(1) == 1
        _lib.check(_lib.cuda_lib().odb_ce_fwd_bwd(_p(logits), _p(labels), R, V, logits.stride(0), _p(gscale), _p(loss_sum),
                                                  None, _p(sumsq), _lib.stream_ptr(logits)), "ce_fwd_bwd")
        _lib.count_launch()
    else:
        x = logits.float()
        if sumsq is not None:
            sumsq.add_(x.pow(2).sum())
        valid = labels >= 0
        lse = torch.logsumexp(x, dim=-1)
        safe = labels.clamp(min=0)
        xy = x.gather(1, safe[:, None])[:, 0]
        loss_sum.add_(((lse - xy) * valid).sum())
        p = torch.softmax(x, dim=-1)
        p.scatter_add_(1, safe[:, None], -torch.ones_like(p[:, :1]))
        p = p * gscale * valid[:, None]
        logits.copy_(p.to(logits.dtype))


def ce_fwd(logits: torch.Tensor, labels: torch.Tensor, loss_sum: torch.Tensor) -> None:
    R, V = logits.shape
    if logits.is_cuda and logits.dtype == BF16:
        assert logits.stride(1) == 1
        _lib.check(_lib.cuda_lib().odb_ce_fwd(_p(logits), _p(labels), R, V, logits.stride(0), _p(loss_sum),
                                              _lib.stream_ptr(logits)), "ce_fwd")
        _lib.count_launch()
    else:
        x = logits.float()
        valid = labels >= 0
        lse = torch.logsumexp(x, dim=-1)
        xy = x.gather(1, labels.clamp(min=0)[:, None])[:, 0]
        loss_sum.add_(((lse - xy) * valid).sum())


# ------------------------------------------------------------------------------------------------ fused linear-cross-entropy helpers
import ctypes as _ct

_lib.register_optional("odb_lce_prep", [_ct.c_void_p, _ct.c_void_p, _ct.c_int, _ct.c_int, _ct.c_float, _ct.c_void_p, _ct.c_void_p,
                                       _ct.c_void_p, _ct.c_void_p])
_lib.register_optional("odb_lce_label_dot", [_ct.c_void_p, _ct.c_longlong, _ct.c_void_p, _ct.c_longlong, _ct.c_void_p, _ct.c_void_p,
                                            _ct.c_int, _ct.c_int, _ct.c_void_p])
_lib.register_optional("odb_lce_finalize", [_ct.c_void_p, _ct.c_int, _ct.c_int, _ct.c_void_p, _ct.c_void_p, _ct.c_void_p, _ct.c_void_p,
                                           _ct.c_void_p, _ct.c_void_p, _ct.c_longlong, _ct.c_void_p, _ct.c_longlong, _ct.c_void_p,
                                           _ct.c_longlong, _ct.c_int, _ct.c_void_p])


def lce_prep(labels_in: torch.Tensor, labels_out: torch.Tensor, B: int, S: int, loss_scale: float, n_valid: torch.Tensor,
             gscale: torch.Tensor, loss_sum: torch.Tensor) -> None:
    """HF label shift (position s predicts token s+1, last position of every sequence ignored; loss_utils.py:45-67) +
    n_valid = max(#labels >= 0, 1) + gscale = loss_scale / n_valid + loss_sum = 0, in one launch."""
    if labels_out.is_cuda:
        assert labels_in.dtype == torch.int64 and labels_in.is_contiguous() and labels_out.is_contiguous()
        _lib.check(_lib.cuda_lib().odb_lce_prep(_p(labels_in), _p(labels_out), B, S, float(loss_scale), _p(n_valid), _p(gscale),
                                                _p(loss_sum), _lib.stream_ptr(labels_out)), "lce_prep")
        _lib.count_launch()
        return
    lab = labels_out.view(B, S)
    lab[:, : S - 1].copy_(labels_in.reshape(B, S)[:, 1:])
    lab[:, S - 1].fill_(-100)
    n_valid.copy_((labels_out >= 0).sum().to(torch.float32).clamp(min=1.0).reshape(1))
    gscale.copy_(float(loss_scale) / n_valid)
    loss_sum.zero_()


def lce_label_dot(x: torch.Tensor, w: torch.Tensor, labels: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[t] = x[t] . w[labels[t]] + 40 in fp32 (0 for ignored rows): the shift of the exponentials of the fused LCE
    (40 nats of head-room above the label logit, see csrc/lce.cu)."""
    T, h = x.shape
    if x.is_cuda and x.dtype == BF16:
        _lib.check(_lib.cuda_lib().odb_lce_label_dot(_p(x), x.stride(0), _p(w), w.stride(0), _p(labels), _p(out), T, h,
                                                     _lib.stream_ptr(x)), "lce_label_dot")
        _lib.count_launch()
    else:
        safe = labels.clamp(min=0)
        out.copy_(((x.float() * w.float()[safe]).sum(-1) + 40.0) * (labels >= 0))
    return out


def lce_finalize(partials: torch.Tensor, planes: int, labels: torch.Tensor, gscale: torch.Tensor, loss_sum: torch.Tensor,
                 sumsq: torch.Tensor | None, rowscale: torch.Tensor | None, x: torch.Tensor, xs: torch.Tensor | None,
                 dw: torch.Tensor | None) -> None:
    """Row sums of the partial planes -> loss_sum += sum_t log S_t ; rowscale = gscale / S ; xs = bf16(rowscale * x) ;
    dw[labels[t]] -= gscale * x[t] (the one-hot term of the LM-head weight gradient).  CUDA only (the CPU path of the
    engine uses the materialising reference)."""
    T, h = x.shape
    _lib.check(_lib.cuda_lib().odb_lce_finalize(_p(partials), planes, T, _p(labels), _p(gscale), _p(loss_sum), _p(sumsq),
                                                _p(rowscale), _p(x), x.stride(0), _p(xs), xs.stride(0) if xs is not None else 0,
                                                _p(dw), dw.stride(0) if dw is not None else 0, h, _lib.stream_ptr(x)),
               "lce_finalize")
    _lib.count_launch()


# ------------------------------------------------------------------------------------------------ optimizer kernels
HP_LR, HP_B1, HP_B2, HP_EPS, HP_WD, HP_BC1, HP_BC2, HP_MAXNORM, HP_INVSCALE = range(9)
HP_SIZE = 16
MAX_PARTIALS = 2048


def grad_sqnorm(g: torch.Tensor, partials: torch.Tensor, flag: torch.Tensor) -> int:
    """Per-CTA partial sums of squares of the flat fp32 gradient; returns the number of partials written."""
    n = g.numel()
    if g.is_cuda:
        assert g.dtype == torch.float32 and n % 4 == 0
        rc = _lib.cuda_lib().odb_grad_sqnorm(_p(g), n, _p(partials), _p(flag), _lib.stream_ptr(g))
        if rc <= 0:
            raise RuntimeError(f"grad_sqnorm failed: {rc}")
        _lib.count_launch()
        return rc
    partials[0] = g.double().pow(2).sum().float()
    if not torch.isfinite(partials[0]):
        flag.fill_(1)
    return 1


def adamw_step(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, shadow: torch.Tensor | None,
               hp: torch.Tensor, partials: torch.Tensor, n_partials: int, found_inf: torch.Tensor | None,
               stats: torch.Tensor | None, zero_grad: bool = True) -> None:
    """Fused clip + AdamW + bf16 shadow + zero-grad over the flat arena.  hp: fp32 [HP_SIZE] on the same device.

    Math is torch.optim.AdamW's (decoupled decay, lerp'd first moment, bias-corrected): reference inner optimizer
    train_fsdp.py:250 / train_diloco_torch.py:186 ; clipping = clip_grad_norm_(1.0) train_fsdp.py:395.
    """
    n = p.numel()
    if p.is_cuda:
        assert n % 4 == 0
        _lib.check(_lib.cuda_lib().odb_adamw_step(_p(p), _p(g), _p(m), _p(v), _p(shadow), n, _p(hp), _p(partials), n_partials,
                                                  _p(found_inf), _p(stats), int(zero_grad), _lib.stream_ptr(p)), "adamw_step")
        _lib.count_launch()
        return
    lr, b1, b2, eps, wd, bc1, bc2, max_norm, inv_scale = (float(hp[i]) for i in range(9))
    gnorm = math.sqrt(float(partials[:n_partials].sum())) * inv_scale
    coef, clip = inv_scale, 1.0
    if max_norm > 0:
        clip = min(1.0, max_norm / (gnorm + 1e-6))
        coef *= clip
    if stats is not None:
        stats[0], stats[1] = gnorm, clip
    skip = found_inf is not None and int(found_inf.item()) != 0
    if not skip:
        gr = g * coef
        p.mul_(1 - lr * wd)
        m.lerp_(gr, 1 - b1)
        v.mul_(b2).addcmul_(gr, gr, value=1 - b2)
        denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
        p.addcdiv_(m, denom, value=-lr / bc1)
        if shadow is not None:
            shadow.copy_(p)
    if zero_grad:
        g.zero_()


_lib.register_optional("odb_checksum_i32", [_ct.c_void_p, _ct.c_longlong, _ct.c_void_p, _ct.c_void_p])


def checksum_i32(buf: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """Wrap-around integer checksum of the 32-bit words of ``buf`` (int64 scalar tensor): exact and order independent, so
    two workers hold bit-identical buffers iff the values agree.  CUDA: one pass at HBM speed; CPU: torch sum."""
    if out is None:
        out = torch.zeros(1, dtype=torch.int64, device=buf.device)
    else:
        out.zero_()
    words = buf.view(torch.int32) if buf.element_size() == 4 else buf.view(torch.int16).to(torch.int32)
    if buf.is_cuda and words.numel() % 4 == 0 and buf.element_size() == 4 and _lib.has_symbol("odb_checksum_i32"):
        _lib.check(_lib.cuda_lib().odb_checksum_i32(_p(buf), words.numel(), _p(out), _lib.stream_ptr(buf)), "checksum_i32")
        _lib.count_launch()
    else:
        out.add_(words.sum(dtype=torch.int64))
    return out


def pseudo_grad(theta_outer: torch.Tensor, theta_local: torch.Tensor, delta: torch.Tensor) -> torch.Tensor:
    """delta = theta_outer - theta_local (fp32 or bf16 out).  reference: train_diloco_torch.py:344, hivemind_diloco.py:166"""
    n = theta_outer.numel()
    if theta_outer.is_cuda and n % 4 == 0:
        _lib.check(_lib.cuda_lib().odb_pseudo_grad(_p(theta_outer), _p(theta_local), _p(delta), n, int(delta.dtype == BF16),
                                                   _lib.stream_ptr(delta)), "pseudo_grad")
        _lib.count_launch()
    else:
        delta.copy_(theta_outer - theta_local)
    return delta


def nesterov_outer(theta_outer: torch.Tensor, buf: torch.Tensor, delta: torch.Tensor | None, theta_local: torch.Tensor,
                   shadow: torch.Tensor | None, lr: float, momentum: float, nesterov: bool, dscale: float = 1.0) -> None:
    """torch.optim.SGD(momentum, nesterov) step on theta_outer with gradient dscale*delta, then
    theta_local <- theta_outer (and the bf16 shadow).  delta=None: single-worker form, delta computed in-kernel.
    reference: train_diloco_torch.py:346-353 ; SGD formula ENV/torch/optim/sgd.py:358-367."""
    n = theta_outer.numel()
    if theta_outer.is_cuda and n % 4 == 0:
        _lib.check(_lib.cuda_lib().odb_nesterov_outer(_p(theta_outer), _p(buf), _p(delta),
                                                      int(delta is not None and delta.dtype == BF16), _p(theta_local),
                                                      _p(shadow), n, float(lr), float(momentum), int(nesterov), float(dscale),
                                                      _lib.stream_ptr(theta_outer)), "nesterov_outer")
        _lib.count_launch()
        return
    d = (theta_outer - theta_local) if delta is None else delta.float()
    d = d * dscale
    buf.mul_(momentum).add_(d)
    step = d + momentum * buf if nesterov else buf
    theta_outer.sub_(lr * step)
    theta_local.copy_(theta_outer)
    if shadow is not None:
        shadow.copy_(theta_outer)


# ------------------------------------------------------------------------------------------------ attention mask description
_lib.register_optional("odb_attn_mask_prep", [_ct.c_void_p, _ct.c_void_p, _ct.c_int, _ct.c_int, _ct.c_int, _ct.c_longlong]
                       + [_ct.c_void_p] * 6)


def attn_mask_prep(ids: torch.Tensor, mask: torch.Tensor | None, eos: int, lo: torch.Tensor, vbits: torch.Tensor,
                   kv_lo: torch.Tensor, q_hi: torch.Tensor, lo_hi: torch.Tensor) -> None:
    """Compact description of a padding and/or per-document causal mask (outputs int32, written in place).

    For row b, query s and key t: ``valid[t] = mask[b, t] != 0`` (all ones without a mask); ``docstart[s]`` = 0, or 1 + the
    last p < s with ``ids[b, p] == eos`` (``eos < 0``: no document masking); ``lo[s] = min(s, first t >= docstart[s] with
    valid[t])``; attention is allowed where ``t == s or (lo[s] <= t < s and valid[t])``.

    lo [B*S]; vbits [B, ceil(S/32)] (bit t%32 of word t//32 = valid[t]); per 128-query tile qt: kv_lo = min lo // 128 and
    lo_hi = max lo; per 128-key tile kt: q_hi = max{qt : kv_lo[qt] <= kt}.  ids int64 [B, S]; mask [B, S] of any integer
    or bool dtype."""
    B, S = ids.shape
    if ids.is_cuda:
        assert ids.dtype == torch.int64 and ids.is_contiguous()
        assert mask is None or (mask.shape == ids.shape and mask.is_contiguous() and mask.device == ids.device)
        for t in (lo, vbits, kv_lo, q_hi, lo_hi):
            assert t.dtype == torch.int32 and t.is_contiguous()
        _lib.check(_lib.cuda_lib().odb_attn_mask_prep(_p(ids), _p(mask), mask.element_size() if mask is not None else 0, B, S,
                                                      int(eos), _p(lo), _p(vbits), _p(kv_lo), _p(q_hi), _p(lo_hi),
                                                      _lib.stream_ptr(ids)), "attn_mask_prep")
        _lib.count_launch()
        return
    dev = ids.device
    pos = torch.arange(S, device=dev)
    valid = torch.ones(B, S, dtype=torch.bool, device=dev) if mask is None else (mask != 0)
    if eos >= 0:
        after = torch.where(ids == eos, pos + 1, 0).cummax(dim=1).values      # 1 + last EOS at or before p
        docstart = torch.cat([torch.zeros(B, 1, dtype=after.dtype, device=dev), after[:, :-1]], dim=1)
    else:
        docstart = torch.zeros(B, S, dtype=torch.int64, device=dev)
    nv = torch.where(valid, pos, S).flip(1).cummin(dim=1).values.flip(1)     # first valid position >= p
    l = torch.minimum(pos[None], nv.gather(1, docstart))
    lo.copy_(l.reshape(-1))
    nw, nq = (S + 31) // 32, (S + 127) // 128
    vb = torch.zeros(B, nw * 32, dtype=torch.int64, device=dev)
    vb[:, :S] = valid.long()
    w = (vb.view(B, nw, 32) << torch.arange(32, device=dev)).sum(-1)
    vbits.copy_(torch.where(w >= 2 ** 31, w - 2 ** 32, w))
    lp = torch.full((B, nq * 128), S, dtype=torch.int64, device=dev)
    lp[:, :S] = l
    kmin = lp.view(B, nq, 128).amin(-1)
    lp[:, S:] = -1
    lo_hi.copy_(lp.view(B, nq, 128).amax(-1))
    kv_lo.copy_(kmin // 128)
    tiles = torch.arange(nq, device=dev)
    reach = (kmin // 128)[:, None, :] <= tiles[None, :, None]                 # [B, kt, qt]
    q_hi.copy_(torch.where(reach, tiles[None, None, :], -1).amax(-1))
