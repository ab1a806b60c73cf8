"""Llama causal LM on the flat arena: hand-scheduled forward/backward over sm_100a kernels.

There is no autograd graph on the hot path.  ``LlamaEngine`` runs the layer program explicitly
(K1..K8 of SURVEY.md §2.5), keeps activations in shape-keyed static workspaces (CUDA-graph friendly) and
accumulates weight gradients straight into the fp32 gradient arena.  ``LlamaForCausalLM`` is the user-facing
``nn.Module``: HF-compatible parameter names / state dict / ``forward(input_ids, labels) -> .loss`` whose
``.backward()`` triggers the engine's backward through a single autograd node, so reference-style training loops
(train_fsdp.py:378-383, train_diloco_torch.py:312-318) run unchanged.

Op semantics follow the installed HF implementation the reference delegates to (SURVEY.md E1):
RMSNorm modeling_llama.py:62-67, RoPE :117-168, attention :251-289, MLP :182-184, decoder layer :303-332,
LM head + shifted CE :484-491 / loss_utils.py:45-67.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from pathlib import Path
from typing import Any

import torch
from torch import nn

from .. import _lib
from ..ops import attention as A
from ..ops import gemm as G
from ..ops import kernels as K
from ..ops import tc_gemm as TC
from .arena import ParamArena, hf_param_order
from .config import LlamaConfig

IGNORE_INDEX = -100


def _use_graph() -> bool:
    """CUDA-graph replay of the micro-step (default on; ODB_CUDA_GRAPH=0 for the eager launch sequence).  Measured on B200,
    Llama-150M: GPU busy 98.4 % -> 99.7 % of the step window (4052 inter-kernel gaps of ~2.2 us -> 193), +1.0 % tokens/s
    (profiles/r2_idle_gap.txt)."""
    return os.environ.get("ODB_CUDA_GRAPH", "1") == "1"



@dataclass
class CausalLMOutput:
    loss: torch.Tensor | None = None
    logits: torch.Tensor | None = None

    def __getitem__(self, k):
        return getattr(self, k) if isinstance(k, str) else (self.loss, self.logits)[k]


# ======================================================================================================= engine
class _Workspace:
    """Static activation buffers for one (B, S) shape."""

    def __init__(self, cfg: LlamaConfig, B: int, S: int, device, dtype, lce_chunk: int):
        T, h, i, L = B * S, cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
        e = lambda *shape, dt=dtype: torch.empty(*shape, dtype=dt, device=device)  # noqa: E731
        f32 = torch.float32
        self.B, self.S, self.T = B, S, T
        self.ids = torch.empty(T, dtype=torch.int64, device=device)
        self.labels = torch.empty(T, dtype=torch.int64, device=device)      # HF-shifted labels
        self.labels_in = torch.empty(T, dtype=torch.int64, device=device)   # staging for host / strided label tensors
        # saved per layer
        self.xa = [e(T, h) for _ in range(L)]         # residual stream entering the attention block
        self.rstd1 = [e(T, dt=f32) for _ in range(L)]
        self.xn1 = [e(T, h) for _ in range(L)]
        self.qkv = [e(T, cfg.qkv_dim) for _ in range(L)]
        self.att = [None] * L                          # attention output (+aux) allocated by the attention op
        self.aux = [None] * L
        self.xm = [e(T, h) for _ in range(L)]         # residual stream entering the MLP block
        self.rstd2 = [e(T, dt=f32) for _ in range(L)]
        self.xn2 = [e(T, h) for _ in range(L)]
        self.gu = [e(T, 2 * i) for _ in range(L)]
        self.act = [e(T, i) for _ in range(L)]
        self.xf = e(T, h)                              # residual stream entering the final norm
        self.rstdf = e(T, dt=f32)
        self.xnf = e(T, h)
        # transient
        self.proj = e(T, h)                            # o-proj / down-proj output (the residual delta)
        self.dx = e(T, h)                              # gradient of the residual stream
        self.dn = e(T, h)                              # gradient w.r.t. a normed activation
        self.datt = e(T, h)
        self.dqkv = e(T, cfg.qkv_dim)
        self.dact = e(T, i)
        self.dxnf = e(T, h)
        self.lce_rows = min(lce_chunk, T)
        self._dev, self._dt, self._V = device, dtype, cfg.vocab_size
        self._logits = None          # reference path only (CPU / fp32 / fp16): bf16 kernels never materialise logits
        self._lce = None             # fused LCE buffers, allocated on first use
        self._mask = None            # padding mask (int32 [B, S]) + its attention description, allocated on first use
        self.loss_sum = torch.zeros(1, dtype=f32, device=device)
        self.gscale = torch.ones(1, dtype=f32, device=device)
        self.n_valid = torch.ones(1, dtype=f32, device=device)
        self.sumsq = torch.zeros(1, dtype=f32, device=device)
        self.cos, self.sin = K.rope_tables(S, cfg.head_dim, cfg.rope_theta, device)

    @property
    def logits(self) -> torch.Tensor:
        if self._logits is None:
            self._logits = torch.empty(self.lce_rows, self._V, dtype=self._dt, device=self._dev)
        return self._logits

    def mask_buffers(self) -> tuple[torch.Tensor, A.MaskDesc]:
        """(static device copy of the padding mask, attention mask description) of this shape."""
        if self._mask is None:
            self._mask = (torch.empty(self.B, self.S, dtype=torch.int32, device=self._dev), A.MaskDesc.empty(self.B, self.S, self._dev))
        return self._mask

    def lce_buffers(self, planes: int, h: int):
        """(shift [T], rowscale [T], partials [2*planes, C], e [C, V] bf16, xs [C, h] bf16) of the fused LCE."""
        if self._lce is None:
            C, f32 = self.lce_rows, torch.float32
            mk = lambda *shape, dt: torch.empty(*shape, dtype=dt, device=self._dev)  # noqa: E731
            self._lce = (mk(self.T, dt=f32), mk(self.T, dt=f32), mk(2 * planes * C, dt=f32), mk(C, self._V, dt=self._dt),
                         mk(C, h, dt=self._dt))
        return self._lce


class LlamaEngine:
    def __init__(self, cfg: LlamaConfig, arena: ParamArena, lce_chunk: int = 32768):
        self.cfg, self.arena = cfg, arena
        # rows of the logits tile of the chunked linear-cross-entropy (ODB_LCE_CHUNK overrides: larger = fewer, fuller GEMM
        # launches and less reduce-add traffic into the lm_head gradient, at 64 KB of bf16 logits per row)
        self.lce_chunk = int(os.environ.get("ODB_LCE_CHUNK", lce_chunk))
        self._ws: dict[tuple, _Workspace] = {}
        self.collect_act_norms = False
        self.act_norms: dict[str, torch.Tensor] = {}
        self.module_hooks: dict[str, Any] = {}     # name -> holder module with user forward hooks
        self.head_grad_tmp: torch.Tensor | None = None
        self._graphs: dict[tuple, dict] = {}       # (B, S, loss_scale, labels-alias) -> captured micro-step

    def workspace(self, B: int, S: int) -> _Workspace:
        key = (B, S, str(self.arena.device), self.arena.compute_dtype)
        ws = self._ws.get(key)
        if ws is None:
            if len(self._ws) >= 2:       # keep at most two shapes resident (train + eval)
                old = next(iter(self._ws))
                self._ws.pop(old)
                for gk in [k for k in self._graphs if k[:2] == old[:2]]:      # graphs captured on the evicted buffers
                    del self._graphs[gk]
            ws = _Workspace(self.cfg, B, S, self.arena.device, self.arena.compute_dtype, self.lce_chunk)
            self._ws[key] = ws
        return ws

    # --------------------------------------------------------------------------------------------- forward
    def _fire_hooks(self, name: str, out: torch.Tensor) -> None:
        mod = self.module_hooks.get(name)
        if mod is not None and mod._forward_hooks:
            for hook in list(mod._forward_hooks.values()):
                hook(mod, (), out)

    def describe_mask(self, ws: _Workspace, ids: torch.Tensor, attention_mask: torch.Tensor | None,
                      document_mask: bool = False) -> A.MaskDesc | None:
        """Attention mask description of one micro-batch in the workspace's static buffers (None: plain causal).
        ``attention_mask`` [B, S] as returned by ``_normalize_mask``; ``document_mask`` also keeps every query inside its
        document (documents end with ``config.eos_token_id``)."""
        if attention_mask is None and not document_mask:
            return None
        if attention_mask is not None and tuple(attention_mask.shape) != (ws.B, ws.S):
            raise ValueError(f"attention_mask has shape {tuple(attention_mask.shape)}, expected {(ws.B, ws.S)}")
        eos = -1
        if document_mask:
            if self.cfg.eos_token_id is None or self.cfg.eos_token_id < 0:
                raise ValueError("document_mask needs config.eos_token_id")
            eos = int(self.cfg.eos_token_id)
        ws.ids.copy_(ids.reshape(-1), non_blocking=True)
        mbuf, desc = ws.mask_buffers()
        if attention_mask is not None:
            mbuf.copy_(attention_mask, non_blocking=True)
        return desc.build(ws.ids.view(ws.B, ws.S), mbuf if attention_mask is not None else None, eos)

    def forward_hidden(self, ws: _Workspace, ids: torch.Tensor, mask: A.MaskDesc | None = None) -> torch.Tensor:
        cfg, ar = self.cfg, self.arena
        B, S, L = ws.B, ws.S, cfg.num_hidden_layers
        Hq, Hkv, D = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim
        ws.ids.copy_(ids.reshape(-1), non_blocking=True)
        K.embedding_fwd(ws.ids, ar.w("model.embed_tokens.weight"), out=ws.xa[0])
        delta = None
        for l in range(L):
            p = f"model.layers.{l}."
            x_prev = ws.xa[l] if l == 0 else ws.xm[l - 1]
            # --- attention block:  xa = x_prev + delta ; xn1 = norm(xa)
            K.rmsnorm_fwd(x_prev, ar.w(p + "input_layernorm.weight"), cfg.rms_norm_eps, delta=delta, out=ws.xn1[l],
                          rstd=ws.rstd1[l], x_out=ws.xa[l])
            if D == 64 and TC.usable(ws.xn1[l], ar.qkv_w(l)):
                # tcgen05 GEMM with the rotary embedding applied in the epilogue (no separate RoPE pass over q|k)
                TC.linear_qkv_rope(ws.xn1[l], ar.qkv_w(l), ws.qkv[l], ws.cos, ws.sin, S, (Hq + Hkv) * D)
            else:
                G.mm_nt(ws.xn1[l], ar.qkv_w(l), out=ws.qkv[l])
                K.rope_(ws.qkv[l], ws.cos, ws.sin, S, Hq + Hkv, D)
            ws.att[l], ws.aux[l] = A.attention_fwd(ws.qkv[l], B, S, Hq, Hkv, D, mask=mask)
            G.mm_nt(ws.att[l], ar.w(p + "self_attn.o_proj.weight"), out=ws.proj)
            if self.collect_act_norms:
                self.act_norms[f"activation/{p}self_attn"] = ws.proj.float().norm(p=2)
            self._fire_hooks(p + "self_attn", ws.proj)
            # --- MLP block:  xm = xa + proj ; xn2 = norm(xm)
            K.rmsnorm_fwd(ws.xa[l], ar.w(p + "post_attention_layernorm.weight"), cfg.rms_norm_eps, delta=ws.proj,
                          out=ws.xn2[l], rstd=ws.rstd2[l], x_out=ws.xm[l])
            if cfg.intermediate_size % 64 == 0 and TC.usable(ws.xn2[l], ar.gu_w(l)):
                TC.linear_swiglu(ws.xn2[l], ar.gu_w(l), ws.gu[l], ws.act[l])     # SwiGLU is the GEMM epilogue
            else:
                G.mm_nt(ws.xn2[l], ar.gu_w(l), out=ws.gu[l])
                K.swiglu_fwd(ws.gu[l], out=ws.act[l])
            G.mm_nt(ws.act[l], ar.w(p + "mlp.down_proj.weight"), out=ws.proj)
            delta = ws.proj
        K.rmsnorm_fwd(ws.xm[L - 1], ar.w("model.norm.weight"), cfg.rms_norm_eps, delta=delta, out=ws.xnf, rstd=ws.rstdf,
                      x_out=ws.xf)
        return ws.xnf

    # --------------------------------------------------------------------------------------------- LM head + loss
    def head_loss(self, ws: _Workspace, labels: torch.Tensor | None, loss_scale: float, with_grad: bool,
                  direct: bool) -> torch.Tensor:
        """Linear-cross-entropy of the LM head.  Returns the mean loss (0-dim fp32 tensor on device).

        with_grad: also produce d(xnf) in ws.dxnf and the lm_head weight gradient, scaled by loss_scale / n_valid.
        direct: accumulate the lm_head gradient into the arena now (scale known); otherwise into ``head_grad_tmp`` so
        that autograd can apply the upstream gradient later.

        CUDA bf16: the fused path (``_head_loss_fused``) - logits never exist.  Other dtypes / CPU: the reference path
        that materialises a logits tile per chunk (same math, PyTorch ops).
        Reference call site: train_diloco_torch.py:313-314 / train_fsdp.py:378-379 -> loss_utils.py:45-67.
        """
        cfg, ar = self.cfg, self.arena
        V = cfg.vocab_size
        # HF shift: position s predicts token s+1 ; last position of every sequence is ignored
        src = labels.reshape(-1)
        if src.device != ws.labels.device or src.dtype != torch.int64 or not src.is_contiguous():
            ws.labels_in.copy_(src, non_blocking=True)
            src = ws.labels_in
        K.lce_prep(src, ws.labels, ws.B, ws.S, loss_scale, ws.n_valid, ws.gscale, ws.loss_sum)
        w_lm = ar.w("lm_head.weight")
        hooked = self.module_hooks.get("lm_head")
        want_norm = self.collect_act_norms or (hooked is not None and bool(hooked._forward_hooks))
        if want_norm:
            ws.sumsq.zero_()
        g_lm = None
        if with_grad:
            if direct:
                g_lm = ar.g("lm_head.weight")
            else:
                if self.head_grad_tmp is None:
                    self.head_grad_tmp = torch.zeros(V, cfg.hidden_size, dtype=torch.float32, device=ar.device)
                else:
                    self.head_grad_tmp.zero_()
                g_lm = self.head_grad_tmp
        if TC.lce_usable(ws.xnf, w_lm) and os.environ.get("ODB_LCE_FUSED", "1") != "0":
            self._head_loss_fused(ws, w_lm, g_lm, want_norm)
        else:
            self._head_loss_reference(ws, w_lm, g_lm, want_norm)
        if want_norm:
            nrm = ws.sumsq.sqrt()[0]
            if self.collect_act_norms:
                self.act_norms["activation/lm_head"] = nrm
            if hooked is not None and hooked._forward_hooks:
                self._fire_hooks("lm_head", _NormOnly(nrm))
        return (ws.loss_sum / ws.n_valid)[0]

    def _head_loss_fused(self, ws: _Workspace, w_lm: torch.Tensor, g_lm: torch.Tensor | None, want_norm: bool) -> None:
        """Fused linear-cross-entropy on tcgen05 (SURVEY K7).  Per chunk of rows:

          c_t   = x_t . W[y_t]                               (lce_label_dot: the label logit, 2 x T x h bytes)
          E     = exp(X W^T - c)   + partial row sums        (ONE GEMM, epilogue in registers; bf16 E only when training)
          S_t, loss_t = log S_t, rowscale_t = gscale / S_t, xs = rowscale * x, dW[y_t] -= gscale x_t     (lce_finalize)
          dX    = rowscale * (E W) - gscale W[y]             (dgrad GEMM, W read MN-major, normaliser + one-hot in the epilogue)
          dW   += E^T xs                                     (weight-gradient GEMM)

        softmax - onehot is never formed and there is no pass over a [T, V] tensor outside the three GEMMs: the shift c is
        known before the GEMM, so the exponentials can be emitted by its epilogue, and the per-row normaliser moves to
        the fp32 side of the two gradient GEMMs.  In evaluation (g_lm is None) nothing of size [T, V] is written at all.
        """
        T, h = ws.T, self.cfg.hidden_size
        V = w_lm.shape[0]
        planes = TC.lce_planes(V)
        shift, rowscale, partials, e_buf, xs_buf = ws.lce_buffers(planes, h)
        train = g_lm is not None
        K.lce_label_dot(ws.xnf, w_lm, ws.labels, shift)
        C = ws.lce_rows
        for c0 in range(0, T, C):
            c1 = min(T, c0 + C)
            n = c1 - c0
            x = ws.xnf[c0:c1]
            e = e_buf[:n] if train else None
            TC.lce_fwd(x, w_lm, shift[c0:c1], partials, e, want_sumsq=want_norm)
            K.lce_finalize(partials, planes, ws.labels[c0:c1], ws.gscale, ws.loss_sum, ws.sumsq if want_norm else None,
                           rowscale[c0:c1] if train else None, x, xs_buf[:n] if train else None, g_lm)
            if train:
                TC.lce_dx(e, w_lm, rowscale[c0:c1], ws.labels[c0:c1], ws.gscale, ws.dxnf[c0:c1])
                G.mm_tn_acc(e, xs_buf[:n], g_lm)

    def _head_loss_reference(self, ws: _Workspace, w_lm: torch.Tensor, g_lm: torch.Tensor | None, want_norm: bool) -> None:
        T = ws.T
        C = ws.lce_rows
        for c0 in range(0, T, C):
            c1 = min(T, c0 + C)
            logits = ws.logits[: c1 - c0]
            G.mm_nt(ws.xnf[c0:c1], w_lm, out=logits)
            if g_lm is not None:
                K.ce_fwd_bwd_(logits, ws.labels[c0:c1], ws.gscale, ws.loss_sum, ws.sumsq if want_norm else None)
                G.mm_nn(logits, w_lm, out=ws.dxnf[c0:c1])
                G.mm_tn_acc(logits, ws.xnf[c0:c1], g_lm)
            else:
                if want_norm:
                    ws.sumsq.add_(logits.float().pow(2).sum())
                K.ce_fwd(logits, ws.labels[c0:c1], ws.loss_sum)

    def logits(self, ws: _Workspace) -> torch.Tensor:
        """Materialise full logits [T, V] (inference / debugging only)."""
        return G.mm_nt(ws.xnf, self.arena.w("lm_head.weight"))

    # --------------------------------------------------------------------------------------------- backward
    def backward(self, ws: _Workspace, mask: A.MaskDesc | None = None) -> None:
        """Back-propagate ws.dxnf (gradient w.r.t. the final-norm output) through the stack, accumulating into arena.grad."""
        cfg, ar = self.cfg, self.arena
        B, S, L = ws.B, ws.S, cfg.num_hidden_layers
        Hq, Hkv, D = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim
        K.rmsnorm_bwd(ws.dxnf, ws.xf, ar.w("model.norm.weight"), ws.rstdf, None, ws.dx, ar.g("model.norm.weight"))
        for l in reversed(range(L)):
            p = f"model.layers.{l}."
            # ---- MLP block (ws.dx is the gradient of x_out = xm + down(act))
            G.mm_tn_acc(ws.dx, ws.act[l], ar.g(p + "mlp.down_proj.weight"))
            w_down = ar.w(p + "mlp.down_proj.weight")
            if TC.swiglu_bwd_usable(ws.dx, w_down, ws.gu[l]):
                TC.linear_swiglu_bwd(ws.dx, w_down, ws.gu[l])              # dgrad GEMM with the SwiGLU backward as epilogue
            else:
                G.mm_nn(ws.dx, w_down, out=ws.dact)
                K.swiglu_bwd(ws.dact, ws.gu[l], ws.gu[l])                  # in place: gu <- d(gu)
            G.mm_tn_acc(ws.gu[l], ws.xn2[l], ar.gu_g(l))
            G.mm_nn(ws.gu[l], ar.gu_w(l), out=ws.dn)
            K.rmsnorm_bwd(ws.dn, ws.xm[l], ar.w(p + "post_attention_layernorm.weight"), ws.rstd2[l], ws.dx, ws.dx,
                          ar.g(p + "post_attention_layernorm.weight"))
            # ---- attention block (ws.dx is now the gradient of xm = xa + o(att))
            G.mm_tn_acc(ws.dx, ws.att[l], ar.g(p + "self_attn.o_proj.weight"))
            G.mm_nn(ws.dx, ar.w(p + "self_attn.o_proj.weight"), out=ws.datt)
            parts_ok = cfg.q_dim % 64 == 0 and cfg.kv_dim % 64 == 0 and TC.nn_usable(ws.datt, ar.qkv_w(l))
            res = A.attention_bwd(ws.datt, ws.qkv[l], ws.att[l], ws.aux[l], ws.dqkv, B, S, Hq, Hkv, D, want_parts=parts_ok,
                                  rope=(ws.cos, ws.sin), mask=mask)
            if isinstance(res, tuple):
                # un-packed gradients (cuDNN): rotate dq/dk in place, three wgrads into the row blocks of the fused
                # QKV gradient, and ONE dgrad GEMM whose A operand is read from the three tensors
                dq, dk, dv = res
                K.rope_(dq, ws.cos, ws.sin, S, Hq, D, backward=True)
                K.rope_(dk, ws.cos, ws.sin, S, Hkv, D, backward=True)
                gq = ar.qkv_g(l)
                if cfg.q_dim % 256 == 0 and cfg.kv_dim % 256 == 0 and TC.wgrad_usable(dq, dk, dv, ws.xn1[l]):
                    TC.wgrad_acc((dq, dk, dv), ws.xn1[l], gq)          # one launch, A read from the three tensors
                else:
                    G.mm_tn_acc(dq, ws.xn1[l], gq[: cfg.q_dim])
                    G.mm_tn_acc(dk, ws.xn1[l], gq[cfg.q_dim: cfg.q_dim + cfg.kv_dim])
                    G.mm_tn_acc(dv, ws.xn1[l], gq[cfg.q_dim + cfg.kv_dim:])
                TC.linear_nn_a3(dq, dk, dv, ar.qkv_w(l), ws.dn)
            else:
                if not A.bwd_applies_rope(ws.aux[l]):
                    K.rope_(ws.dqkv, ws.cos, ws.sin, S, Hq + Hkv, D, backward=True)
                G.mm_tn_acc(ws.dqkv, ws.xn1[l], ar.qkv_g(l))
                G.mm_nn(ws.dqkv, ar.qkv_w(l), out=ws.dn)
            K.rmsnorm_bwd(ws.dn, ws.xa[l], ar.w(p + "input_layernorm.weight"), ws.rstd1[l], ws.dx, ws.dx,
                          ar.g(p + "input_layernorm.weight"))
            ws.att[l] = None
            ws.aux[l] = None
        K.embedding_bwd(ws.ids, ws.dx, ar.g("model.embed_tokens.weight"))

    # --------------------------------------------------------------------------------------------- fused entry
    def forward_backward(self, ids: torch.Tensor, labels: torch.Tensor, loss_scale: float = 1.0,
                         attention_mask: torch.Tensor | None = None, document_mask: bool = False) -> torch.Tensor:
        """One micro-batch: forward, loss, backward; gradients (scaled by loss_scale) are ADDED to arena.grad.
        Returns the mean token loss as a device scalar (no host sync).  ``attention_mask``: None or a [B, S] mask that is
        not all ones (``_normalize_mask``; no host sync here, so the call can be captured into a CUDA graph)."""
        B, S = ids.shape
        ws = self.workspace(B, S)
        ar = self.arena
        with torch.no_grad():
            mask = self.describe_mask(ws, ids, attention_mask, document_mask)
            ar.materialize_shadow()            # FULL_SHARD: all-gather the compute weights (no-op otherwise)
            self.forward_hidden(ws, ids, mask)
            loss = self.head_loss(ws, labels, loss_scale, with_grad=True, direct=True)
            if ar.param_sharded:               # reshard after forward, gather again for backward (FSDP FULL_SHARD)
                ar.release_shadow()
                ar.materialize_shadow()
            self.backward(ws, mask)
            ar.release_shadow()
        return loss


    # --------------------------------------------------------------------------------------------- CUDA-graph replay
    def forward_backward_graphed(self, ids: torch.Tensor, labels: torch.Tensor, loss_scale: float,
                                 attention_mask: torch.Tensor | None = None, document_mask: bool = False) -> torch.Tensor:
        """``forward_backward`` with the ~250 launches of a micro-batch captured ONCE per (B, S, loss_scale, masked,
        document_mask) into a CUDA graph and replayed afterwards (every buffer of the micro-step is static: workspace,
        arena, TMA descriptors are baked kernel parameters).  Inputs (ids, labels, the padding mask) are copied into the
        graph's static buffers and the mask description is computed inside the graph; the returned loss is the graph's
        static output (consume it before the next replay).  ``attention_mask`` must be normalised (``_normalize_mask``).
        Falls back to the eager path while hooks / activation-norm collection are active (they run Python between
        kernels)."""
        B, S = ids.shape
        hooked = any(m._forward_hooks for m in self.module_hooks.values())
        if self.collect_act_norms or hooked or not ids.is_cuda:
            return self.forward_backward(ids, labels, loss_scale, attention_mask, document_mask)
        masked = attention_mask is not None
        key = (B, S, float(loss_scale), labels is ids, masked, bool(document_mask))
        st = self._graphs.get(key)
        if st is not None and st.get("version") != self.arena.version:
            st = None                     # an arena buffer was re-homed (symmetric-memory windows): captured pointers are stale
        if st is None:
            st = {"calls": 0, "graph": None, "version": self.arena.version}
            self._graphs[key] = st
        if st["graph"] is None:
            st["calls"] += 1
            if st["calls"] <= 2:          # warm-up: allocations, cudaFuncSetAttribute, library handles
                return self.forward_backward(ids, labels, loss_scale, attention_mask, document_mask)
            g_ids = torch.empty_like(ids)
            g_lab = g_ids if labels is ids else torch.empty_like(labels)
            g_mask = torch.empty(B, S, dtype=torch.int32, device=ids.device) if masked else None
            g_ids.copy_(ids)
            if g_lab is not g_ids:
                g_lab.copy_(labels)
            if masked:
                g_mask.copy_(attention_mask)
            ws = self.workspace(B, S)
            for l in range(self.cfg.num_hidden_layers):
                ws.att[l] = ws.aux[l] = None
            torch.cuda.synchronize(ids.device)
            graph = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            # thread_local: the NCCL watchdog / data-loader threads keep making CUDA calls of their own during the capture
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                loss = self.forward_backward(g_ids, g_lab, loss_scale, g_mask, document_mask)
            # kernels of ours recorded in the graph: every replay launches them again (bench.py's gpu_launches book-keeping)
            st.update(graph=graph, ids=g_ids, labels=g_lab, mask=g_mask, loss=loss, kernels=_lib.launch_count() - n0)
            graph.replay()
            return st["loss"]
        st["ids"].copy_(ids, non_blocking=True)
        if st["labels"] is not st["ids"]:
            st["labels"].copy_(labels, non_blocking=True)
        if masked:
            st["mask"].copy_(attention_mask, non_blocking=True)
        st["graph"].replay()
        _lib.count_launch(st["kernels"])
        return st["loss"]


class _NormOnly:
    """Stand-in handed to lm_head forward hooks: the logits are never materialised, only their L2 norm exists."""

    def __init__(self, nrm: torch.Tensor):
        self._nrm = nrm

    def norm(self, p=2):
        return self._nrm


def _normalize_mask(attention_mask: torch.Tensor | None) -> torch.Tensor | None:
    """None when the mask is absent or all ones (pure causal fast path); otherwise the [B, S] mask as bool."""
    if attention_mask is None:
        return None
    if attention_mask.dim() != 2:
        raise ValueError(f"attention_mask must be 2-D [batch, seq], got shape {tuple(attention_mask.shape)}")
    if bool(attention_mask.all()):
        return None
    return attention_mask.bool()


# ======================================================================================================= nn.Module facade
class _Holder(nn.Module):
    """Parameter holder: the math runs in LlamaEngine, this only gives the weight its HF name."""

    def __init__(self, weight: nn.Parameter | None = None):
        super().__init__()
        if weight is not None:
            self.weight = weight

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("sub-modules of opendiloco_b200.LlamaForCausalLM are parameter holders; call the top-level model")


class _EngineLoss(torch.autograd.Function):
    """Single autograd node bridging loss.backward() to the engine's hand-written backward."""

    @staticmethod
    def forward(ctx, anchor: torch.Tensor, model: "LlamaForCausalLM", ids, labels, mask, document_mask):
        eng = model.engine
        B, S = ids.shape
        ws = eng.workspace(B, S)
        mask = eng.describe_mask(ws, ids, mask, document_mask)
        eng.arena.materialize_shadow()
        eng.forward_hidden(ws, ids, mask)
        loss = eng.head_loss(ws, labels, 1.0, with_grad=True, direct=False)
        eng.arena.release_shadow()
        ctx.model, ctx.ws, ctx.mask = model, ws, mask
        return loss.clone()

    @staticmethod
    def backward(ctx, g):
        eng, ws = ctx.model.engine, ctx.ws
        with torch.no_grad():
            g32 = g.to(torch.float32)
            ws.dxnf.mul_(g32.to(ws.dxnf.dtype))
            eng.arena.g("lm_head.weight").addcmul_(eng.head_grad_tmp, g32.expand_as(eng.head_grad_tmp))
            eng.arena.materialize_shadow()
            eng.backward(ws, ctx.mask)
            eng.arena.release_shadow()
        return None, None, None, None, None, None


class LlamaForCausalLM(nn.Module):
    """Drop-in for the HF class the reference trains (train_fsdp.py:171-174, train_diloco_torch.py:183)."""

    def __init__(self, config: LlamaConfig, device=None, precision: str = "bf16-mixed", seed: int | None = None,
                 init: bool = True, lce_chunk: int = 32768):
        super().__init__()
        self.config = config
        self.precision = precision
        compute = {"bf16-mixed": torch.bfloat16, "fp16-mixed": torch.float16, "32-true": torch.float32}[precision]
        device = torch.device(device if device is not None else "cpu")
        self.arena = ParamArena(config, device, compute)
        self.engine = LlamaEngine(config, self.arena, lce_chunk=lce_chunk)
        self._build_tree()
        if init:
            self.arena.init_weights(seed)

    # ------------------------------------------------------------------ module tree with HF names
    def _build_tree(self) -> None:
        cfg, ar = self.config, self.arena

        def P(name: str) -> nn.Parameter:
            prm = nn.Parameter(ar.p(name), requires_grad=True)
            prm.grad = ar.g(name)
            prm._odb_name = name
            prm._odb_arena = ar
            return prm

        self.model = _Holder()
        self.model.embed_tokens = _Holder(P("model.embed_tokens.weight"))
        layers = []
        for l in range(cfg.num_hidden_layers):
            p = f"model.layers.{l}."
            layer = _Holder()
            layer.self_attn = _Holder()
            for n in ("q_proj", "k_proj", "v_proj", "o_proj"):
                setattr(layer.self_attn, n, _Holder(P(p + f"self_attn.{n}.weight")))
            layer.mlp = _Holder()
            for n in ("gate_proj", "up_proj", "down_proj"):
                setattr(layer.mlp, n, _Holder(P(p + f"mlp.{n}.weight")))
            layer.input_layernorm = _Holder(P(p + "input_layernorm.weight"))
            layer.post_attention_layernorm = _Holder(P(p + "post_attention_layernorm.weight"))
            layers.append(layer)
            self.engine.module_hooks[p + "self_attn"] = layer.self_attn
        self.model.layers = nn.ModuleList(layers)
        self.model.norm = _Holder(P("model.norm.weight"))
        self.lm_head = _Holder(P("lm_head.weight"))
        self.engine.module_hooks["lm_head"] = self.lm_head

    def _rebind(self) -> None:
        for _, prm in self.named_parameters():
            prm.data = self.arena.p(prm._odb_name)
            prm.grad = self.arena.g(prm._odb_name)

    # ------------------------------------------------------------------ device / dtype management
    def to(self, *args, **kwargs):
        device = kwargs.get("device")
        for a in args:
            if isinstance(a, (str, torch.device, int)):
                device = a
            elif isinstance(a, torch.dtype):
                raise TypeError("opendiloco_b200 models keep fp32 master weights; choose `precision=` at construction")
        if device is not None:
            device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
            if device.type == "cuda" and device.index is None:
                device = torch.device("cuda", torch.cuda.current_device())
            if device != self.arena.device:
                self.arena.migrate(device)
                self.engine._ws.clear()
                self.engine._graphs.clear()
                self.engine.head_grad_tmp = None
                self._rebind()
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", device if device is not None else torch.cuda.current_device()))

    def cpu(self):
        return self.to("cpu")

    @property
    def device(self) -> torch.device:
        return self.arena.device

    # ------------------------------------------------------------------ forward
    def forward(self, input_ids: torch.Tensor, attention_mask: torch.Tensor | None = None,
                labels: torch.Tensor | None = None, return_logits: bool = False, document_mask: bool = False,
                **_unused) -> CausalLMOutput:
        """``attention_mask`` [B, S]: 0 marks padding keys.  ``document_mask``: attention also stays inside the documents of
        a packed row, each ending with ``config.eos_token_id`` (labels are not changed)."""
        eng = self.engine
        if input_ids.device != self.arena.device:
            input_ids = input_ids.to(self.arena.device, non_blocking=True)
        if labels is not None and labels.device != self.arena.device:
            labels = labels.to(self.arena.device, non_blocking=True)
        mask = _normalize_mask(attention_mask)
        B, S = input_ids.shape
        if labels is not None and torch.is_grad_enabled() and self.training:
            loss = _EngineLoss.apply(self.lm_head.weight, self, input_ids, labels, mask, document_mask)
            return CausalLMOutput(loss=loss)
        with torch.no_grad():
            ws = eng.workspace(B, S)
            desc = eng.describe_mask(ws, input_ids, mask, document_mask)
            self.arena.materialize_shadow()
            eng.forward_hidden(ws, input_ids, desc)
            loss = eng.head_loss(ws, labels, 1.0, with_grad=False, direct=False).clone() if labels is not None else None
            logits = eng.logits(ws).view(B, S, -1) if (return_logits or labels is None) else None
            self.arena.release_shadow()
        return CausalLMOutput(loss=loss, logits=logits)

    def forward_backward(self, input_ids: torch.Tensor, labels: torch.Tensor, loss_scale: float = 1.0,
                         attention_mask: torch.Tensor | None = None, document_mask: bool = False) -> torch.Tensor:
        """Native fast path: one micro-batch forward+backward, grads += loss_scale * dL/dw. Returns the device loss.
        With ODB_CUDA_GRAPH=1 the micro-step is replayed from a CUDA graph (masked or not).  ``attention_mask`` /
        ``document_mask`` as in ``forward``."""
        mask = _normalize_mask(attention_mask)
        if _use_graph() and input_ids.is_cuda and self.arena.compute_dtype == torch.bfloat16 and not self.arena.param_sharded:
            return self.engine.forward_backward_graphed(input_ids, labels, loss_scale, mask, document_mask)
        return self.engine.forward_backward(input_ids, labels, loss_scale, mask, document_mask)

    # ------------------------------------------------------------------ state dict / checkpoints
    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        res = super().load_state_dict(state_dict, strict=strict, assign=False)
        self.arena.sync_shadow()
        return res

    def sync_compute_weights(self) -> None:
        """Call after writing to parameters outside the fused optimizers (torch optimizers, manual edits)."""
        self.arena.sync_shadow()

    @classmethod
    def from_config(cls, config: LlamaConfig, **kw) -> "LlamaForCausalLM":
        return cls(config, **kw)

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path: str, config: LlamaConfig | None = None, device=None,
                        precision: str = "bf16-mixed", seed: int | None = 0, **_unused) -> "LlamaForCausalLM":
        """Load config (+ ``model.safetensors`` if present).  A bare config / preset name yields seeded random init —
        the offline equivalent of the reference's ``*-fresh`` hub checkpoints (init_weights.py:10-25)."""
        from ..utils.safetensors_io import load_safetensors

        cfg = config if isinstance(config, LlamaConfig) else LlamaConfig.from_pretrained(pretrained_model_name_or_path)
        path = Path(pretrained_model_name_or_path)
        st = path / "model.safetensors" if path.is_dir() else None
        model = cls(cfg, device=device, precision=precision, seed=seed, init=not (st and st.is_file()))
        if st is not None and st.is_file():
            tensors = load_safetensors(str(st))
            with torch.no_grad():
                for name in hf_param_order(cfg):
                    model.arena.p(name).copy_(tensors[name].to(torch.float32))
            model.arena.sync_shadow()
        return model

    def save_pretrained(self, directory: str) -> None:
        from ..utils.safetensors_io import save_safetensors

        os.makedirs(directory, exist_ok=True)
        self.config.save_pretrained(directory)
        save_safetensors({n: self.arena.p(n).detach().cpu().contiguous() for n in hf_param_order(self.config)},
                         os.path.join(directory, "model.safetensors"), metadata={"format": "pt"})

    def num_parameters(self) -> int:
        return self.config.num_parameters()

    @torch.no_grad()
    def clip_grad_norm_(self, max_norm: float, norm_type: float = 2.0) -> torch.Tensor:
        """FSDP-style method the reference calls (train_fsdp.py:395).  If a FusedAdamW owns the arena the scaling is
        folded into its next step (one reduction pass, zero extra sweeps); otherwise grads are scaled here."""
        assert norm_type == 2.0
        ref = getattr(self.arena, "fused_optimizer", None)
        opt = ref() if ref is not None else None
        if opt is not None:
            return opt.compute_grad_norm_partials(max_norm)
        total = self.arena.grad.norm(2)
        coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
        self.arena.grad.mul_(coef)
        return total
