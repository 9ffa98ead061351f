"""LinearWeights - the query-conditioned field mixture (mfar/modeling/weighting.py:3-29).

Same constructor, parameter name/shape and forward signature as the reference module:
  ``LinearWeights(emb_size, num_fields, query_cond)``, ``.weight`` [emb_size, num_fields]
  (init ones, weighting.py:14), ``forward(x[B,S,F] or [S,F], q[B,E] or None) -> [B,S]``.
When ``query_cond`` is False the reference constructs it as ``LinearWeights(num_fields, 1)``
(contrastive.py:285), i.e. weight is [F,1] and the softmax runs over its transpose.

``forward`` runs the CUDA kernels behind ``mfar_mixture_weights`` / ``mfar_mixture_apply`` (fp32).  When autograd
is recording and any of x / q / weight requires grad, it goes through ``MixtureFunction`` whose backward is
``mfar_mixture_bwd`` (dx, dW, dq) - the training-time use inside the contrastive losses (losses.py:197-202); an [S,F]
x is expanded to [B,S,F] first, so it stays differentiable as in the reference.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import _native as nv


class MixtureFunction(torch.autograd.Function):
    """out[b,s] = sum_f softmax(q @ W)[b,f] * x[b,s,f]  (weighting.py:24-29) with a CUDA backward."""

    @staticmethod
    def forward(ctx, x3: torch.Tensor, q: Optional[torch.Tensor], W: torch.Tensor, query_cond: bool):
        B, S, F = x3.shape
        Wc = W.detach().contiguous().float()
        if query_cond:
            qe = q.detach().contiguous().float()
            E = qe.shape[1]
            w = torch.empty((B, F), dtype=torch.float32, device=x3.device)
            nv.check(nv.lib().mfar_mixture_weights(nv.ptr(qe), nv.ptr(Wc), 0, B, E, F, 1, nv.ptr(w), nv.stream()),
                     "mixture_weights")
        else:
            qe, E = None, 0
            w = torch.empty((1, F), dtype=torch.float32, device=x3.device)
            nv.check(nv.lib().mfar_mixture_weights(0, nv.ptr(Wc), 0, 1, 0, F, 0, nv.ptr(w), nv.stream()),
                     "mixture_weights")
        xc = x3.detach().contiguous().float()
        out = torch.empty((B, S), dtype=torch.float32, device=x3.device)
        nv.check(nv.lib().mfar_mixture_apply(nv.ptr(xc), nv.ptr(w), B, S, F, w.shape[0], nv.ptr(out), nv.stream()),
                 "mixture_apply")
        ctx.save_for_backward(xc, qe if qe is not None else torch.empty(0, device=x3.device), Wc, w)
        ctx.query_cond, ctx.E = query_cond, E
        return out

    @staticmethod
    def backward(ctx, g: torch.Tensor):
        xc, qe, Wc, w = ctx.saved_tensors
        B, S, F = xc.shape
        g = g.contiguous().float()
        need_x, need_q, _, _ = ctx.needs_input_grad
        dx = torch.empty_like(xc) if need_x else None
        dW = torch.empty_like(Wc)
        dq = torch.empty_like(qe) if (ctx.query_cond and need_q) else None
        scratch = torch.empty((B, F), dtype=torch.float32, device=xc.device)
        nv.check(nv.lib().mfar_mixture_bwd(nv.ptr(xc), nv.ptr(qe) if ctx.query_cond else 0, nv.ptr(Wc), nv.ptr(w),
                                           w.shape[0], nv.ptr(g), B, S, ctx.E, F, int(ctx.query_cond), nv.ptr(dx),
                                           nv.ptr(dW), nv.ptr(dq), nv.ptr(scratch), nv.stream()), "mixture_bwd")
        return dx, dq, dW, None


class LinearWeights(torch.nn.Module):

    def __init__(self, emb_size: int, num_fields: int, query_cond: bool = False):
        super().__init__()
        self.query_cond = query_cond
        self.weight = torch.nn.Parameter(torch.ones(emb_size, num_fields), requires_grad=True)   # weighting.py:14

    @property
    def num_fields(self) -> int:
        return self.weight.shape[1] if self.query_cond else self.weight.shape[0]

    @torch.no_grad()
    def field_weights(self, q: Optional[torch.Tensor], mask: Optional[torch.Tensor] = None,
                      batch: Optional[int] = None) -> torch.Tensor:
        """softmax field weights [Q,F] (times the 0/1 field mask, un-renormalised)."""
        W = self.weight.detach()
        nv.require_device(W, "LinearWeights.weight")
        W = W.contiguous().float()
        F = self.num_fields
        if self.query_cond:
            if q is None:
                raise ValueError("query_cond=True needs the query embedding")
            nv.require_device(q, "q")
            qe = q.detach().contiguous().float()
            Q, E = qe.shape
            if E != W.shape[0]:
                raise RuntimeError(f"q is [*,{E}] but weight is [{W.shape[0]},{W.shape[1]}]")
        else:
            qe, Q, E = None, (batch or 1), 0
        m = None
        if mask is not None:
            m = mask.detach().to(device=W.device, dtype=torch.float32).reshape(-1).contiguous()
            if m.numel() != F:
                raise RuntimeError(f"mask has {m.numel()} entries for {F} fields")
        out = torch.empty((Q, F), dtype=torch.float32, device=W.device)
        nv.check(nv.lib().mfar_mixture_weights(nv.ptr(qe), nv.ptr(W), nv.ptr(m), Q, E, F, int(self.query_cond),
                                               nv.ptr(out), nv.stream()), "mixture_weights")
        return out

    def forward(self, x: torch.Tensor, q: Optional[torch.Tensor]) -> torch.Tensor:
        nv.require_device(x, "x")
        if torch.is_grad_enabled() and x.dim() in (2, 3) and (
                x.requires_grad or self.weight.requires_grad or (q is not None and q.requires_grad)):
            nv.require_device(self.weight, "LinearWeights.weight")
            if x.shape[-1] != self.num_fields:
                raise RuntimeError(f"x has {x.shape[-1]} fields, layer has {self.num_fields}")
            if self.query_cond and q is None:
                raise ValueError("query_cond=True needs the query embedding")
            if x.dim() == 2:                         # [S,F] against every query (weighting.py:29); expand's backward
                B = q.shape[0] if self.query_cond else 1     # sums dx over the queries
                x = x.unsqueeze(0).expand(B, *x.shape)
            if self.query_cond and q.shape[0] != x.shape[0]:
                raise RuntimeError("batch size of x and q must match (weighting.py:21-23)")
            return MixtureFunction.apply(x, q if self.query_cond else None, self.weight, self.query_cond)
        with torch.no_grad():
            return self._forward_nograd(x, q)

    def _forward_nograd(self, x: torch.Tensor, q: Optional[torch.Tensor]) -> torch.Tensor:
        squeeze = x.dim() == 2                       # trec_eval_step passes [S,F] (contrastive.py:694)
        x3 = (x.unsqueeze(0) if squeeze else x).contiguous().float()
        B, S, F = x3.shape
        if F != self.num_fields:
            raise RuntimeError(f"x has {F} fields, layer has {self.num_fields}")
        w = self.field_weights(q)                    # [Q,F] or [1,F]
        if squeeze and w.shape[0] > 1:               # [S,F] against B queries broadcasts to [B,S] (weighting.py:29)
            B = w.shape[0]
            x3 = x3.expand(B, S, F).contiguous()
        if w.shape[0] not in (1, B):
            raise RuntimeError("batch size of x and q must match (weighting.py:21-23)")
        out = torch.empty((B, S), dtype=torch.float32, device=x3.device)
        nv.check(nv.lib().mfar_mixture_apply(nv.ptr(x3), nv.ptr(w), B, S, F, w.shape[0], nv.ptr(out), nv.stream()),
                 "mixture_apply")
        return out
