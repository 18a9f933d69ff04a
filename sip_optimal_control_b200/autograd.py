"""``torch.autograd`` bindings of the batched LQR and Newton-KKT solves.

``factor_solve(lqr, inp)`` runs ``LQR.factor_solve`` on the engine-layout tensors of ``inp``
(keys Q, M, R, q, r, A, B, c, delta) and returns ``(x, u, y, status)``; x, u, y carry
gradients back to every input that requires them through ``sipoc_lqr_vjp`` (one more LQR
solve on the same kernels plus the gradient-assembly kernel).  Both directions run on
torch's current stream.

Conventions (include/sipoc.h, sipoc_lqr_vjp):
- The engine reads only the lower triangles of Q and R; their gradient is that of the solve
  as a function of the SYMMETRIC matrices.  Form Q = (P + P^T) / 2 (per block) from a free
  tensor P to get dL/dP right.
- Problems whose factorization fails (status != 0) and the padding lanes
  batch <= b < batch_stride get zero gradients.

``kkt_factor_solve(cp, model, w, r1, r2, r3, b)`` does the same for the Newton-KKT solve
(``CallbackProvider.factor`` + ``solve``) and returns ``(sol, ok)``; sol carries gradients
back to the model blocks (theta blocks included), w, r1, r2, r3 and b through
``sipoc_kkt_vjp`` (one more KKT factor and solve plus the gradient-assembly kernel).  The
symmetric Hessian blocks (node_hxx, edge_hxx, edge_huu, node_htt, edge_htt) get the
symmetric gradient, and problems with ok == 0 and the padding lanes get zeros.
"""
from __future__ import annotations

import torch

from ._capi import KKT_MODEL_FIELDS, KKT_THETA_FIELDS, LQR_INPUT_FIELDS


class _FactorSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lqr, *arrays):
        inp = {k: a.contiguous() for k, a in zip(LQR_INPUT_FIELDS, arrays)}
        out = lqr.alloc_output()
        status = lqr.factor_solve(inp, out)
        ctx.lqr = lqr
        ctx.save_for_backward(*(inp[k] for k in ("Q", "M", "R", "A", "B", "delta")),
                              out["x"], out["u"], out["y"])
        ctx.mark_non_differentiable(status)
        return out["x"], out["u"], out["y"], status

    @staticmethod
    def backward(ctx, gx, gu, gy, _gstatus):
        Q, M, R, A, B, delta, x, u, y = ctx.saved_tensors
        want = {k for k, need in zip(LQR_INPUT_FIELDS, ctx.needs_input_grad[1:]) if need}
        if not want:
            return (None,) * (1 + len(LQR_INPUT_FIELDS))
        # autograd may hand out stride-0 expanded tensors (e.g. from .sum()) or None
        cot = {k: torch.zeros_like(ref) if g is None else g.contiguous()
               for k, g, ref in (("x", gx, x), ("u", gu, u), ("y", gy, y))}
        inp = dict(Q=Q, M=M, R=R, A=A, B=B, delta=delta)
        grads = ctx.lqr.vjp(inp, dict(x=x, u=u, y=y), cot, want=want)
        return (None,) + tuple(grads.get(k) for k in LQR_INPUT_FIELDS)


def factor_solve(lqr, inp: dict):
    """Differentiable ``lqr.factor_solve``: returns (x, u, y, status), status not
    differentiable.  ``inp`` holds float64 CUDA tensors in the engine layout
    ``[size, batch_stride]`` (``LQR.alloc_input`` / ``LQR.pack_input``)."""
    return _FactorSolve.apply(lqr, *(inp[k] for k in LQR_INPUT_FIELDS))


_KKT_VECTORS = ("w", "r1", "r2", "r3", "b")


class _KktFactorSolve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cp, n_model, *arrays):
        fields = (KKT_MODEL_FIELDS + KKT_THETA_FIELDS)[:n_model]
        model = {k: a.contiguous() for k, a in zip(fields, arrays[:n_model])}
        w, r1, r2, r3, b = (a.contiguous() for a in arrays[n_model:])
        ok = cp.factor(model, w, r1, r2, r3)
        sol = cp.engine.zeros(cp.sizes["kkt_dim"])
        cp.solve(model, b, sol)
        ctx.cp, ctx.fields = cp, fields
        ctx.save_for_backward(*model.values(), w, r1, r2, r3, sol)
        ctx.mark_non_differentiable(ok)
        return sol, ok

    @staticmethod
    def backward(ctx, gsol, _gok):
        saved = ctx.saved_tensors
        n = len(ctx.fields)
        names = ctx.fields + _KKT_VECTORS
        want = {k for k, need in zip(names, ctx.needs_input_grad[2:]) if need}
        if not want or gsol is None:
            return (None,) * (2 + len(names))
        model = dict(zip(ctx.fields, saved[:n]))
        w, r1, r2, r3, sol = saved[n:]
        # autograd may hand out stride-0 expanded tensors (e.g. from .sum())
        grads = ctx.cp.vjp(model, w, r1, r2, r3, sol, gsol.contiguous(), want=want)
        return (None, None) + tuple(grads.get(k) for k in names)


def kkt_factor_solve(cp, model: dict, w, r1, r2, r3, b):
    """Differentiable ``cp.factor`` + ``cp.solve``: returns (sol, ok), ok not differentiable.
    Every array is a float64 CUDA tensor in the engine layout ``[size, batch_stride]``
    (``CallbackProvider.pack_model`` / ``Engine.pack``); ``model`` holds the twelve model
    blocks and, when theta_dim > 0, the ten theta blocks."""
    fields = KKT_MODEL_FIELDS + (KKT_THETA_FIELDS if cp.sizes["theta_dim"] > 0 else ())
    return _KktFactorSolve.apply(cp, len(fields), *(model[k] for k in fields), w, r1, r2, r3, b)
