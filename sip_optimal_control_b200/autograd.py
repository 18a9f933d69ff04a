"""``torch.autograd`` binding of the batched LQR solve.

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
"""
from __future__ import annotations

import torch

from ._capi import LQR_INPUT_FIELDS


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
