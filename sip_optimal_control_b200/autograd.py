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

Both Functions also differentiate in forward mode (``torch.autograd.forward_ad`` dual tensors,
``torch.func.jvp``, ``gradcheck(..., check_forward_ad=True)``): the tangent of the solution is
one more solve of the same system whose right-hand side the tangents of the inputs build
(``sipoc_lqr_jvp`` / ``sipoc_kkt_jvp``).  Absent tangents cost nothing; the symmetric blocks
enter through their symmetric parts, the transpose of the gradient convention above; failed
problems and padding lanes get a zero tangent.  ``torch.func.vmap``, ``jacfwd`` and ``jacrev``
are not supported: they need a solve with many right-hand sides at once, and raise.
"""
from __future__ import annotations

import torch
from torch._C import _functorch

from ._capi import KKT_MODEL_FIELDS, KKT_THETA_FIELDS, LQR_INPUT_FIELDS


def _plain(t):
    """The storage-backed tensor under any functorch wrappers: under ``torch.func.jvp`` the
    tensors saved for forward (and the tangents) reach ``jvp`` wrapped, and the engine needs
    their device pointers.  The values are the primal ones.  Call it, and the engine, under
    ``_DisableFuncTorch``, so that the tensors they allocate are plain too."""
    while _functorch.is_functorch_wrapped_tensor(t):
        t = _functorch.get_unwrapped(t)
    return t.contiguous()


_LQR_KEPT = ("Q", "M", "R", "A", "B", "delta")  # the inputs either derivative reads


class _FactorSolve(torch.autograd.Function):
    @staticmethod
    def forward(lqr, *arrays):
        inp = {k: a.contiguous() for k, a in zip(LQR_INPUT_FIELDS, arrays)}
        out = lqr.alloc_output()
        status = lqr.factor_solve(inp, out)
        return out["x"], out["u"], out["y"], status

    @staticmethod
    def setup_context(ctx, inputs, output):
        lqr, *arrays = inputs
        x, u, y, status = output
        inp = dict(zip(LQR_INPUT_FIELDS, arrays))
        kept = tuple(inp[k] for k in _LQR_KEPT) + (x, u, y)
        ctx.lqr = lqr
        ctx.save_for_backward(*kept)
        ctx.save_for_forward(*kept)
        ctx.mark_non_differentiable(status)

    @staticmethod
    def backward(ctx, gx, gu, gy, _gstatus):
        Q, M, R, A, B, delta, x, u, y = (a.contiguous() for a in ctx.saved_tensors)
        want = {k for k, need in zip(LQR_INPUT_FIELDS, ctx.needs_input_grad[1:]) if need}
        if not want:
            return (None,) * (1 + len(LQR_INPUT_FIELDS))
        # autograd may hand out stride-0 expanded tensors (e.g. from .sum()) or None
        cot = {k: torch.zeros_like(ref) if g is None else g.contiguous()
               for k, g, ref in (("x", gx, x), ("u", gu, u), ("y", gy, y))}
        inp = dict(Q=Q, M=M, R=R, A=A, B=B, delta=delta)
        grads = ctx.lqr.vjp(inp, dict(x=x, u=u, y=y), cot, want=want)
        return (None,) + tuple(grads.get(k) for k in LQR_INPUT_FIELDS)

    @staticmethod
    def jvp(ctx, _lqr_t, *tangents):
        with torch._C._DisableFuncTorch():
            saved = [_plain(a) for a in ctx.saved_tensors]
            # forward_ad may hand out stride-0 expanded tangents; None is a zero tangent
            tan = {k: _plain(t) for k, t in zip(LQR_INPUT_FIELDS, tangents) if t is not None}
            res = ctx.lqr.jvp(dict(zip(_LQR_KEPT, saved[:6])), dict(zip("xuy", saved[6:])), tan)
        return res["x"], res["u"], res["y"], None


def factor_solve(lqr, inp: dict):
    """Differentiable ``lqr.factor_solve``: returns (x, u, y, status), status not
    differentiable.  ``inp`` holds float64 CUDA tensors in the engine layout
    ``[size, batch_stride]`` (``LQR.alloc_input`` / ``LQR.pack_input``)."""
    return _FactorSolve.apply(lqr, *(inp[k] for k in LQR_INPUT_FIELDS))


_KKT_VECTORS = ("w", "r1", "r2", "r3", "b")


class _KktFactorSolve(torch.autograd.Function):
    @staticmethod
    def forward(cp, n_model, *arrays):
        fields = (KKT_MODEL_FIELDS + KKT_THETA_FIELDS)[:n_model]
        model = {k: a.contiguous() for k, a in zip(fields, arrays[:n_model])}
        w, r1, r2, r3, b = (a.contiguous() for a in arrays[n_model:])
        ok = cp.factor(model, w, r1, r2, r3)
        sol = cp.engine.zeros(cp.sizes["kkt_dim"])
        cp.solve(model, b, sol)
        return sol, ok

    @staticmethod
    def setup_context(ctx, inputs, output):
        cp, n_model, *arrays = inputs
        sol, ok = output
        ctx.cp, ctx.fields = cp, (KKT_MODEL_FIELDS + KKT_THETA_FIELDS)[:n_model]
        kept = tuple(arrays[:n_model + 4]) + (sol,)  # the model, w, r1, r2, r3 and sol; not b
        ctx.save_for_backward(*kept)
        ctx.save_for_forward(*kept)
        ctx.mark_non_differentiable(ok)

    @staticmethod
    def backward(ctx, gsol, _gok):
        saved = [a.contiguous() for a in ctx.saved_tensors]
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

    @staticmethod
    def jvp(ctx, _cp_t, _n_t, *tangents):
        n = len(ctx.fields)
        names = ctx.fields + _KKT_VECTORS
        with torch._C._DisableFuncTorch():
            saved = [_plain(a) for a in ctx.saved_tensors]
            tan = {k: _plain(t) for k, t in zip(names, tangents) if t is not None}
            w, r1, r2, r3, sol = saved[n:]
            res = ctx.cp.jvp(dict(zip(ctx.fields, saved[:n])), w, r1, r2, r3, sol, tan)
        return res["sol"], None


def kkt_factor_solve(cp, model: dict, w, r1, r2, r3, b):
    """Differentiable ``cp.factor`` + ``cp.solve``: returns (sol, ok), ok not differentiable.
    Every array is a float64 CUDA tensor in the engine layout ``[size, batch_stride]``
    (``CallbackProvider.pack_model`` / ``Engine.pack``); ``model`` holds the twelve model
    blocks and, when theta_dim > 0, the ten theta blocks."""
    fields = KKT_MODEL_FIELDS + (KKT_THETA_FIELDS if cp.sizes["theta_dim"] > 0 else ())
    return _KktFactorSolve.apply(cp, len(fields), *(model[k] for k in fields), w, r1, r2, r3, b)
