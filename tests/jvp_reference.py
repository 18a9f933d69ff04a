"""CPU reference of the LQR and Newton-KKT JVPs (sipoc_lqr_jvp / sipoc_kkt_jvp), for the tests.

The tangent right-hand side is built with numpy from the formulas of include/sipoc.h, then
solved with the oracle's own factor + solve (oracle/riccati_oracle.cpp, kkt_oracle.cpp,
theta_oracle.cpp): the tangent is the same system with a new right-hand side.  Problem-major
arrays, like pyoracle; a tangent dict may hold any subset of the input names (absent: zero).
"""
from __future__ import annotations

import numpy as np

from kkt_vjp_reference import SYMMETRIC, block_table, kkt_solve, layout
from oracle import pyoracle
from vjp_reference import offsets


def _block(a, off, rows, cols):  # [batch, flat] -> [batch, rows, cols] of a column-major block
    return a[:, off:off + rows * cols].reshape(a.shape[0], cols, rows).swapaxes(1, 2)


def _mv(D, v):  # [batch, r, c] @ [batch, c] -> [batch, r]
    return np.einsum("bij,bj->bi", D, v)


def lqr_tangent_rhs(s: pyoracle.Structure, sol: dict, tan: dict) -> dict:
    """t = dK z + dh in the (q, r, c) layout for the tangents ``tan`` at the solution ``sol``."""
    x, u, y = (np.asarray(sol[k], dtype=np.float64) for k in ("x", "u", "y"))
    zeros = lambda k, size: np.asarray(tan[k], dtype=np.float64) if k in tan else \
        np.zeros((x.shape[0], size))
    o = offsets(s)
    sd, cd = [int(v) for v in s.state_dims], [int(v) for v in s.control_dims]
    nx, nu = x.shape[1], u.shape[1]
    tq, tr = zeros("q", nx).copy(), zeros("r", nu).copy()
    tc = zeros("c", nx) - zeros("delta", nx) * y
    nsl = lambda i: slice(o["n"][i], o["n"][i + 1])
    msl = lambda e: slice(o["m"][e], o["m"][e + 1])
    dQ, dM, dR = zeros("Q", o["nn"][-1]), zeros("M", o["nm"][-1]), zeros("R", o["mm"][-1])
    dA, dB = zeros("A", o["a"][-1]), zeros("B", o["b"][-1])
    for i, n in enumerate(sd):
        Q = _block(dQ, o["nn"][i], n, n)
        tq[:, nsl(i)] += _mv(0.5 * (Q + Q.swapaxes(1, 2)), x[:, nsl(i)])
    for e, m in enumerate(cd):
        p, c = int(s.parents[e]), int(s.children[e])
        xp, ue, yc = x[:, nsl(p)], u[:, msl(e)], y[:, nsl(c)]
        M = _block(dM, o["nm"][e], sd[p], m)
        R = _block(dR, o["mm"][e], m, m)
        A = _block(dA, o["a"][e], sd[c], sd[p])
        B = _block(dB, o["b"][e], sd[c], m)
        tq[:, nsl(p)] += _mv(M, ue) + _mv(A.swapaxes(1, 2), yc)
        tr[:, msl(e)] += _mv(0.5 * (R + R.swapaxes(1, 2)), ue) + _mv(M.swapaxes(1, 2), xp) + \
            _mv(B.swapaxes(1, 2), yc)
        tc[:, nsl(c)] += _mv(A, xp) + _mv(B, ue)
    return dict(q=tq, r=tr, c=tc)


def lqr_jvp(s: pyoracle.Structure, inputs: dict, sol: dict, tan: dict) -> dict:
    """Tangent x, u, y of the solution, ``rhs`` (dict q, r, c) and ``status``; problems whose
    status != 0 get zeros."""
    rhs = lqr_tangent_rhs(s, sol, tan)
    out = pyoracle.lqr_factor_solve(s, {**inputs, **rhs}, residual=False)
    failed = out["status"] != 0
    res = {k: np.where(failed[:, None], 0.0, out[k]) for k in ("x", "u", "y")}
    res.update(rhs=rhs, status=out["status"])
    return res


def kkt_tangent_rhs(s: pyoracle.Structure, p: int, sol, tan: dict):
    """t = db - dK sol over the full [x | y | z] vector for the tangents ``tan``."""
    sol = np.asarray(sol, dtype=np.float64)
    L = layout(s, p)
    xd, yd = L["x_dim"], L["y_dim"]
    t = np.asarray(tan["b"], dtype=np.float64).copy() if "b" in tan else np.zeros_like(sol)
    for name, blocks in block_table(s, p).items():
        if name not in tan:
            continue
        D, off = np.asarray(tan[name], dtype=np.float64), 0
        for r0, nr, c0, nc in blocks:
            B = _block(D, off, nr, nc)
            off += nr * nc
            if name in SYMMETRIC:
                t[:, r0:r0 + nr] -= _mv(0.5 * (B + B.swapaxes(1, 2)), sol[:, r0:r0 + nr])
            else:
                t[:, r0:r0 + nr] -= _mv(B, sol[:, c0:c0 + nc])
                t[:, c0:c0 + nc] -= _mv(B.swapaxes(1, 2), sol[:, r0:r0 + nr])
    v = lambda k, size: np.asarray(tan[k], dtype=np.float64) if k in tan else \
        np.zeros((sol.shape[0], size))
    t[:, :xd] -= v("r1", xd) * sol[:, :xd]
    t[:, xd:xd + yd] += v("r2", yd) * sol[:, xd:xd + yd]
    t[:, xd + yd:] += (v("w", L["z_dim"]) + v("r3", L["z_dim"])) * sol[:, xd + yd:]
    return t


def kkt_jvp(s: pyoracle.Structure, p: int, model: dict, theta, w, r1, r2, r3, sol,
            tan: dict) -> dict:
    """Tangent ``sol`` of the solution, ``rhs`` and ``ok``; problems with ok == 0 get zeros."""
    rhs = kkt_tangent_rhs(s, p, sol, tan)
    out = kkt_solve(s, p, model, theta, w, r1, r2, r3, rhs)
    dsol = np.where((out["ok"] == 0)[:, None], 0.0, out["sol"])
    return dict(sol=dsol, rhs=rhs, ok=out["ok"])
