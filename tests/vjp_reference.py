"""CPU reference of the LQR VJP (sipoc_lqr_vjp), for the tests.

The adjoint is the oracle's own factor + solve (oracle/riccati_oracle.cpp) with the
cotangent as (q, r, c) -- K is symmetric, so mu = -K^-1 g is that solve -- and the gradient
table of include/sipoc.h is applied block by block.  Problem-major arrays, like pyoracle.
"""
from __future__ import annotations

import numpy as np

from oracle import pyoracle

GRAD_NAMES = pyoracle.LQR_INPUT_NAMES


def offsets(s: pyoracle.Structure) -> dict:
    """Start of every node / edge block in the flat per-problem arrays (sizes appended)."""
    sd, cd = np.asarray(s.state_dims), np.asarray(s.control_dims)
    par, chi = np.asarray(s.parents), np.asarray(s.children)
    cum = lambda v: np.concatenate([[0], np.cumsum(v)]).astype(int)
    return dict(nn=cum(sd * sd), n=cum(sd), nm=cum(sd[par] * cd), mm=cum(cd * cd), m=cum(cd),
                a=cum(sd[chi] * sd[par]), b=cum(sd[chi] * cd))


def _colmajor(G):  # [batch, rows, cols] -> [batch, rows * cols], column-major
    return np.swapaxes(G, 1, 2).reshape(G.shape[0], -1)


def _outer(a, b):  # [batch, r], [batch, c] -> [batch, r, c]
    return a[:, :, None] * b[:, None, :]


def lqr_vjp(s: pyoracle.Structure, inputs: dict, sol: dict, cot: dict) -> dict:
    """Gradients of L w.r.t. the nine input arrays for dL/d(x, u, y) = cot[x, u, y] at the
    solution sol[x, u, y].  Returns the nine arrays, ``adjoint`` (dict x, u, y) and
    ``status``; problems whose status != 0 get zero gradients."""
    adj_in = dict(inputs)
    adj_in.update(q=cot["x"], r=cot["u"], c=cot["y"])
    adj = pyoracle.lqr_factor_solve(s, adj_in, residual=False)
    mx, mu, my = adj["x"], adj["u"], adj["y"]
    x, u, y = (np.asarray(sol[k], dtype=np.float64) for k in ("x", "u", "y"))
    batch = x.shape[0]
    o = offsets(s)
    N, E = len(s.state_dims), s.num_edges
    nsl = lambda i: slice(o["n"][i], o["n"][i + 1])
    msl = lambda e: slice(o["m"][e], o["m"][e + 1])
    g = {k: [] for k in ("Q", "M", "R", "A", "B")}
    for i in range(N):
        X, MX = x[:, nsl(i)], mx[:, nsl(i)]
        g["Q"].append(_colmajor(0.5 * (_outer(MX, X) + _outer(X, MX))))
    for e in range(E):
        p, c = s.parents[e], s.children[e]
        Xp, MXp, Yc, MYc = x[:, nsl(p)], mx[:, nsl(p)], y[:, nsl(c)], my[:, nsl(c)]
        U, MU = u[:, msl(e)], mu[:, msl(e)]
        g["M"].append(_colmajor(_outer(MXp, U) + _outer(Xp, MU)))
        g["R"].append(_colmajor(0.5 * (_outer(MU, U) + _outer(U, MU))))
        g["A"].append(_colmajor(_outer(Yc, MXp) + _outer(MYc, Xp)))
        g["B"].append(_colmajor(_outer(Yc, MU) + _outer(MYc, U)))
    out = {k: (np.concatenate(v, axis=1) if v else np.zeros((batch, 0))) for k, v in g.items()}
    out.update(q=mx.copy(), r=mu.copy(), c=my.copy(), delta=-my * y)
    failed = adj["status"] != 0
    for k in GRAD_NAMES:
        out[k][failed] = 0.0
    out["adjoint"] = dict(x=mx, u=mu, y=my)
    out["status"] = adj["status"]
    return out
