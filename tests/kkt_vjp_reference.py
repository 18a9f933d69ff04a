"""CPU reference of the Newton-KKT VJP (sipoc_kkt_vjp), for the tests.

The adjoint is the oracle's own factor + solve (oracle/kkt_oracle.cpp, theta_oracle.cpp) with
the cotangent as right-hand side -- K is symmetric, so lam = K^-1 g is that solve -- and the
gradient table of include/sipoc.h is applied block by block.  Problem-major arrays, vectors in
the full layout [x_s, theta | y | z], like pyoracle.
"""
from __future__ import annotations

import numpy as np

from oracle import pyoracle

MODEL_NAMES = pyoracle.KKT_MODEL_NAMES
THETA_NAMES = pyoracle.THETA_MODEL_NAMES
VECTOR_NAMES = ("b", "w", "r1", "r2", "r3")
# symmetric Hessian blocks: gradient with respect to the symmetric matrix
SYMMETRIC = ("node_hxx", "edge_hxx", "edge_huu", "node_htt", "edge_htt")


def _dims(s: pyoracle.Structure):
    sd, cd = np.asarray(s.state_dims), np.asarray(s.control_dims)
    N, E = len(sd), len(cd)
    z = lambda a, k: np.zeros(k, int) if a is None else np.asarray(a, int)
    return sd, cd, z(s.node_c, N), z(s.node_g, N), z(s.edge_c, E), z(s.edge_g, E)


def layout(s: pyoracle.Structure, p: int) -> dict:
    """Row starts of every node / edge segment in the full [x_s, theta | y | z] vector, and the
    full sizes."""
    sz = pyoracle.kkt_sizes(s)
    o = {k: np.asarray(v, int) for k, v in pyoracle.kkt_offsets(s).items()}
    sx = sz["x_dim"]
    xd, yd, zd = sx + p, sz["y_dim"], sz["z_dim"]
    return dict(x_state=o["x_state"], x_control=o["x_control"], y_dyn=xd + o["y_dyn"],
                y_node_c=xd + o["y_node_c"], y_edge_c=xd + o["y_edge_c"],
                z_node=xd + yd + o["z_node"], z_edge=xd + yd + o["z_edge"], theta=sx,
                x_dim=xd, y_dim=yd, z_dim=zd, kkt_dim=xd + yd + zd)


def block_table(s: pyoracle.Structure, p: int = 0) -> dict:
    """name -> [(row start, rows, column start, columns)], one entry per block of that array in
    storage order: block k of the array is the column-major rows x columns matrix at
    K[row start:, column start:] (its transpose at K[column start:, row start:])."""
    sd, cd, nc, ng, ec, eg = _dims(s)
    L = layout(s, p)
    par, chi = np.asarray(s.parents, int), np.asarray(s.children, int)
    th = L["theta"]
    t = {k: [] for k in MODEL_NAMES + (THETA_NAMES if p else ())}
    for i in range(len(sd)):
        n, xs = sd[i], L["x_state"][i]
        t["node_hxx"].append((xs, n, xs, n))
        t["node_jc"].append((L["y_node_c"][i], nc[i], xs, n))
        t["node_jg"].append((L["z_node"][i], ng[i], xs, n))
        if p:
            t["node_hxt"].append((xs, n, th, p))
            t["node_jct"].append((L["y_node_c"][i], nc[i], th, p))
            t["node_jgt"].append((L["z_node"][i], ng[i], th, p))
            t["node_htt"].append((th, p, th, p))
    for e in range(len(cd)):
        pa, ch, m = par[e], chi[e], cd[e]
        xp, npa, xu, yc = L["x_state"][pa], sd[pa], L["x_control"][e], L["y_dyn"][ch]
        t["edge_hxx"].append((xp, npa, xp, npa))
        t["edge_hxu"].append((xp, npa, xu, m))
        t["edge_huu"].append((xu, m, xu, m))
        t["edge_A"].append((yc, sd[ch], xp, npa))
        t["edge_B"].append((yc, sd[ch], xu, m))
        t["edge_jcx"].append((L["y_edge_c"][e], ec[e], xp, npa))
        t["edge_jcu"].append((L["y_edge_c"][e], ec[e], xu, m))
        t["edge_jgx"].append((L["z_edge"][e], eg[e], xp, npa))
        t["edge_jgu"].append((L["z_edge"][e], eg[e], xu, m))
        if p:
            t["edge_hxt"].append((xp, npa, th, p))
            t["edge_hut"].append((xu, m, th, p))
            t["edge_dynt"].append((yc, sd[ch], th, p))
            t["edge_jct"].append((L["y_edge_c"][e], ec[e], th, p))
            t["edge_jgt"].append((L["z_edge"][e], eg[e], th, p))
            t["edge_htt"].append((th, p, th, p))
    return t


def _colmajor(G):  # [batch, rows, cols] -> [batch, rows * cols], column-major
    return np.swapaxes(G, 1, 2).reshape(G.shape[0], -1)


def kkt_solve(s, p, model, theta, w, r1, r2, r3, b):
    """The oracle's factor + solve on the full layout: dict(sol, ok)."""
    if p:
        return pyoracle.kkt_theta_factor_solve(s, p, model, theta, w, r1, r2, r3, b)
    out = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, b, residual=False)
    return dict(sol=out["sol"], ok=out["ok"])


def kkt_vjp(s: pyoracle.Structure, p: int, model: dict, theta, w, r1, r2, r3, sol, cot) -> dict:
    """Gradients of L w.r.t. every model block (theta blocks when p > 0), b, w, r1, r2, r3 for
    dL/dsol = cot at the solution sol.  Returns those arrays, ``adjoint`` and ``ok``; problems
    with ok == 0 get zero gradients."""
    adj = kkt_solve(s, p, model, theta, w, r1, r2, r3, cot)
    lam, x = adj["sol"], np.asarray(sol, dtype=np.float64)
    batch = x.shape[0]
    out = {}
    for name, blocks in block_table(s, p).items():
        scale = 0.5 if name in SYMMETRIC else 1.0
        parts = []
        for r0, nr, c0, nc in blocks:
            lr, sr = lam[:, r0:r0 + nr], x[:, r0:r0 + nr]
            lc, sc = lam[:, c0:c0 + nc], x[:, c0:c0 + nc]
            G = -scale * (lr[:, :, None] * sc[:, None, :] + sr[:, :, None] * lc[:, None, :])
            parts.append(_colmajor(G))
        out[name] = np.concatenate(parts, axis=1) if parts else np.zeros((batch, 0))
    L = layout(s, p)
    xd, yd = L["x_dim"], L["y_dim"]
    prod = lam * x
    out.update(b=lam.copy(), r1=-prod[:, :xd], r2=prod[:, xd:xd + yd], w=prod[:, xd + yd:],
               r3=prod[:, xd + yd:].copy())
    failed = adj["ok"] == 0
    for k in out:
        out[k][failed] = 0.0
    out["adjoint"] = lam
    out["ok"] = adj["ok"]
    return out
