"""CPU reference of the policy JVP (sipoc_lqr_policy_jvp): the tangent Riccati sweep in numpy,
over any tree, vectorised over the problems of a batch, in the statement order of
policy_jvp.cuh and of both kernels of policy_jvp.cu.

Arrays are problem-major [batch, flat per-problem index] in the flat layout of include/sipoc.h
(policy_reference.py).  dQ and dR enter through their symmetric parts, and the root's dc and
ddelta are not read, the transposes of the conventions of ``policy_vjp_reference.policy_vjp``."""
import numpy as np

from oracle import pyoracle
from policy_reference import SIZE_OF, layout, lqr_policy
from policy_vjp_reference import INPUT_NAMES, _add, _mat, _mv, _sym


def _T(X):
    return X.transpose(0, 2, 1)


def policy_jvp(s, inputs, tan):
    """Tangents (dict K, k, V, v) of the policy for every problem.  ``tan`` holds the tangents
    of any subset of the nine input names (absent: zero).  Every problem must factor."""
    L = layout(s)
    _st, co, ce, _pre, post = pyoracle.compile_topology(s)
    x = {k: np.asarray(inputs[k], np.float64) for k in INPUT_NAMES}
    batch = x["q"].shape[0]
    sz = pyoracle.lqr_sizes(s)
    t = {k: (np.asarray(tan[k], np.float64) if k in tan else np.zeros((batch, sz[k])))
         for k in INPUT_NAMES}
    pol = lqr_policy(s, inputs)
    out = {k: np.zeros((batch, sz[SIZE_OF[k]])) for k in ("K", "k", "V", "v")}
    nv = lambda i: slice(L["nv"][i], L["nv"][i] + int(L["n"][i]))
    dV, dv = {}, {}
    for p in post:
        n = int(L["n"][p])
        dVp = _sym(_mat(t["Q"], L["nn"][p], n, n))  # dV_p = sym(dQ_p), dv_p = dq_p
        dvp = t["q"][:, nv(p)].copy()
        for e in ce[co[p]:co[p + 1]]:  # child_offsets order
            c = int(L["chi"][e])
            nc, m = int(L["n"][c]), int(L["m"][e])
            A, dA = _mat(x["A"], L["a"][e], nc, n), _mat(t["A"], L["a"][e], nc, n)
            B, dB = _mat(x["B"], L["b"][e], nc, m), _mat(t["B"], L["b"][e], nc, m)
            M, dM = _mat(x["M"], L["nm"][e], n, m), _mat(t["M"], L["nm"][e], n, m)
            R, dR = _mat(x["R"], L["mm"][e], m, m), _mat(t["R"], L["mm"][e], m, m)
            r = x["r"][:, L["mv"][e]:L["mv"][e] + m]
            dr = t["r"][:, L["mv"][e]:L["mv"][e] + m]
            Vc, vc = _mat(pol["V"], L["nn"][c], nc, nc), pol["v"][:, nv(c)]
            d, cc = x["delta"][:, nv(c)], x["c"][:, nv(c)]
            dd, dc = t["delta"][:, nv(c)], t["c"][:, nv(c)]
            # primal (policy_common.cuh, edge_primal)
            sd = np.sqrt(d)
            sdi = 1.0 / sd
            P = np.linalg.inv(np.eye(nc) + sd[:, :, None] * Vc * sd[:, None, :])
            P = np.tril(P) + _T(np.tril(P, -1))
            W = sdi[:, :, None] * (np.eye(nc) - P) * sdi[:, None, :]
            WB = W @ B
            G = R + _T(B) @ WB
            Y = W @ A
            K = -np.linalg.solve(G, _T(M) + _T(B) @ Y)
            f = d * vc - cc
            g = vc - _mv(W, f)
            h = r + _mv(_T(B), g)
            k = -np.linalg.solve(G, h[:, :, None])[:, :, 0]
            # tangent: T = dV_c S, dW = S' T - W dD W  (S = D^1/2 P D^-1/2)
            S = sd[:, :, None] * P * sdi[:, None, :]
            Tm = dV[c] @ S
            dW = _T(S) @ Tm - W @ (dd[:, :, None] * W)
            dWB = dW @ B
            dWA = dW @ A
            dG = _sym(dR) + _T(dB) @ WB + _T(WB) @ dB + _T(B) @ dWB
            df = dd * vc + d * dv[c] - dc
            dY = dWA + W @ dA
            dg = dv[c] - _mv(dW, f) - _mv(W, df)
            dH = _T(dM) + _T(dB) @ Y + _T(B) @ dY
            dh = dr + _mv(_T(dB), g) + _mv(_T(B), dg)
            dGK = dG @ K
            dK = -np.linalg.solve(G, dH + dGK)
            dk = -np.linalg.solve(G, (dh + _mv(dG, k))[:, :, None])[:, :, 0]
            inc = (_T(dA) @ Y + _T(Y) @ dA + _T(A) @ dWA) + (_T(dH) @ K + _T(K) @ dH + _T(K) @ dGK)
            inc = np.tril(inc) + _T(np.tril(inc, -1))  # one triangle, mirrored
            dVp = dVp + inc
            dvp = dvp + (_mv(_T(dA), g) + _mv(_T(A), dg)) + (_mv(_T(dK), h) + _mv(_T(K), dh))
            _add(out["K"], L["nm"][e], dK)
            out["k"][:, L["mv"][e]:L["mv"][e] + m] = dk
        dV[p], dv[p] = dVp, dvp
        _add(out["V"], L["nn"][p], dVp)
        out["v"][:, nv(p)] = dvp
    return out
