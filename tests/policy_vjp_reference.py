"""CPU references of the policy VJP (sipoc_lqr_policy_vjp).

- ``policy_vjp``: the adjoint Riccati sweep in numpy, over any tree, vectorised over the
  problems of a batch, in the statement order of include/sipoc.h and policy_vjp.cuh (the
  order the kernels mirror).
- ``torch_policy``: a float64 torch restatement of ``policy_reference.lqr_policy``, the
  autograd truth the sweep is checked against.

Arrays are problem-major [batch, flat per-problem index] in the flat layout of include/sipoc.h
(policy_reference.py).  Q and R are read whole by ``torch_policy`` (as ``lqr_policy`` does);
the sweep returns the gradient with respect to the symmetric matrices, so callers compare it
with the symmetrised autograd gradient."""
import numpy as np
import torch

from oracle import pyoracle
from policy_reference import SIZE_OF, layout

INPUT_NAMES = pyoracle.LQR_INPUT_NAMES  # Q, M, R, q, r, A, B, c, delta


def _mat(flat, off, rows, cols):  # column-major blocks -> [batch, rows, cols]
    return flat[:, off:off + rows * cols].reshape(-1, cols, rows).transpose(0, 2, 1)


def _add(flat, off, mat):
    b, rows, cols = mat.shape
    flat[:, off:off + rows * cols] += mat.transpose(0, 2, 1).reshape(b, rows * cols)


def _sym(X):
    return 0.5 * (X + X.transpose(0, 2, 1))


def _mv(A, x):
    return (A @ x[:, :, None])[:, :, 0]


def policy_vjp(s, inputs, cot):
    """Gradients (dict of the nine input names) of <cot, policy> for every problem.  ``cot``
    holds any subset of K, k, V, v (absent: zero).  Every problem must factor."""
    L = layout(s)
    _st, co, ce, pre, _post = pyoracle.compile_topology(s)
    x = {k: np.asarray(inputs[k], np.float64) for k in INPUT_NAMES}
    batch = x["q"].shape[0]
    sz = pyoracle.lqr_sizes(s)
    ct = {k: (np.asarray(cot[k], np.float64) if k in cot else np.zeros((batch, sz[SIZE_OF[k]])))
          for k in ("K", "k", "V", "v")}
    from policy_reference import lqr_policy
    pol = lqr_policy(s, inputs)
    g = {k: np.zeros((batch, sz[k])) for k in INPUT_NAMES}
    nv = lambda i: slice(L["nv"][i], L["nv"][i] + int(L["n"][i]))
    Vb, vb = {}, {}
    root = s.root
    n0 = int(L["n"][root])
    Vb[root] = _sym(_mat(ct["V"], L["nn"][root], n0, n0))
    vb[root] = ct["v"][:, nv(root)].copy()
    for p in pre:
        n = int(L["n"][p])
        _add(g["Q"], L["nn"][p], Vb[p])  # Qb_p = Vb_p, qb_p = vb_p
        g["q"][:, nv(p)] += vb[p]
        for e in ce[co[p]:co[p + 1]]:
            c = int(L["chi"][e])
            nc, m = int(L["n"][c]), int(L["m"][e])
            A = _mat(x["A"], L["a"][e], nc, n)
            B = _mat(x["B"], L["b"][e], nc, m)
            M = _mat(x["M"], L["nm"][e], n, m)
            R = _mat(x["R"], L["mm"][e], m, m)
            Vc = _mat(pol["V"], L["nn"][c], nc, nc)
            vc = pol["v"][:, nv(c)]
            d, cc = x["delta"][:, nv(c)], x["c"][:, nv(c)]
            r = x["r"][:, L["mv"][e]:L["mv"][e] + m]
            # forward, recomputed: P_c, W_c, G, Y, H, K, f, g, h, k
            sd = np.sqrt(d)
            P = np.linalg.inv(np.eye(nc) + sd[:, :, None] * Vc * sd[:, None, :])
            W = (1 / sd)[:, :, None] * (np.eye(nc) - P) * (1 / sd)[:, None, :]
            Bt = B.transpose(0, 2, 1)
            G = R + Bt @ W @ B
            Y = W @ A
            H = M.transpose(0, 2, 1) + Bt @ Y
            K = -np.linalg.solve(G, H)
            f = d * vc - cc
            gg = vc - _mv(W, f)
            h = r + _mv(Bt, gg)
            k = -np.linalg.solve(G, h[:, :, None])[:, :, 0]
            # adjoint
            Vp, vp = Vb[p], vb[p]
            Kb = _mat(ct["K"], L["nm"][e], m, n) + h[:, :, None] * vp[:, None, :]
            kb = ct["k"][:, L["mv"][e]:L["mv"][e] + m]
            GiKb = np.linalg.solve(G, Kb)
            Gikb = np.linalg.solve(G, kb[:, :, None])[:, :, 0]
            Kt = K.transpose(0, 2, 1)
            hb = _mv(K, vp) - Gikb
            Hb = 2 * K @ Vp - GiKb
            Gb = _sym(K @ Vp @ Kt - GiKb @ Kt - Gikb[:, :, None] * k[:, None, :])
            gb = _mv(A, vp) + _mv(B, hb)
            Yb = B @ Hb
            fb = -_mv(W, gb)
            g["r"][:, L["mv"][e]:L["mv"][e] + m] += hb
            _add(g["M"], L["nm"][e], Hb.transpose(0, 2, 1))
            _add(g["R"], L["mm"][e], Gb)
            _add(g["A"], L["a"][e], gg[:, :, None] * vp[:, None, :] + 2 * Y @ Vp + W @ Yb)
            _add(g["B"], L["b"][e], gg[:, :, None] * hb[:, None, :] + Y @ Hb.transpose(0, 2, 1)
                 + 2 * W @ B @ Gb)
            At = A.transpose(0, 2, 1)
            Wb = _sym(A @ Vp @ At + Yb @ At + B @ Gb @ Bt - gb[:, :, None] * f[:, None, :])
            g["c"][:, nv(c)] += -fb
            g["delta"][:, nv(c)] += fb * vc - np.diagonal(W @ Wb @ W, axis1=1, axis2=2)
            S = sd[:, :, None] * P * (1 / sd)[:, None, :]
            Vb[c] = _sym(_mat(ct["V"], L["nn"][c], nc, nc)) + S @ Wb @ S.transpose(0, 2, 1)
            vb[c] = ct["v"][:, nv(c)] + gb + d * fb
    return g


def _tmat(flat, off, rows, cols):
    return flat[:, off:off + rows * cols].reshape(-1, cols, rows).transpose(1, 2)


def torch_policy(s, t):
    """policy_reference.lqr_policy in float64 torch: ``t`` holds the nine inputs as
    [batch, size] tensors; returns dict K, k, V, v of [batch, size] tensors."""
    L = layout(s)
    _st, co, ce, _pre, post = pyoracle.compile_topology(s)
    batch = t["q"].shape[0]
    blocks = {k: {} for k in ("K", "k", "V", "v")}
    W, V, v = {}, {}, {}
    for node in post:
        n = int(L["n"][node])
        Vi = _tmat(t["Q"], L["nn"][node], n, n)
        vi = t["q"][:, L["nv"][node]:L["nv"][node] + n]
        for e in ce[co[node]:co[node + 1]]:
            c = int(L["chi"][e])
            nc, me = int(L["n"][c]), int(L["m"][e])
            A = _tmat(t["A"], L["a"][e], nc, n)
            B = _tmat(t["B"], L["b"][e], nc, me)
            M = _tmat(t["M"], L["nm"][e], n, me)
            R = _tmat(t["R"], L["mm"][e], me, me)
            Wc = W[c]
            G = R + B.transpose(1, 2) @ Wc @ B
            F = Wc @ A
            H = M.transpose(1, 2) + B.transpose(1, 2) @ F
            K = -torch.linalg.solve(G, H)
            Vi = Vi + A.transpose(1, 2) @ F + K.transpose(1, 2) @ H
            dc = t["delta"][:, L["nv"][c]:L["nv"][c] + nc]
            cc = t["c"][:, L["nv"][c]:L["nv"][c] + nc]
            f = dc * v[c] - cc
            g = v[c] - (Wc @ f[:, :, None])[:, :, 0]
            h = t["r"][:, L["mv"][e]:L["mv"][e] + me] + (B.transpose(1, 2) @ g[:, :, None])[:, :, 0]
            k = -torch.linalg.solve(G, h[:, :, None])[:, :, 0]
            vi = vi + (A.transpose(1, 2) @ g[:, :, None])[:, :, 0] \
                + (K.transpose(1, 2) @ h[:, :, None])[:, :, 0]
            blocks["K"][e] = K.transpose(1, 2).reshape(batch, -1)
            blocks["k"][e] = k
        d = t["delta"][:, L["nv"][node]:L["nv"][node] + n]
        sd = d.sqrt()
        eye = torch.eye(n, dtype=torch.float64)
        Fi = torch.linalg.inv(eye + sd[:, :, None] * Vi * sd[:, None, :])
        W[node] = (1 / sd)[:, :, None] * (eye - Fi) * (1 / sd)[:, None, :]
        V[node], v[node] = Vi, vi
        blocks["V"][node] = Vi.transpose(1, 2).reshape(batch, -1)
        blocks["v"][node] = vi
    E, N = s.num_edges, s.num_edges + 1
    cat = lambda parts, count: torch.cat([parts[i] for i in range(count)], 1) if count else \
        torch.zeros(batch, 0, dtype=torch.float64)
    return dict(K=cat(blocks["K"], E), k=cat(blocks["k"], E), V=cat(blocks["V"], N),
                v=cat(blocks["v"], N))


def autograd_policy_vjp(s, inputs, cot):
    """torch.autograd gradients of <cot, torch_policy> (dict of the nine names, numpy), Q and
    R symmetrised per block (the convention of the sweep and the kernels)."""
    t = {k: torch.tensor(np.asarray(inputs[k], np.float64), requires_grad=True)
         for k in INPUT_NAMES}
    pol = torch_policy(s, t)
    loss = sum((torch.as_tensor(np.asarray(cot[k], np.float64)) * pol[k]).sum() for k in cot)
    names = [k for k in INPUT_NAMES]
    grads = torch.autograd.grad(loss, [t[k] for k in names], allow_unused=True)
    out = {k: (np.zeros_like(np.asarray(inputs[k], np.float64)) if gr is None else gr.numpy())
           for k, gr in zip(names, grads)}
    L = layout(s)
    for key, off, dims in (("Q", "nn", L["n"]), ("R", "mm", L["m"])):
        for i, d in enumerate(dims):
            d = int(d)
            blk = _mat(out[key], L[off][i], d, d)
            out[key][:, L[off][i]:L[off][i] + d * d] = \
                _sym(blk).transpose(0, 2, 1).reshape(-1, d * d)
    return out
