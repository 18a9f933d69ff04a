"""CPU reference of the LQR feedback policy (sipoc_lqr_factor_solve_policy): the reference's
K, k, V, v after factor_with_status + solve (lqr.cpp:645-796, restated statement by statement
in oracle/riccati_oracle.cpp), in numpy, vectorised over the problems of a batch.

Arrays are problem-major [batch, flat per-problem index] in the flat layout of include/sipoc.h:
K per edge m_e x n_parent column-major (the element count of M), k per edge (that of r), V per
node n_i x n_i (that of Q), v per node (that of q).  Problems whose factorization fails get
unspecified values; callers mask them with the oracle's status."""
import numpy as np

from oracle import pyoracle

POLICY_NAMES = ("K", "k", "V", "v")
SIZE_OF = dict(K="M", k="r", V="Q", v="q")


def layout(s):
    """Flat offsets of every block (oracle FlatLayout, riccati_oracle.hpp)."""
    n = np.asarray(s.state_dims, np.int64)
    m = np.asarray(s.control_dims, np.int64)[: s.num_edges]
    par, chi = np.asarray(s.parents), np.asarray(s.children)
    cum = lambda sizes: np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return dict(n=n, m=m, par=par, chi=chi, nn=cum(n * n), nv=cum(n), nm=cum(n[par] * m),
                mm=cum(m * m), mv=cum(m), a=cum(n[chi] * n[par]), b=cum(n[chi] * m))


def _mat(flat, off, rows, cols):  # column-major blocks -> [batch, rows, cols]
    return flat[:, off:off + rows * cols].reshape(-1, cols, rows).transpose(0, 2, 1)


def _put(flat, off, mat):
    b, rows, cols = mat.shape
    flat[:, off:off + rows * cols] = mat.transpose(0, 2, 1).reshape(b, rows * cols)


def lqr_policy(s, inputs):
    """dict K, k, V, v of the reference for every problem of `inputs` (pyoracle layout)."""
    L = layout(s)
    st, co, ce, pre, post = pyoracle.compile_topology(s)
    assert st == 0
    x = {k: np.asarray(inputs[k], np.float64) for k in pyoracle.LQR_INPUT_NAMES}
    batch = x["q"].shape[0]
    sz = pyoracle.lqr_sizes(s)
    out = {k: np.zeros((batch, sz[SIZE_OF[k]])) for k in POLICY_NAMES}
    V, v, W = {}, {}, {}
    for node in post:
        n = int(L["n"][node])
        Vi = _mat(x["Q"], L["nn"][node], n, n).copy()  # :658
        vi = x["q"][:, L["nv"][node]:L["nv"][node] + n].copy()  # :744
        for e in ce[co[node]:co[node + 1]]:
            c = int(L["chi"][e])
            nc, me = int(L["n"][c]), int(L["m"][e])
            A = _mat(x["A"], L["a"][e], nc, n)
            B = _mat(x["B"], L["b"][e], nc, me)
            M = _mat(x["M"], L["nm"][e], n, me)
            R = _mat(x["R"], L["mm"][e], me, me)
            Wc = W[c]
            G = R + B.transpose(0, 2, 1) @ Wc @ B  # :692-694
            F = Wc @ A  # :703
            H = M.transpose(0, 2, 1) + B.transpose(0, 2, 1) @ F  # :704-705
            K = -np.linalg.solve(G, H)  # :707-713
            Vi = Vi + A.transpose(0, 2, 1) @ F  # :715
            Vi = Vi + K.transpose(0, 2, 1) @ H  # :716-719
            dc = x["delta"][:, L["nv"][c]:L["nv"][c] + nc]
            cc = x["c"][:, L["nv"][c]:L["nv"][c] + nc]
            f = dc * v[c] - cc  # :778-779
            g = v[c] - (Wc @ f[:, :, None])[:, :, 0]  # :780-781
            h = x["r"][:, L["mv"][e]:L["mv"][e] + me] + (B.transpose(0, 2, 1) @ g[:, :, None])[:, :, 0]
            k = -np.linalg.solve(G, h[:, :, None])[:, :, 0]  # :785-791
            vi = vi + (A.transpose(0, 2, 1) @ g[:, :, None])[:, :, 0] \
                + (K.transpose(0, 2, 1) @ h[:, :, None])[:, :, 0]  # :793-794
            _put(out["K"], L["nm"][e], K)
            out["k"][:, L["mv"][e]:L["mv"][e] + me] = k
        d = x["delta"][:, L["nv"][node]:L["nv"][node] + n]
        # W = D^-1/2 (I - F^-1) D^-1/2, F = I + D^1/2 V D^1/2 (lqr.cpp:475-529)
        sd = np.sqrt(np.abs(d))
        Fm = np.eye(n) + sd[:, :, None] * Vi * sd[:, None, :]
        Fi = np.linalg.inv(Fm)
        sdi = 1.0 / np.where(sd > 0, sd, 1.0)
        W[node] = sdi[:, :, None] * (np.eye(n) - Fi) * sdi[:, None, :]
        V[node], v[node] = Vi, vi
        _put(out["V"], L["nn"][node], Vi)
        out["v"][:, L["nv"][node]:L["nv"][node] + n] = vi
    return out


def policy_residuals(s, inputs, pol, x, u, y):
    """Per problem: max |u_e - k_e - K_e x_p| / scale and max |y_i - v_i - V_i x_i| / scale."""
    L = layout(s)
    ru = np.zeros(x.shape[0])
    ry = np.zeros(x.shape[0])
    for e in range(s.num_edges):
        p, me, np_ = int(L["par"][e]), int(L["m"][e]), int(L["n"][L["par"][e]])
        K = _mat(pol["K"], L["nm"][e], me, np_)
        xp = x[:, L["nv"][p]:L["nv"][p] + np_]
        ue = u[:, L["mv"][e]:L["mv"][e] + me]
        Kx = (K @ xp[:, :, None])[:, :, 0]
        pred = pol["k"][:, L["mv"][e]:L["mv"][e] + me] + Kx
        scale = 1.0 + np.abs(ue).max(1) + np.abs(Kx).max(1, initial=0.0)
        ru = np.maximum(ru, np.abs(ue - pred).max(1, initial=0.0) / scale)
    for i in range(s.num_edges + 1):
        n = int(L["n"][i])
        Vi = _mat(pol["V"], L["nn"][i], n, n)
        xi = x[:, L["nv"][i]:L["nv"][i] + n]
        yi = y[:, L["nv"][i]:L["nv"][i] + n]
        Vx = (Vi @ xi[:, :, None])[:, :, 0]
        pred = pol["v"][:, L["nv"][i]:L["nv"][i] + n] + Vx
        scale = 1.0 + np.abs(yi).max(1) + np.abs(Vx).max(1, initial=0.0)
        ry = np.maximum(ry, np.abs(yi - pred).max(1, initial=0.0) / scale)
    return ru, ry
