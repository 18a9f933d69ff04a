"""The CPU reference of the LQR VJP (vjp_reference.py: the oracle's solve with the cotangent as
right-hand side, then the gradient table of include/sipoc.h) against two independent
derivatives of the same solve:
- torch.autograd through a dense torch.linalg.solve of the KKT system (assembled here, with
  Q = (P + P^T) / 2 and R likewise, so dL/dP is the symmetric gradient), 1e-10;
- central finite differences of the oracle's own solve (symmetric perturbations of Q, R),
  1e-6 relative."""
import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import rel_err
from oracle import pyoracle
from vjp_reference import GRAD_NAMES, lqr_vjp, offsets


def _benchmark_chain():
    return pg.lqr_benchmark_batch(4, 2, 5, 1, seed=3, dense_M=True)


CASES = {
    "nonuniform_delta_chain": lambda: _flat(fx.nonuniform_delta_chain()),
    "branch_tree": lambda: _flat(fx.branch_tree()),
    "variable_dim_branch_tree": lambda: _flat(fx.variable_dim_branch_tree()),
    "benchmark_chain": _benchmark_chain,
}


def _flat(sp):
    s, p = sp
    return s, fx.pack_problem(**p)


def _case(name, seed=0):
    s, host = CASES[name]()
    sz = pyoracle.lqr_sizes(s)
    rng = np.random.default_rng(seed)
    cot = {k: rng.standard_normal((1, sz[k])) for k in ("x", "u", "y")}
    sol = pyoracle.lqr_factor_solve(s, host)
    assert (sol["status"] == 0).all()
    return s, host, sol, cot


def _dense_loss(s, f, cot):
    """L = cot . z with z the dense solve of K z = -h; f: flat 1-D torch arrays of one problem."""
    o = offsets(s)
    sd, cd = [int(v) for v in s.state_dims], [int(v) for v in s.control_dims]
    N, E = len(sd), len(cd)
    blk = lambda k, off, r, c: f[k][off:off + r * c].reshape(c, r).T  # column-major block
    nx, nu = o["n"][-1], o["m"][-1]
    dim = 2 * nx + nu
    xo = lambda i: int(o["n"][i])
    uo = lambda e: nx + int(o["m"][e])
    yo = lambda i: nx + nu + int(o["n"][i])
    K = torch.zeros(dim, dim, dtype=torch.float64)
    h = torch.zeros(dim, dtype=torch.float64)
    for i in range(N):  # stationarity in x_i
        n, r0 = sd[i], xo(i)
        P = blk("Q", o["nn"][i], n, n)
        K[r0:r0 + n, xo(i):xo(i) + n] += 0.5 * (P + P.T)
        K[r0:r0 + n, yo(i):yo(i) + n] -= torch.eye(n, dtype=torch.float64)
        h[r0:r0 + n] = f["q"][o["n"][i]:o["n"][i + 1]]
    for e in range(E):
        p, c, m = int(s.parents[e]), int(s.children[e]), cd[e]
        npar, nc = sd[p], sd[c]
        M = blk("M", o["nm"][e], npar, m)
        P = blk("R", o["mm"][e], m, m)
        A = blk("A", o["a"][e], nc, npar)
        B = blk("B", o["b"][e], nc, m)
        K[xo(p):xo(p) + npar, uo(e):uo(e) + m] += M
        K[xo(p):xo(p) + npar, yo(c):yo(c) + nc] += A.T
        K[uo(e):uo(e) + m, xo(p):xo(p) + npar] += M.T
        K[uo(e):uo(e) + m, uo(e):uo(e) + m] += 0.5 * (P + P.T)
        K[uo(e):uo(e) + m, yo(c):yo(c) + nc] += B.T
        h[uo(e):uo(e) + m] = f["r"][o["m"][e]:o["m"][e + 1]]
        K[yo(c):yo(c) + nc, xo(p):xo(p) + npar] += A
        K[yo(c):yo(c) + nc, uo(e):uo(e) + m] += B
    for i in range(N):  # dynamics rows (the root's: -x - delta y + c = 0)
        n = sd[i]
        K[yo(i):yo(i) + n, xo(i):xo(i) + n] -= torch.eye(n, dtype=torch.float64)
        K[yo(i):yo(i) + n, yo(i):yo(i) + n] -= torch.diag(f["delta"][o["n"][i]:o["n"][i + 1]])
        h[yo(i):yo(i) + n] = f["c"][o["n"][i]:o["n"][i + 1]]
    z = torch.linalg.solve(K, -h)
    g = torch.from_numpy(np.concatenate([cot["x"][0], cot["u"][0], cot["y"][0]]))
    return (g * z).sum(), z


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_vjp_matches_dense_autograd(name):
    s, host, sol, cot = _case(name)
    ref = lqr_vjp(s, host, sol, cot)
    f = {k: torch.tensor(host[k][0], dtype=torch.float64, requires_grad=True) for k in GRAD_NAMES}
    loss, z = _dense_loss(s, f, cot)
    nx = sol["x"].shape[1]
    assert np.abs(z.detach().numpy()[:nx] - sol["x"][0]).max() < 1e-10  # the same solve
    loss.backward()
    for k in GRAD_NAMES:
        if ref[k].shape[1] == 0:
            continue
        err = rel_err(ref[k], f[k].grad.numpy()[None])[0]
        assert err < 1e-10, (k, err)


def _perturbations(s, host):
    """Central-difference directions: one per entry, Q / R off-diagonal pairs together.
    Yields (name, [flat indices], weight that maps the directional derivative to the entry)."""
    o = offsets(s)
    sd, cd = s.state_dims, s.control_dims
    for name, off, dims in (("Q", o["nn"], sd), ("R", o["mm"], cd)):
        for blk, n in enumerate(dims):
            for j in range(n):
                for i in range(j, n):
                    idx = [off[blk] + i + j * n] + ([off[blk] + j + i * n] if i != j else [])
                    yield name, idx, 1.0 / len(idx)
    for name in ("M", "q", "r", "A", "B", "c", "delta"):
        for k in range(host[name].shape[1]):
            yield name, [k], 1.0


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_vjp_matches_finite_differences(name):
    s, host, sol, cot = _case(name, seed=1)
    ref = lqr_vjp(s, host, sol, cot)
    dirs = list(_perturbations(s, host))
    eps = 1e-6
    # every perturbed problem is one problem of a single oracle batch: +eps rows, then -eps
    batch = {k: np.repeat(host[k], 2 * len(dirs), axis=0) for k in GRAD_NAMES}
    for d, (k, idx, _) in enumerate(dirs):
        for i in idx:
            batch[k][d, i] += eps
            batch[k][len(dirs) + d, i] -= eps
    out = pyoracle.lqr_factor_solve(s, batch, residual=False)
    assert (out["status"] == 0).all()
    L = sum(out[k] @ cot[k][0] for k in ("x", "u", "y"))
    fd = {k: np.zeros_like(host[k]) for k in GRAD_NAMES}
    for d, (k, idx, w) in enumerate(dirs):
        for i in idx:
            fd[k][0, i] = w * (L[d] - L[len(dirs) + d]) / (2 * eps)
    for k in GRAD_NAMES:
        if ref[k].shape[1] == 0:
            continue
        err = rel_err(ref[k], fd[k])[0]
        assert err < 1e-6, (k, err)


def test_failed_problems_get_zero_gradients():
    s, host = pg.lqr_benchmark_batch(2, 1, 2, 3, seed=4, dense_M=True)
    host["delta"][1, 4] = 0.0  # INVALID_DELTA
    sol = pyoracle.lqr_factor_solve(s, host)
    sz = pyoracle.lqr_sizes(s)
    cot = {k: np.ones((3, sz[k])) for k in ("x", "u", "y")}
    ref = lqr_vjp(s, host, sol, cot)
    assert ref["status"].tolist() == [0, 1, 0]
    for k in GRAD_NAMES:
        assert not ref[k][1].any() and ref[k][0].any(), k
