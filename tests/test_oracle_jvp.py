"""The CPU reference of the LQR and Newton-KKT JVPs (jvp_reference.py: the tangent right-hand
side of include/sipoc.h, then the oracle's own solve) against:
- torch.func.jvp through a dense torch.linalg.solve of the assembled system (the dense K of
  the VJP tests, symmetric blocks formed as (P + P^T) / 2), 1e-10;
- central finite differences of the oracle's solve along the tangent, 1e-6 relative;
- the reference VJPs through the adjoint identity <JVP(t), g> = <t, VJP(g)>, 1e-12 relative,
  with NON-symmetric tangents on the symmetric blocks: the identity pins the convention that
  those blocks enter through their symmetric parts."""
import numpy as np
import pytest
import torch

import test_oracle_kkt_vjp as okv
import test_oracle_vjp as ov
from jvp_reference import kkt_jvp, lqr_jvp
from kkt_vjp_reference import SYMMETRIC, block_table, kkt_solve, kkt_vjp
from oracle import pyoracle
from vjp_reference import GRAD_NAMES, lqr_vjp, offsets

LQR_CASES = list(ov.CASES)
KKT_CASES = list(okv.CASES)


def _tangents(arrays: dict, names, seed):
    rng = np.random.default_rng(seed)
    return {k: rng.standard_normal(arrays[k].shape) for k in names}


def _symmetrized(tan: dict, blocks: dict):
    """The tangents with every symmetric block replaced by its symmetric part; blocks: name ->
    [(offset, n)]."""
    out = {k: v.copy() for k, v in tan.items()}
    for k, bl in blocks.items():
        for off, n in bl:
            if n == 0:
                continue
            B = out[k][:, off:off + n * n].reshape(-1, n, n)
            out[k][:, off:off + n * n] = (0.5 * (B + B.swapaxes(1, 2))).reshape(-1, n * n)
    return out


def _lqr_sym_blocks(s):
    o = offsets(s)
    return {"Q": [(o["nn"][i], int(n)) for i, n in enumerate(s.state_dims)],
            "R": [(o["mm"][e], int(m)) for e, m in enumerate(s.control_dims)]}


def _kkt_sym_blocks(s, p):
    out = {}
    for name, blocks in block_table(s, p).items():
        if name in SYMMETRIC:
            offs = np.cumsum([0] + [int(nr) * int(nc) for _, nr, _, nc in blocks])
            out[name] = [(int(offs[j]), int(b[1])) for j, b in enumerate(blocks)]
    return out


def _lqr_flat(ref):
    return np.concatenate([ref["x"][0], ref["u"][0], ref["y"][0]])


# ---- LQR -----------------------------------------------------------------------------------

@pytest.mark.parametrize("name", LQR_CASES)
def test_lqr_reference_jvp_matches_torch_func_jvp(name):
    s, host, sol, _ = ov._case(name)
    tan = _tangents(host, GRAD_NAMES, 11)
    ref = lqr_jvp(s, host, sol, tan)
    cot0 = {k: np.zeros_like(sol[k]) for k in ("x", "u", "y")}
    prim = tuple(torch.tensor(host[k][0], dtype=torch.float64) for k in GRAD_NAMES)
    tans = tuple(torch.tensor(tan[k][0], dtype=torch.float64) for k in GRAD_NAMES)
    z_of = lambda *a: ov._dense_loss(s, dict(zip(GRAD_NAMES, a)), cot0)[1]
    _, dz = torch.func.jvp(z_of, prim, tans)
    dz = dz.numpy()
    err = np.abs(_lqr_flat(ref) - dz).max() / max(1.0, np.abs(dz).max())
    assert err < 1e-10, err


@pytest.mark.parametrize("name", LQR_CASES)
def test_lqr_reference_jvp_matches_finite_differences(name):
    s, host, sol, _ = ov._case(name)
    tan = _tangents(host, GRAD_NAMES, 12)
    ref = lqr_jvp(s, host, sol, tan)
    # the oracle reads the lower triangles of Q, R: step along the symmetric parts
    step = _symmetrized(tan, _lqr_sym_blocks(s))
    eps = 1e-6
    batch = {k: np.concatenate([host[k] + eps * step[k], host[k] - eps * step[k]])
             for k in GRAD_NAMES}
    out = pyoracle.lqr_factor_solve(s, batch, residual=False)
    assert (out["status"] == 0).all()
    fd = np.concatenate([(out[k][0] - out[k][1]) / (2 * eps) for k in ("x", "u", "y")])
    err = np.abs(_lqr_flat(ref) - fd).max() / max(1.0, np.abs(fd).max())
    assert err < 1e-6, err


@pytest.mark.parametrize("name", LQR_CASES)
def test_lqr_adjoint_identity(name):
    s, host, sol, cot = ov._case(name, seed=2)
    tan = _tangents(host, GRAD_NAMES, 13)  # Q, R tangents not symmetric
    fwd = lqr_jvp(s, host, sol, tan)
    rev = lqr_vjp(s, host, sol, cot)
    lhs = sum(float(fwd[k][0] @ cot[k][0]) for k in ("x", "u", "y"))
    terms = [tan[k][0] * rev[k][0] for k in GRAD_NAMES]
    rhs = sum(float(t.sum()) for t in terms)
    scale = max(abs(lhs), sum(float(np.abs(t).sum()) for t in terms))
    assert abs(lhs - rhs) <= 1e-12 * scale, (lhs, rhs)


def test_lqr_failed_problems_get_zero_tangents():
    import problem_gen as pg
    s, host = pg.lqr_benchmark_batch(2, 1, 2, 3, seed=4, dense_M=True)
    host["delta"][1, 4] = 0.0  # INVALID_DELTA
    sol = pyoracle.lqr_factor_solve(s, host)
    ref = lqr_jvp(s, host, sol, _tangents(host, GRAD_NAMES, 5))
    assert ref["status"].tolist() == [0, 1, 0]
    for k in ("x", "u", "y"):
        assert not ref[k][1].any() and ref[k][0].any(), k


# ---- Newton-KKT ----------------------------------------------------------------------------

def _kkt(name, seed=0):
    s, p, arrays, sol, cot = okv._case(name, seed)
    names = okv._names(p)
    model, theta = okv._split(s, p, arrays)
    return s, p, arrays, names, model, theta, sol, cot


def _kkt_ref(s, p, arrays, model, theta, sol, tan):
    return kkt_jvp(s, p, model, theta, arrays["w"], arrays["r1"], arrays["r2"], arrays["r3"],
                   sol, tan)


@pytest.mark.parametrize("name", KKT_CASES)
def test_kkt_reference_jvp_matches_torch_func_jvp(name):
    s, p, arrays, names, model, theta, sol, _ = _kkt(name)
    tan = _tangents(arrays, names, 21)
    ref = _kkt_ref(s, p, arrays, model, theta, sol, tan)
    prim = tuple(torch.tensor(arrays[k][0], dtype=torch.float64) for k in names)
    tans = tuple(torch.tensor(tan[k][0], dtype=torch.float64) for k in names)

    def z_of(*a):
        f = dict(zip(names, a))
        return torch.linalg.solve(okv.dense_K(s, p, f), f["b"])

    _, dz = torch.func.jvp(z_of, prim, tans)
    dz = dz.numpy()
    err = np.abs(ref["sol"][0] - dz).max() / max(1.0, np.abs(dz).max())
    assert err < 1e-10, err


@pytest.mark.parametrize("name", KKT_CASES)
def test_kkt_reference_jvp_matches_finite_differences(name):
    s, p, arrays, names, model, theta, sol, _ = _kkt(name)
    tan = _tangents(arrays, names, 22)
    ref = _kkt_ref(s, p, arrays, model, theta, sol, tan)
    step = _symmetrized(tan, _kkt_sym_blocks(s, p))
    eps = 1e-6
    batch = {k: np.concatenate([arrays[k] + eps * step[k], arrays[k] - eps * step[k]])
             for k in names}
    bm, bt = okv._split(s, p, batch)
    out = kkt_solve(s, p, bm, bt, batch["w"], batch["r1"], batch["r2"], batch["r3"], batch["b"])
    assert (out["ok"] == 1).all()
    fd = (out["sol"][0] - out["sol"][1]) / (2 * eps)
    err = np.abs(ref["sol"][0] - fd).max() / max(1.0, np.abs(fd).max())
    assert err < 1e-6, err


@pytest.mark.parametrize("name", KKT_CASES)
def test_kkt_adjoint_identity(name):
    s, p, arrays, names, model, theta, sol, cot = _kkt(name, seed=2)
    tan = _tangents(arrays, names, 23)  # Hessian tangents not symmetric
    fwd = _kkt_ref(s, p, arrays, model, theta, sol, tan)
    rev = kkt_vjp(s, p, model, theta, arrays["w"], arrays["r1"], arrays["r2"], arrays["r3"],
                  sol, cot)
    lhs = float(fwd["sol"][0] @ cot[0])
    terms = [tan[k][0] * rev[k][0] for k in names]
    rhs = sum(float(t.sum()) for t in terms)
    scale = max(abs(lhs), sum(float(np.abs(t).sum()) for t in terms))
    assert abs(lhs - rhs) <= 1e-12 * scale, (lhs, rhs)

