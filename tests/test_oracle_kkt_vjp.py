"""The CPU reference of the Newton-KKT VJP (kkt_vjp_reference.py: the oracle's solve with the
cotangent as right-hand side, then the gradient table of include/sipoc.h) against:
- the block table itself: K assembled densely from it reproduces the oracle's operator
  (kkt_apply / kkt_theta_apply) on random vectors, 1e-12;
- torch.autograd through a dense torch.linalg.solve of that K (symmetric Hessian blocks formed
  as (P + P^T) / 2, so dL/dP is the symmetric gradient), 1e-10;
- central finite differences of the oracle's own solve (symmetric perturbations of the
  Hessian blocks), 1e-6 relative."""
import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import rel_err
from kkt_vjp_reference import (MODEL_NAMES, SYMMETRIC, THETA_NAMES, VECTOR_NAMES, block_table,
                               kkt_solve, kkt_vjp, layout)
from oracle import pyoracle
from oracle.pyoracle import Structure

REG_NAMES = ("w", "r1", "r2", "r3")


def _fixture(build):
    s = build()
    sz = pyoracle.kkt_sizes(s)
    w, r1, r2, r3, _ = fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"])
    return s, 0, fx.kkt_model(s), None, dict(w=w, r1=r1, r2=r2, r3=r3)


def _schur():
    s, p, diag = fx.kkt_case_schur()
    sz = pyoracle.kkt_sizes(s)
    w, r1, r2, r3, _ = fx.kkt_regularization(sz["x_dim"] + p, sz["y_dim"], sz["z_dim"])
    return s, p, fx.kkt_model(s), fx.kkt_theta_model(s, p, diag), dict(w=w, r1=r1, r2=r2, r3=r3)


def _newton_chain():
    s = Structure.chain(3, 3, 2, node_c=[0, 0, 0, 2], node_g=[0, 0, 0, 2], edge_c=[1, 1, 1],
                        edge_g=[2, 2, 2])
    model, w, r1, r2, r3, _ = pg.newton_kkt_batch(s, 1, seed=17, r2_max=1e3)
    return s, 0, model, None, dict(w=w, r1=r1, r2=r2, r3=r3)


CASES = {
    "chain": lambda: _fixture(fx.kkt_case_chain),
    "siblings": lambda: _fixture(fx.kkt_case_siblings),
    "zero_dim_root": lambda: _fixture(fx.kkt_case_zero_dim_root),
    "schur": _schur,
    "newton_chain": _newton_chain,
}


def _case(name, seed=0):
    s, p, model, theta, reg = CASES[name]()
    kd = layout(s, p)["kkt_dim"]
    rng = np.random.default_rng(seed)
    b, cot = rng.standard_normal((1, kd)), rng.standard_normal((1, kd))
    out = kkt_solve(s, p, model, theta, reg["w"], reg["r1"], reg["r2"], reg["r3"], b)
    assert out["ok"].tolist() == [1]
    arrays = {**model, **(theta or {}), **reg, "b": b}
    return s, p, arrays, out["sol"], cot


def _split(s, p, arrays):
    model = {k: arrays[k] for k in MODEL_NAMES}
    theta = {k: arrays[k] for k in THETA_NAMES} if p else None
    return model, theta


def _names(p):
    return MODEL_NAMES + (THETA_NAMES if p else ()) + VECTOR_NAMES


def dense_K(s, p, f):
    """K of one problem from the block table; f: name -> 1-D torch array."""
    L = layout(s, p)
    kd = L["kkt_dim"]
    K = torch.zeros(kd, kd, dtype=torch.float64)
    for name, blocks in block_table(s, p).items():
        off = 0
        for r0, nr, c0, nc in blocks:
            r0, nr, c0, nc = int(r0), int(nr), int(c0), int(nc)
            B = f[name][off:off + nr * nc].reshape(nc, nr).T  # column-major block
            off += nr * nc
            if name in SYMMETRIC:
                K[r0:r0 + nr, c0:c0 + nc] += 0.5 * (B + B.T)
            else:
                K[r0:r0 + nr, c0:c0 + nc] += B
                K[c0:c0 + nc, r0:r0 + nr] += B.T
    for i, n in enumerate(int(v) for v in s.state_dims):  # the -I of every dynamics row
        ys, xs = int(L["y_dyn"][i]), int(L["x_state"][i])
        eye = torch.eye(n, dtype=torch.float64)
        K[ys:ys + n, xs:xs + n] -= eye
        K[xs:xs + n, ys:ys + n] -= eye
    reg = torch.cat([f["r1"], -f["r2"], -(f["w"] + f["r3"])])
    return K + torch.diag(reg)


def _oracle_apply(s, p, arrays, x):
    model, theta = _split(s, p, arrays)
    reg = [arrays[k] for k in REG_NAMES]
    if p:
        return pyoracle.kkt_theta_apply(s, p, model, theta, *reg, x)
    return pyoracle.kkt_apply(s, model, *reg, x)


@pytest.mark.parametrize("name", list(CASES))
def test_block_table_assembles_the_oracle_operator(name):
    s, p, arrays, sol, _ = _case(name)
    K = dense_K(s, p, {k: torch.from_numpy(v[0]) for k, v in arrays.items()}).numpy()
    assert np.abs(K - K.T).max() == 0.0
    x = np.random.default_rng(3).standard_normal((4, K.shape[0]))
    ref = _oracle_apply(s, p, {k: np.repeat(v, 4, axis=0) for k, v in arrays.items()}, x)
    assert np.abs(x @ K.T - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("name", list(CASES))
def test_reference_vjp_matches_dense_autograd(name):
    s, p, arrays, sol, cot = _case(name)
    model, theta = _split(s, p, arrays)
    ref = kkt_vjp(s, p, model, theta, arrays["w"], arrays["r1"], arrays["r2"], arrays["r3"],
                  sol, cot)
    f = {k: torch.tensor(arrays[k][0], dtype=torch.float64, requires_grad=True)
         for k in _names(p)}
    K = dense_K(s, p, f)
    z = torch.linalg.solve(K, f["b"])
    assert np.abs(z.detach().numpy() - sol[0]).max() < 1e-10 * np.abs(sol).max()  # same solve
    (torch.from_numpy(cot[0]) * z).sum().backward()
    for k in _names(p):
        if ref[k].shape[1] == 0:
            continue
        err = rel_err(ref[k], f[k].grad.numpy()[None])[0]
        assert err < 1e-10, (k, err)


def _perturbations(s, p, arrays):
    """Central-difference directions: one per entry, symmetric off-diagonal pairs together.
    Yields (name, [flat indices], weight that maps the directional derivative to the entry)."""
    table = block_table(s, p)
    for name in _names(p):
        if name in SYMMETRIC:
            off = 0
            for _, n, _, _ in table[name]:
                n = int(n)
                for j in range(n):
                    for i in range(j, n):
                        idx = [off + i + j * n] + ([off + j + i * n] if i != j else [])
                        yield name, idx, 1.0 / len(idx)
                off += n * n
        else:
            for k in range(arrays[name].shape[1]):
                yield name, [k], 1.0


@pytest.mark.parametrize("name", list(CASES))
def test_reference_vjp_matches_finite_differences(name):
    s, p, arrays, sol, cot = _case(name, seed=1)
    model, theta = _split(s, p, arrays)
    ref = kkt_vjp(s, p, model, theta, arrays["w"], arrays["r1"], arrays["r2"], arrays["r3"],
                  sol, cot)
    dirs = list(_perturbations(s, p, arrays))
    eps = 1e-6
    # every perturbed problem is one problem of a single oracle batch: +eps rows, then -eps
    batch = {k: np.repeat(arrays[k], 2 * len(dirs), axis=0) for k in _names(p)}
    for d, (k, idx, _) in enumerate(dirs):
        for i in idx:
            batch[k][d, i] += eps
            batch[k][len(dirs) + d, i] -= eps
    bm, bt = _split(s, p, batch)
    out = kkt_solve(s, p, bm, bt, batch["w"], batch["r1"], batch["r2"], batch["r3"], batch["b"])
    assert (out["ok"] == 1).all()
    L = out["sol"] @ cot[0]
    fd = {k: np.zeros_like(arrays[k]) for k in _names(p)}
    for d, (k, idx, wgt) in enumerate(dirs):
        for i in idx:
            fd[k][0, i] = wgt * (L[d] - L[len(dirs) + d]) / (2 * eps)
    for k in _names(p):
        if ref[k].shape[1] == 0:
            continue
        err = rel_err(ref[k], fd[k])[0]
        assert err < 1e-6, (k, err)


def test_failed_problems_get_zero_gradients():
    s = fx.kkt_case_chain()
    sz = pyoracle.kkt_sizes(s)
    model = {k: np.repeat(v, 3, axis=0) for k, v in fx.kkt_model(s).items()}
    w, r1, r2, r3, rhs = (np.repeat(a, 3, axis=0) for a in
                          fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"]))
    r2[1, 2] = 0.0  # non-positive r2: the factor rejects the problem
    sol = kkt_solve(s, 0, model, None, w, r1, r2, r3, rhs)
    ref = kkt_vjp(s, 0, model, None, w, r1, r2, r3, sol["sol"], np.ones_like(rhs))
    assert ref["ok"].tolist() == [1, 0, 1]
    for k in _names(0):
        if ref[k].shape[1]:
            assert not ref[k][1].any() and ref[k][0].any(), k
