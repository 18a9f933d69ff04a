"""The CPU reference of the LQR feedback policy (policy_reference.py) against the oracle's
solve: the policy reproduces the solution (u_e = k_e + K_e x_p, y_i = v_i + V_i x_i), V is
symmetric, K and V do not depend on (q, r, c), and V is the matrix that n + 1 solves with
different (q, r, c) recover from their solutions."""
import numpy as np
import pytest

import problem_gen as pg
import reference_fixtures as fx
from oracle import pyoracle
from policy_reference import layout, lqr_policy, policy_residuals


def _flat(sp):
    s, p = sp
    return s, fx.pack_problem(**p)


CASES = {
    "nonuniform_delta_chain": lambda: _flat(fx.nonuniform_delta_chain()),
    "branch_tree": lambda: _flat(fx.branch_tree()),
    "variable_dim_branch_tree": lambda: _flat(fx.variable_dim_branch_tree()),
    "five_node_tree": lambda: _flat(fx.five_node_tree()),
    "benchmark_chain": lambda: pg.lqr_benchmark_batch(4, 2, 6, 3, seed=3, dense_M=True),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_policy_reproduces_the_solution(name):
    s, host = CASES[name]()
    sol = pyoracle.lqr_factor_solve(s, host)
    assert (sol["status"] == 0).all()
    pol = lqr_policy(s, host)
    ru, ry = policy_residuals(s, host, pol, sol["x"], sol["u"], sol["y"])
    assert ru.max() <= 1e-12 and ry.max() <= 1e-12, (ru.max(), ry.max())


@pytest.mark.parametrize("name", sorted(CASES))
def test_V_symmetric_and_independent_of_qrc(name):
    s, host = CASES[name]()
    pol = lqr_policy(s, host)
    L = layout(s)
    for i in range(s.num_edges + 1):
        n = int(L["n"][i])
        Vi = pol["V"][:, L["nn"][i]:L["nn"][i] + n * n].reshape(-1, n, n)
        scale = 1.0 + np.abs(Vi).max()
        assert np.abs(Vi - Vi.transpose(0, 2, 1)).max() <= 1e-13 * scale
    rng = np.random.default_rng(5)
    other = dict(host)
    for k in ("q", "r", "c"):
        other[k] = rng.standard_normal(host[k].shape)
    pol2 = lqr_policy(s, other)
    np.testing.assert_array_equal(pol2["K"], pol["K"])
    np.testing.assert_array_equal(pol2["V"], pol["V"])


@pytest.mark.parametrize("name", ["nonuniform_delta_chain", "variable_dim_branch_tree",
                                  "benchmark_chain"])
def test_V_from_solves(name):
    # y_i - v_i = V_i x_i for every (q, r, c): n_i + 1 solves with random (q, r, c) whose x_i
    # span R^{n_i} determine V_i
    s, host = CASES[name]()
    host = {k: v[:1] for k, v in host.items()}
    L = layout(s)
    nmax = int(L["n"].max())
    rng = np.random.default_rng(11)
    xs, ys, vs = [], [], []
    for _ in range(nmax + 1):
        h = dict(host)
        for k in ("q", "r", "c"):
            h[k] = rng.standard_normal(host[k].shape)
        sol = pyoracle.lqr_factor_solve(s, h)
        assert (sol["status"] == 0).all()
        xs.append(sol["x"][0])
        ys.append(sol["y"][0])
        vs.append(lqr_policy(s, h)["v"][0])
    X, Y, Vv = np.array(xs), np.array(ys), np.array(vs)
    pol = lqr_policy(s, host)
    for i in range(s.num_edges + 1):
        n, o = int(L["n"][i]), int(L["nv"][i])
        if n == 0:
            continue
        Xi = X[:, o:o + n]
        Ri = Y[:, o:o + n] - Vv[:, o:o + n]
        Vrec = np.linalg.lstsq(Xi, Ri, rcond=None)[0].T  # Ri = Xi Vi'
        Vi = pol["V"][0, L["nn"][i]:L["nn"][i] + n * n].reshape(n, n).T
        assert np.abs(Vrec - Vi).max() <= 1e-8 * (1.0 + np.abs(Vi).max()), i
