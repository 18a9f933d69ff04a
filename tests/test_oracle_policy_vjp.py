"""The CPU adjoint Riccati sweep (policy_vjp_reference.policy_vjp) against torch.autograd on a
float64 restatement of the policy, and both against central differences of the numpy policy
(policy_reference.lqr_policy), on the reference fixtures and a benchmark chain."""
import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from oracle import pyoracle
from policy_reference import SIZE_OF, layout, lqr_policy
from policy_vjp_reference import INPUT_NAMES, autograd_policy_vjp, policy_vjp, torch_policy


def _flat(sp):
    s, p = sp
    return s, fx.pack_problem(**p)


CASES = {
    "nonuniform_delta_chain": lambda: _flat(fx.nonuniform_delta_chain()),
    "branch_tree": lambda: _flat(fx.branch_tree()),
    "variable_dim_branch_tree": lambda: _flat(fx.variable_dim_branch_tree()),
    "benchmark_chain": lambda: pg.lqr_benchmark_batch(5, 2, 6, 3, seed=3, dense_M=True),
}


def _cot(s, batch, seed, names=("K", "k", "V", "v")):
    """Random cotangents; V's blocks are not symmetric."""
    rng = np.random.default_rng(seed)
    sz = pyoracle.lqr_sizes(s)
    return {k: rng.standard_normal((batch, sz[SIZE_OF[k]])) for k in names}


def _rel(a, b):
    return np.abs(a - b).max(initial=0.0) / (1.0 + np.abs(b).max(initial=0.0))


@pytest.mark.parametrize("name", sorted(CASES))
def test_torch_forward_matches_reference(name):
    s, host = CASES[name]()
    ref = lqr_policy(s, host)
    got = torch_policy(s, {k: torch.tensor(host[k], dtype=torch.float64) for k in INPUT_NAMES})
    for k in ref:
        assert _rel(got[k].numpy(), ref[k]) <= 1e-13, k


@pytest.mark.parametrize("name", sorted(CASES))
def test_sweep_matches_autograd(name):
    s, host = CASES[name]()
    cot = _cot(s, host["q"].shape[0], 1)
    got = policy_vjp(s, host, cot)
    want = autograd_policy_vjp(s, host, cot)
    for k in INPUT_NAMES:
        assert _rel(got[k], want[k]) <= 1e-12, (k, _rel(got[k], want[k]))


@pytest.mark.parametrize("name", sorted(CASES))
def test_central_differences(name):
    s, host = CASES[name]()
    batch = host["q"].shape[0]
    cot = _cot(s, batch, 2)
    grads = policy_vjp(s, host, cot)
    auto = autograd_policy_vjp(s, host, cot)
    rng = np.random.default_rng(3)
    L = layout(s)
    direction = {k: rng.standard_normal(host[k].shape) for k in INPUT_NAMES}
    for key, off, dims in (("Q", "nn", L["n"]), ("R", "mm", L["m"])):  # symmetric directions
        for i, d in enumerate(dims):
            d = int(d)
            o = int(L[off][i])
            blk = direction[key][:, o:o + d * d].reshape(-1, d, d)
            direction[key][:, o:o + d * d] = (blk + blk.transpose(0, 2, 1)).reshape(-1, d * d) / 2
    direction["delta"] *= 1e-2 * np.abs(host["delta"])  # stay inside delta > 0

    def loss(t):
        pol = lqr_policy(s, {k: host[k] + t * direction[k] for k in INPUT_NAMES})
        return sum((cot[k] * pol[k]).sum(1) for k in cot)

    eps = 1e-5
    fd = (loss(eps) - loss(-eps)) / (2 * eps)
    for g in (grads, auto):
        dot = sum((g[k] * direction[k]).sum(1) for k in INPUT_NAMES)
        assert np.abs(dot - fd).max() <= 1e-6 * (1.0 + np.abs(fd).max()), (dot, fd)


@pytest.mark.parametrize("name", sorted(CASES))
def test_K_and_V_do_not_depend_on_qrc(name):
    s, host = CASES[name]()
    g = policy_vjp(s, host, _cot(s, host["q"].shape[0], 4, names=("K", "V")))
    for k in ("q", "r", "c"):
        assert not g[k].any(), k
    assert g["Q"].any() and g["A"].any()


@pytest.mark.parametrize("name", sorted(CASES))
def test_root_c_and_delta_get_zero(name):
    s, host = CASES[name]()
    g = policy_vjp(s, host, _cot(s, host["q"].shape[0], 5))
    L = layout(s)
    o, n = int(L["nv"][s.root]), int(L["n"][s.root])
    assert not g["c"][:, o:o + n].any()
    assert not g["delta"][:, o:o + n].any()
