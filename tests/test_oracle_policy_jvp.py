"""The CPU tangent Riccati sweep (policy_jvp_reference.policy_jvp) against torch.func.jvp of a
float64 restatement of the policy, central differences of the numpy policy
(policy_reference.lqr_policy), and the reference adjoint sweep through <cot, JVP(t)> =
<t, VJP(cot)>, on the reference fixtures, a benchmark chain and a random tree."""
import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from oracle import pyoracle
from policy_jvp_reference import policy_jvp
from policy_reference import SIZE_OF, layout, lqr_policy
from policy_vjp_reference import INPUT_NAMES, policy_vjp, torch_policy
from test_gpu_fuzz import random_structure

POLICY = ("K", "k", "V", "v")


def _flat(sp):
    s, p = sp
    return s, fx.pack_problem(**p)


def _random_tree():
    rng = np.random.default_rng(4100)
    s = random_structure(rng)
    return s, pg.variable_tree_batch(s, 3, seed=7)


CASES = {
    "nonuniform_delta_chain": lambda: _flat(fx.nonuniform_delta_chain()),
    "branch_tree": lambda: _flat(fx.branch_tree()),
    "variable_dim_branch_tree": lambda: _flat(fx.variable_dim_branch_tree()),
    "benchmark_chain": lambda: pg.lqr_benchmark_batch(5, 2, 6, 3, seed=3, dense_M=True),
    "variable_dim_chain": lambda: (lambda s: (s, pg.variable_tree_batch(s, 3, seed=4)))(
        pyoracle.Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])),
    "random_tree": _random_tree,
}


def _tan(host, seed, names=INPUT_NAMES):
    """Random tangents; the Q and R blocks are not symmetric."""
    rng = np.random.default_rng(seed)
    return {k: rng.standard_normal(host[k].shape) for k in names}


def _sym_blocks(s, tan):
    """The tangents with every Q and R block replaced by its symmetric part."""
    L = layout(s)
    out = {k: v.copy() for k, v in tan.items()}
    for key, off, dims in (("Q", "nn", L["n"]), ("R", "mm", L["m"])):
        if key not in out:
            continue
        for i, d in enumerate(dims):
            d, o = int(d), int(L[off][i])
            blk = out[key][:, o:o + d * d].reshape(-1, d, d)
            out[key][:, o:o + d * d] = ((blk + blk.transpose(0, 2, 1)) / 2).reshape(-1, d * d)
    return out


def _rel(a, b):
    return np.abs(a - b).max(initial=0.0) / (1.0 + np.abs(b).max(initial=0.0))


@pytest.mark.parametrize("name", sorted(CASES))
def test_sweep_matches_torch_func_jvp(name):
    s, host = CASES[name]()
    tan = _tan(host, 1)
    got = policy_jvp(s, host, tan)
    sym = _sym_blocks(s, tan)

    def f(*a):
        pol = torch_policy(s, dict(zip(INPUT_NAMES, a)))
        return tuple(pol[k] for k in POLICY)

    _, want = torch.func.jvp(f, tuple(torch.tensor(host[k]) for k in INPUT_NAMES),
                             tuple(torch.tensor(sym[k]) for k in INPUT_NAMES))
    for k, w in zip(POLICY, want):
        assert _rel(got[k], w.numpy()) <= 1e-12, (k, _rel(got[k], w.numpy()))


@pytest.mark.parametrize("name", sorted(CASES))
def test_central_differences(name):
    s, host = CASES[name]()
    direction = _sym_blocks(s, _tan(host, 2))
    direction["delta"] *= 1e-2 * np.abs(host["delta"])  # stay inside delta > 0
    got = policy_jvp(s, host, direction)
    eps = 1e-5
    plus = lqr_policy(s, {k: host[k] + eps * direction[k] for k in INPUT_NAMES})
    minus = lqr_policy(s, {k: host[k] - eps * direction[k] for k in INPUT_NAMES})
    for k in POLICY:
        fd = (plus[k] - minus[k]) / (2 * eps)
        assert np.abs(got[k] - fd).max() <= 1e-6 * (1.0 + np.abs(fd).max()), k


@pytest.mark.parametrize("name", sorted(CASES))
def test_adjoint_identity(name):
    s, host = CASES[name]()
    batch = host["q"].shape[0]
    tan = _tan(host, 3)  # non-symmetric Q, R blocks and a tangent of the root's c, delta
    sz = pyoracle.lqr_sizes(s)
    rng = np.random.default_rng(4)
    cot = {k: rng.standard_normal((batch, sz[SIZE_OF[k]])) for k in POLICY}
    jvp = policy_jvp(s, host, tan)
    vjp = policy_vjp(s, host, cot)
    lhs = sum((cot[k] * jvp[k]).sum(1) for k in POLICY)
    rhs = sum((tan[k] * vjp[k]).sum(1) for k in INPUT_NAMES)
    assert np.abs(lhs - rhs).max() <= 1e-12 * np.abs(lhs).max(), (lhs, rhs)


@pytest.mark.parametrize("name", sorted(CASES))
def test_K_and_V_do_not_depend_on_qrc(name):
    s, host = CASES[name]()
    got = policy_jvp(s, host, _tan(host, 5, names=("q", "r", "c")))
    assert not got["K"].any() and not got["V"].any()
    assert got["k"].any() and got["v"].any()


@pytest.mark.parametrize("name", sorted(CASES))
def test_dV_exactly_symmetric(name):
    s, host = CASES[name]()
    got = policy_jvp(s, host, _tan(host, 6))
    L = layout(s)
    for i, d in enumerate(L["n"]):
        d, o = int(d), int(L["nn"][i])
        blk = got["V"][:, o:o + d * d].reshape(-1, d, d)
        assert np.array_equal(blk, blk.transpose(0, 2, 1)), i


def test_root_c_and_delta_are_not_read():
    s, host = CASES["branch_tree"]()
    tan = _tan(host, 7)
    base = policy_jvp(s, host, tan)
    L = layout(s)
    o, n = int(L["nv"][s.root]), int(L["n"][s.root])
    for k in ("c", "delta"):
        tan[k][:, o:o + n] = 1e3
    moved = policy_jvp(s, host, tan)
    for k in POLICY:
        assert np.array_equal(base[k], moved[k]), k
