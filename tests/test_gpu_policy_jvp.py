"""sipoc_lqr_policy_jvp (the forward-mode derivative of the feedback policy K, k, V, v) against
the CPU tangent sweep (policy_jvp_reference.py) on every plan family and structure, plus its
contract: the kernel each structure runs, NULL tangents bitwise equal to zero ones, NULL outputs
untouched, zeros in failed problems and padding lanes, bitwise repeatable (eager and graph
replay), the adjoint identity against the device sipoc_lqr_policy_vjp, a directional finite
difference of the device policy, and the torch binding autograd.factor_solve_policy_fwd.

Tolerance, as in test_gpu_policy_vjp.py: REL_TOL (1e-9 relative per problem and array) on k, v;
2 * REL_TOL on K, V.  After a parallel-in-time forward, 1e-8."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from oracle.pyoracle import Structure
from policy_jvp_reference import policy_jvp
from policy_reference import POLICY_NAMES, SIZE_OF
from policy_vjp_reference import INPUT_NAMES
from sip_optimal_control_b200 import LQR, autograd
from sip_optimal_control_b200 import _capi
from sip_optimal_control_b200._capi import lib
from test_gpu_fuzz import random_structure

pytestmark = pytest.mark.gpu

CHAIN_SHAPES = [(n, m) for n in (4, 6, 8) for m in (1, 2, 3, 4)] + [(12, 4)]
SUB = "policy_jvp_subwarp"
GEN = "policy_jvp_generic_kernel"


def _tol(k, tol=REL_TOL):
    return 2 * tol if k in ("K", "V") else tol


def _tan(host, seed, names=INPUT_NAMES):
    rng = np.random.default_rng(seed)
    return {k: rng.standard_normal(host[k].shape) for k in names}


def _launches(e):
    launches = {}
    for i in range(lib.sipoc_profile_collect(e._handle)):
        nm, cnt = ctypes.c_char_p(), ctypes.c_int64()
        e._check(lib.sipoc_profile_get(e._handle, i, ctypes.byref(nm), None, ctypes.byref(cnt)))
        launches[nm.value.decode()] = cnt.value
    return launches


def _forward(s, host, **kw):
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, host["q"].shape[0], **kw)
    inp = lqr.pack_input(host)
    pol = lqr.factor_solve_policy(inp, lqr.alloc_output())
    return lqr, inp, pol


def _check(s, host, kernel=None, tol=REL_TOL, seed=1, **kw):
    assert (pyoracle.lqr_factor_solve(s, host)["status"] == 0).all()
    tan = _tan(host, seed)
    ref = policy_jvp(s, host, tan)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    lib.sipoc_profile_enable(e._handle, 1)
    _launches(e)
    dtan = {k: e.pack(v) for k, v in tan.items()}
    before = e.launch_count
    res = lqr.policy_jvp(inp, pol, pol["status"], dtan)
    assert e.launch_count - before == 1
    launches = {k: v for k, v in _launches(e).items() if k.startswith("policy_jvp")}
    lib.sipoc_profile_enable(e._handle, 0)
    if kernel is not None:
        assert launches == {kernel: 1}, launches
    for k in POLICY_NAMES:
        got = e.unpack(res[k], e.lqr_sizes[SIZE_OF[k]])
        if got.shape[1]:
            err = rel_err(got, ref[k]).max()
            assert err <= _tol(k, tol), (k, float(err), e.kernel_variant)
    return lqr


@pytest.mark.parametrize("n,m", CHAIN_SHAPES)
def test_chain_shapes(n, m):
    s, host = pg.lqr_benchmark_batch(n, m, 7, 37, seed=n * 10 + m, dense_M=True)
    _check(s, host, SUB)


@pytest.mark.parametrize("n,m,T", [(16, 4, 5), (32, 8, 3), (64, 24, 2), (5, 4, 6), (10, 3, 4)])
def test_generic_kernel_shapes(n, m, T):
    s, host = pg.lqr_benchmark_batch(n, m, T, 33, seed=n + T, dense_M=True)
    _check(s, host, GEN)


@pytest.mark.parametrize("seed", range(6))
def test_random_trees(seed):
    rng = np.random.default_rng(5000 + seed)
    s = random_structure(rng)
    host = pg.variable_tree_batch(s, int(rng.integers(1, 71)), seed=seed)
    for force_generic in (False, True):
        _check(s, host, seed=seed, force_generic=force_generic)


@pytest.mark.parametrize("builder", [fx.five_node_tree, fx.variable_dim_branch_tree,
                                     fx.nonuniform_delta_chain])
def test_reference_fixtures(builder):
    s, p = builder()
    _check(s, {k: np.repeat(v, 5, axis=0) for k, v in fx.pack_problem(**p).items()})


@pytest.mark.parametrize("kw,tol", [
    ({}, REL_TOL),
    (dict(force_generic=True), REL_TOL),
    (dict(parallel_in_time=True), 1e-8),
])
def test_forward_plan_families(kw, tol):
    # the JVP depends on the structure only; the forward's plan changes V, v by rounding
    s, host = pg.lqr_benchmark_batch(12, 4, 64 if kw.get("parallel_in_time") else 12, 19,
                                     seed=21, dense_M=True)
    lqr = _check(s, host, SUB, tol=tol, **kw)
    if kw:
        assert ("generic" if "force_generic" in kw else "scan_") in lqr.engine.kernel_variant


@pytest.mark.parametrize("pad_variable_dims", [False, True])
def test_padded_and_strict_forwards(pad_variable_dims):
    s = Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])
    host = pg.variable_tree_batch(s, 40, seed=4)
    lqr = _check(s, host, GEN, pad_variable_dims=pad_variable_dims)
    assert "padded_to_" in lqr.engine.kernel_variant


def test_strict_forward():
    # (5, 4) is not a fast-plan shape: the forward runs the strict plan, the JVP the generic kernel
    s, host = pg.lqr_benchmark_batch(5, 4, 4, 21, seed=31, dense_M=True)
    _check(s, host, GEN)


@pytest.mark.parametrize("batch", [1, 31, 33, 97])
@pytest.mark.parametrize("n,m", [(6, 2), (12, 4)])
def test_ragged_batches(batch, n, m):
    s, host = pg.lqr_benchmark_batch(n, m, 5, batch, seed=batch, dense_M=True)
    _check(s, host, SUB)


def test_large_batch_sample():
    n, m, T, batch = 12, 4, 3, 41000
    s = Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    inp = lqr.generate_benchmark(seed=5)
    pol = lqr.factor_solve_policy(inp, lqr.alloc_output())
    assert (pol["status"][:batch] == 0).all()
    rng = np.random.default_rng(8)
    tan = {k: torch.from_numpy(rng.standard_normal(tuple(inp[k].shape))).to(inp[k].device)
           for k in INPUT_NAMES}
    res = lqr.policy_jvp(inp, pol, pol["status"], tan)
    torch.cuda.synchronize()
    idx = torch.from_numpy(rng.choice(batch, 48, replace=False)).to(e.torch_device())
    sample = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: sample(inp[k], e.lqr_sizes[k]) for k in INPUT_NAMES}
    ref = policy_jvp(s, host, {k: sample(tan[k], e.lqr_sizes[k]) for k in INPUT_NAMES})
    for k in POLICY_NAMES:
        err = rel_err(sample(res[k], e.lqr_sizes[SIZE_OF[k]]), ref[k]).max()
        assert err <= _tol(k), (k, float(err))


def _call(lqr, inp, pol, status, tan, out, stream=None):
    e = lqr.engine
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in INPUT_NAMES])
    st = _capi.LqrInput(*[tan[k].data_ptr() if tan.get(k) is not None else None
                          for k in INPUT_NAMES])
    so = _capi.LqrPolicy(*[out[k].data_ptr() if k in out else None for k in POLICY_NAMES])
    e._check(lib.sipoc_lqr_policy_jvp(e._handle, ctypes.byref(si), pol["V"].data_ptr(),
                                      pol["v"].data_ptr(), status.data_ptr(), ctypes.byref(st),
                                      ctypes.byref(so), e.stream_ptr(stream)))


def _outs(e):
    return {k: e.empty(e.lqr_sizes[SIZE_OF[k]]) for k in POLICY_NAMES}


def _rand_like(rng, inp, names):
    return {k: torch.from_numpy(rng.standard_normal(tuple(inp[k].shape))).to(inp[k].device)
            for k in names}


@pytest.mark.parametrize("n,m,kw", [(12, 4, {}), (5, 2, {}), (12, 4, dict(force_generic=True))])
def test_null_tangents_and_null_outputs(n, m, kw):
    s, host = pg.lqr_benchmark_batch(n, m, 6, 37, seed=3, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    rng = np.random.default_rng(2)
    for keep in (("A",), ("Q", "R", "delta"), ("q", "r", "c"), ("M", "B")):
        tan = _rand_like(rng, inp, keep)
        zeros = dict(tan, **{k: torch.zeros_like(inp[k]) for k in INPUT_NAMES if k not in keep})
        o1, o2 = _outs(e), _outs(e)
        _call(lqr, inp, pol, pol["status"], tan, o1)
        _call(lqr, inp, pol, pol["status"], zeros, o2)
        torch.cuda.synchronize()
        for k in POLICY_NAMES:
            assert torch.equal(o1[k], o2[k]), (keep, k)
        if keep == ("q", "r", "c"):  # K and V do not depend on q, r, c
            assert not o1["K"].any() and not o1["V"].any()
    full = _rand_like(rng, inp, INPUT_NAMES)
    ref = _outs(e)
    _call(lqr, inp, pol, pol["status"], full, ref)
    for want in (("K",), ("k", "v"), ("V",), ("K", "V", "v")):
        o = {k: torch.full_like(ref[k], float("nan")) for k in POLICY_NAMES}
        _call(lqr, inp, pol, pol["status"], full, {k: o[k] for k in want})
        torch.cuda.synchronize()
        for k in POLICY_NAMES:
            if k in want:
                assert torch.equal(o[k], ref[k]), (want, k)
            else:
                assert torch.isnan(o[k]).all(), (want, k)
    before = e.launch_count
    _call(lqr, inp, pol, pol["status"], full, {})  # nothing requested: nothing launched
    assert e.launch_count == before


@pytest.mark.parametrize("n,m,force_generic", [(4, 1, False), (4, 1, True), (12, 4, False)])
def test_failed_problems_and_padding_lanes_are_zero(n, m, force_generic):
    T, batch = 3, 6
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=10, dense_M=True)
    host["delta"][1, T * n + 0] = 0.0
    host["R"][3, (T - 1) * m * m] = -50.0
    ref_status = pyoracle.lqr_factor_solve(s, host)["status"]
    assert ref_status[1] != 0 and ref_status[3] != 0 and (ref_status[[0, 2, 4, 5]] == 0).all()
    good = ref_status == 0
    tan = _tan(host, 6)
    ref = policy_jvp(s, {k: v[good] for k, v in host.items()}, {k: v[good] for k, v in tan.items()})
    lqr, inp, pol = _forward(s, host, force_generic=force_generic)
    e = lqr.engine
    out = {k: torch.full_like(v, float("nan")) for k, v in _outs(e).items()}
    lqr.policy_jvp(inp, pol, pol["status"], {k: e.pack(v) for k, v in tan.items()}, dpolicy=out)
    assert pol["status"][:batch].cpu().numpy().tolist() == ref_status.tolist()
    for k in POLICY_NAMES:
        full = out[k][: e.lqr_sizes[SIZE_OF[k]]].cpu().numpy()
        assert not full[:, batch:].any(), k
        assert not full[:, :batch][:, ~good].any(), k
        assert rel_err(full[:, :batch].T[good], ref[k]).max() <= _tol(k), k


@pytest.mark.parametrize("n,m,kw", [(12, 4, {}), (3, 2, {})])
def test_bitwise_repeatable_and_graph_replay(n, m, kw):
    s, host = pg.lqr_benchmark_batch(n, m, 8, 37, seed=9, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    tan = _rand_like(np.random.default_rng(4), inp, INPUT_NAMES)
    side = torch.cuda.Stream()
    o1, o2 = _outs(e), _outs(e)
    torch.cuda.synchronize()
    _call(lqr, inp, pol, pol["status"], tan, o1, stream=side)
    _call(lqr, inp, pol, pol["status"], tan, o2, stream=side)
    side.synchronize()
    for k in POLICY_NAMES:
        assert torch.equal(o1[k], o2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _call(lqr, inp, pol, pol["status"], tan, o2, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for k in POLICY_NAMES:
        o2[k].fill_(float("nan"))
    torch.cuda.synchronize()
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    for k in POLICY_NAMES:
        assert torch.equal(o1[k], o2[k]), k
    lib.sipoc_graph_destroy(graph)


@pytest.mark.parametrize("n,m,T,kw", [(12, 4, 6, {}), (6, 2, 5, {}), (5, 3, 5, {}),
                                      (6, 2, 5, dict(force_generic=True))])
def test_adjoint_identity_with_device_vjp(n, m, T, kw):
    s, host = pg.lqr_benchmark_batch(n, m, T, 37, seed=14, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    rng = np.random.default_rng(15)
    tan = _rand_like(rng, inp, INPUT_NAMES)  # Q, R blocks not symmetric
    cot = _rand_like(rng, pol, POLICY_NAMES)
    jvp = lqr.policy_jvp(inp, pol, pol["status"], tan)
    vjp = lqr.policy_vjp(inp, pol, pol["status"], cot)
    b = lqr.batch
    lhs = sum((cot[k] * jvp[k]).sum(0) for k in POLICY_NAMES)[:b]
    rhs = sum((tan[k] * vjp[k]).sum(0) for k in INPUT_NAMES)[:b]
    assert ((lhs - rhs).abs() <= 1e-10 * lhs.abs().max()).all(), (lhs, rhs)


@pytest.mark.parametrize("n,m", [(6, 2), (12, 4), (5, 3)])
def test_directional_finite_difference(n, m):
    T = 5
    s, host = pg.lqr_benchmark_batch(n, m, T, 9, seed=12, dense_M=True)
    lqr, inp, pol = _forward(s, host)
    e = lqr.engine
    L = {k: e.lqr_sizes[k] for k in INPUT_NAMES}
    torch.manual_seed(13)
    direction = {k: torch.randn_like(inp[k]) for k in INPUT_NAMES}
    for key, dims in (("Q", [n] * (T + 1)), ("R", [m] * T)):  # symmetric directions
        d = dims[0]
        t = direction[key][: L[key]].reshape(len(dims), d, d, -1)
        direction[key][: L[key]] = ((t + t.transpose(1, 2)) / 2).reshape(L[key], -1)
    direction["delta"] *= 1e-2 * inp["delta"].abs()
    jvp = lqr.policy_jvp(inp, pol, pol["status"], direction)

    def policy(t):
        return lqr.factor_solve_policy({k: inp[k] + t * direction[k] for k in INPUT_NAMES},
                                       lqr.alloc_output())

    eps = 1e-6
    plus, minus = policy(eps), policy(-eps)
    for k in POLICY_NAMES:
        fd = ((plus[k] - minus[k]) / (2 * eps))[:, : lqr.batch]
        got = jvp[k][:, : lqr.batch]
        assert ((got - fd).abs() <= 1e-6 * (1 + fd.abs().max())).all(), k


def _autograd_case(n=4, m=2, T=3, batch=3):
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=17, dense_M=True)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    return s, lqr, lqr.pack_input(host)


def test_binding_forward_and_backward_match_factor_solve_policy():
    _s, lqr, inp = _autograd_case(6, 2, 5, 37)
    names = ("x", "u", "y") + POLICY_NAMES
    la = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    lb = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    a = autograd.factor_solve_policy(lqr, la)
    b = autograd.factor_solve_policy_fwd(lqr, lb)
    for k, ta, tb in zip(names + ("status",), a, b):
        assert torch.equal(ta, tb), k
    torch.manual_seed(3)
    cot = [torch.randn_like(t) for t in a[:7]]
    sum((c * t).sum() for c, t in zip(cot, a[:7])).backward()
    sum((c * t).sum() for c, t in zip(cot, b[:7])).backward()
    for k in INPUT_NAMES:
        assert torch.equal(la[k].grad, lb[k].grad), k


def test_binding_tangents_match_engine_calls():
    _s, lqr, inp = _autograd_case(6, 2, 5, 37)
    e = lqr.engine
    torch.manual_seed(5)
    tan = {k: torch.randn_like(v) for k, v in inp.items()}
    out = lqr.alloc_output()
    pol = lqr.factor_solve_policy(inp, out)
    sol = lqr.jvp({k: inp[k] for k in ("Q", "M", "R", "A", "B", "delta")}, out, tan)
    ptan = lqr.policy_jvp(inp, pol, pol["status"], tan)
    want = [sol["x"], sol["u"], sol["y"]] + [ptan[k] for k in POLICY_NAMES]

    def f(*arrays):
        return autograd.factor_solve_policy_fwd(lqr, dict(zip(INPUT_NAMES, arrays)))[:7]

    _, got = torch.func.jvp(f, tuple(inp[k] for k in INPUT_NAMES),
                            tuple(tan[k] for k in INPUT_NAMES))
    for k, g, w in zip(("x", "u", "y") + POLICY_NAMES, got, want):
        assert torch.equal(g, w), k
    fa = torch.autograd.forward_ad
    with fa.dual_level():
        dual = {k: fa.make_dual(inp[k], tan[k]) for k in INPUT_NAMES}
        outs = autograd.factor_solve_policy_fwd(lqr, dual)
        for k, o, w in zip(("x", "u", "y") + POLICY_NAMES, outs[:7], want):
            assert torch.equal(fa.unpack_dual(o).tangent, w), k
    assert e.launch_count > 0


def _sym_blocks(P, d):
    t = P.reshape(-1, d, d, P.shape[1])
    return ((t + t.transpose(1, 2)) / 2).reshape(P.shape)


def test_gradcheck_forward_and_backward():
    n, m = 4, 2
    _s, lqr, inp = _autograd_case(n, m)
    PQ = inp["Q"].clone().requires_grad_(True)
    PR = inp["R"].clone().requires_grad_(True)
    A = inp["A"].clone().requires_grad_(True)
    delta = inp["delta"].clone().requires_grad_(True)
    M = inp["M"].clone().requires_grad_(True)
    c = inp["c"].clone().requires_grad_(True)

    def f(PQ, PR, A, delta, M, c):
        arrays = dict(inp, Q=_sym_blocks(PQ, n), R=_sym_blocks(PR, m), A=A, delta=delta, M=M, c=c)
        return autograd.factor_solve_policy_fwd(lqr, arrays)[:7]

    assert torch.autograd.gradcheck(f, (PQ, PR, A, delta, M, c), eps=1e-6, atol=1e-6,
                                    rtol=1e-5, fast_mode=True, check_forward_ad=True,
                                    check_backward_ad=True)
