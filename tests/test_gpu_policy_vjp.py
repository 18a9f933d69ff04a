"""sipoc_lqr_policy_vjp (the reverse-mode derivative of the feedback policy K, k, V, v) against
the CPU adjoint sweep (policy_vjp_reference.py) on every plan family and structure, plus its
contract: the kernel each structure runs, NULL cotangents bitwise equal to zero ones, NULL
gradients untouched, zeros in failed problems and padding lanes, bitwise repeatable (eager and
graph replay), a directional finite difference of the device policy, and the torch.autograd
binding (gradcheck, a combined loss, forward outputs).

Tolerance, as in test_gpu_vjp.py: REL_TOL (1e-9 relative per problem and array) on q, r, c;
2 * REL_TOL on Q, M, R, A, B, delta.  After a parallel-in-time forward, whose V and v differ
from the serial recursion's by reassociation, 1e-8."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from oracle.pyoracle import Structure
from policy_reference import POLICY_NAMES, SIZE_OF, lqr_policy
from policy_vjp_reference import INPUT_NAMES, policy_vjp
from sip_optimal_control_b200 import LQR, autograd
from sip_optimal_control_b200 import _capi
from sip_optimal_control_b200._capi import lib
from test_gpu_fuzz import random_structure

pytestmark = pytest.mark.gpu

PRODUCTS = ("Q", "M", "R", "A", "B", "delta")
CHAIN_SHAPES = [(n, m) for n in (4, 6, 8) for m in (1, 2, 3, 4)] + [(12, 4)]


def _tol(k, tol=REL_TOL):
    return 2 * tol if k in PRODUCTS else tol


def _cot(s, batch, seed, names=POLICY_NAMES):
    rng = np.random.default_rng(seed)
    sz = pyoracle.lqr_sizes(s)
    return {k: rng.standard_normal((batch, sz[SIZE_OF[k]])) for k in names}


def _launches(e):
    launches = {}
    for i in range(lib.sipoc_profile_collect(e._handle)):
        nm, cnt = ctypes.c_char_p(), ctypes.c_int64()
        e._check(lib.sipoc_profile_get(e._handle, i, ctypes.byref(nm), None, ctypes.byref(cnt)))
        launches[nm.value.decode()] = cnt.value
    return launches


def _forward(s, host, **kw):
    dims, topo = to_structs(s)
    batch = host["q"].shape[0]
    lqr = LQR(dims, topo, batch, **kw)
    inp = lqr.pack_input(host)
    pol = lqr.factor_solve_policy(inp, lqr.alloc_output())
    return lqr, inp, pol


def _device_grads(lqr, inp, pol, cot, want=None):
    """Gradients (host arrays) and the engine launches of the policy_vjp call alone."""
    e = lqr.engine
    dcot = {k: e.pack(v) for k, v in cot.items()}
    before = e.launch_count
    res = lqr.policy_vjp(inp, pol, pol["status"], dcot, want=want)
    launches = e.launch_count - before
    return {k: e.unpack(res[k], e.lqr_sizes[k]) for k in INPUT_NAMES if k in res}, launches


def _check(s, host, kernel=None, tol=REL_TOL, seed=1, **kw):
    assert (pyoracle.lqr_factor_solve(s, host)["status"] == 0).all()
    cot = _cot(s, host["q"].shape[0], seed)
    ref = policy_vjp(s, host, cot)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    lib.sipoc_profile_enable(e._handle, 1)
    _launches(e)
    got, count = _device_grads(lqr, inp, pol, cot)
    assert count == 1
    launches = {k: v for k, v in _launches(e).items() if k.startswith("policy_vjp")}
    lib.sipoc_profile_enable(e._handle, 0)
    if kernel is not None:
        assert launches == {kernel: 1}, launches
    for k in INPUT_NAMES:
        if got[k].shape[1]:
            err = rel_err(got[k], ref[k]).max()
            assert err <= _tol(k, tol), (k, float(err), e.kernel_variant)
    return lqr, got


@pytest.mark.parametrize("n,m", CHAIN_SHAPES)
def test_chain_shapes(n, m):
    s, host = pg.lqr_benchmark_batch(n, m, 7, 37, seed=n * 10 + m, dense_M=True)
    _check(s, host, "policy_vjp_kernel")


@pytest.mark.parametrize("n,m,T", [(16, 4, 5), (32, 8, 3), (64, 24, 2), (5, 4, 6), (10, 3, 4)])
def test_generic_kernel_shapes(n, m, T):
    # the CTA plans' shapes and shapes that run on a padded plan: the generic kernel
    s, host = pg.lqr_benchmark_batch(n, m, T, 33, seed=n + T, dense_M=True)
    _check(s, host, "policy_vjp_generic_kernel")


@pytest.mark.parametrize("seed", range(6))
def test_random_trees(seed):
    rng = np.random.default_rng(4000 + seed)
    s = random_structure(rng)
    batch = int(rng.integers(1, 71))
    host = pg.variable_tree_batch(s, batch, seed=seed)
    for force_generic in (False, True):
        _check(s, host, seed=seed, force_generic=force_generic)


@pytest.mark.parametrize("builder", [fx.five_node_tree, fx.variable_dim_branch_tree,
                                     fx.nonuniform_delta_chain])
def test_reference_fixtures(builder):
    s, p = builder()
    host = {k: np.repeat(v, 5, axis=0) for k, v in fx.pack_problem(**p).items()}
    _check(s, host)


@pytest.mark.parametrize("kw,kernel,tol", [
    ({}, "policy_vjp_kernel", REL_TOL),
    (dict(force_generic=True), "policy_vjp_kernel", REL_TOL),
    (dict(parallel_in_time=True), "policy_vjp_kernel", 1e-8),
])
def test_forward_plan_families(kw, kernel, tol):
    # the VJP depends on the structure only; the forward's plan changes V, v by rounding
    s, host = pg.lqr_benchmark_batch(12, 4, 64 if kw.get("parallel_in_time") else 12, 19,
                                     seed=21, dense_M=True)
    lqr, _ = _check(s, host, kernel, tol=tol, **kw)
    if kw:
        assert ("generic" if "force_generic" in kw else "scan_") in lqr.engine.kernel_variant


@pytest.mark.parametrize("pad_variable_dims", [False, True])
def test_padded_and_strict_forwards(pad_variable_dims):
    s = Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])
    host = pg.variable_tree_batch(s, 40, seed=4)
    lqr, _ = _check(s, host, "policy_vjp_generic_kernel", pad_variable_dims=pad_variable_dims)
    assert "padded_to_" in lqr.engine.kernel_variant


@pytest.mark.parametrize("batch", [1, 31, 33, 97])
def test_ragged_batches(batch):
    s, host = pg.lqr_benchmark_batch(6, 2, 5, batch, seed=batch, dense_M=True)
    lqr, _ = _check(s, host, "policy_vjp_kernel")


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
    cot = {k: torch.from_numpy(rng.standard_normal(tuple(pol[k].shape))).to(pol[k].device)
           for k in POLICY_NAMES}
    res = lqr.policy_vjp(inp, pol, pol["status"], cot)
    torch.cuda.synchronize()
    idx = torch.from_numpy(rng.choice(batch, 48, replace=False)).to(e.torch_device())
    sample = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: sample(inp[k], e.lqr_sizes[k]) for k in INPUT_NAMES}
    ref = policy_vjp(s, host, {k: sample(cot[k], e.lqr_sizes[SIZE_OF[k]]) for k in POLICY_NAMES})
    for k in INPUT_NAMES:
        err = rel_err(sample(res[k], e.lqr_sizes[k]), ref[k]).max()
        assert err <= _tol(k), (k, float(err))


def _call(lqr, inp, pol, status, cot, grad, stream=None):
    e = lqr.engine
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in INPUT_NAMES])
    sc = _capi.LqrPolicyCotangent(*[cot[k].data_ptr() if cot.get(k) is not None else None
                                    for k in POLICY_NAMES])
    sg = _capi.LqrGrad(*[grad[k].data_ptr() if k in grad else None for k in INPUT_NAMES])
    e._check(lib.sipoc_lqr_policy_vjp(e._handle, ctypes.byref(si), pol["V"].data_ptr(),
                                      pol["v"].data_ptr(), status.data_ptr(), ctypes.byref(sc),
                                      ctypes.byref(sg), e.stream_ptr(stream)))


@pytest.mark.parametrize("n,m,kw", [(12, 4, {}), (5, 2, {}), (12, 4, dict(force_generic=True))])
def test_null_cotangents_and_null_grads(n, m, kw):
    s, host = pg.lqr_benchmark_batch(n, m, 6, 37, seed=3, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    rng = np.random.default_rng(2)
    for keep in (("K",), ("V", "v"), ("k", "v")):
        cot = {k: torch.from_numpy(rng.standard_normal(tuple(pol[k].shape))).to(pol[k].device)
               for k in keep}
        zeros = dict(cot, **{k: torch.zeros_like(pol[k]) for k in POLICY_NAMES if k not in keep})
        g1 = {k: e.empty(e.lqr_sizes[k]) for k in INPUT_NAMES}
        g2 = {k: e.empty(e.lqr_sizes[k]) for k in INPUT_NAMES}
        _call(lqr, inp, pol, pol["status"], cot, g1)
        _call(lqr, inp, pol, pol["status"], zeros, g2)
        torch.cuda.synchronize()
        for k in INPUT_NAMES:
            assert torch.equal(g1[k], g2[k]), (keep, k)
    full = {k: torch.from_numpy(rng.standard_normal(tuple(pol[k].shape))).to(pol[k].device)
            for k in POLICY_NAMES}
    ref = {k: e.empty(e.lqr_sizes[k]) for k in INPUT_NAMES}
    _call(lqr, inp, pol, pol["status"], full, ref)
    for want in (("q",), ("A", "delta"), ("Q", "R", "c")):
        g = {k: torch.full_like(ref[k], float("nan")) for k in INPUT_NAMES}
        _call(lqr, inp, pol, pol["status"], full, {k: g[k] for k in want})
        torch.cuda.synchronize()
        for k in INPUT_NAMES:
            if k in want:
                assert torch.equal(g[k], ref[k]), (want, k)
            else:
                assert torch.isnan(g[k]).all(), (want, k)
    before = e.launch_count
    _call(lqr, inp, pol, pol["status"], full, {})  # nothing requested: nothing launched
    assert e.launch_count == before
    # only K and V: the gradients of q, r, c are exactly zero
    g = {k: e.empty(e.lqr_sizes[k]) for k in INPUT_NAMES}
    _call(lqr, inp, pol, pol["status"], {k: full[k] for k in ("K", "V")}, g)
    for k in ("q", "r", "c"):
        assert not g[k].any(), k


@pytest.mark.parametrize("force_generic", [False, True])
def test_failed_problems_and_padding_lanes_are_zero(force_generic):
    n, m, T, batch = 4, 1, 3, 6
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=10, dense_M=True)
    host["delta"][1, T * n + 0] = 0.0
    host["R"][3, (T - 1) * m * m] = -50.0
    ref_status = pyoracle.lqr_factor_solve(s, host)["status"]
    assert ref_status[1] != 0 and ref_status[3] != 0 and (ref_status[[0, 2, 4, 5]] == 0).all()
    good = ref_status == 0
    cot = _cot(s, batch, 6)
    ref = policy_vjp(s, {k: v[good] for k, v in host.items()}, {k: v[good] for k, v in cot.items()})
    lqr, inp, pol = _forward(s, host, force_generic=force_generic)
    e = lqr.engine
    res = lqr.policy_vjp(inp, pol, pol["status"], {k: e.pack(v) for k, v in cot.items()})
    assert pol["status"][:batch].cpu().numpy().tolist() == ref_status.tolist()
    for k in INPUT_NAMES:
        full = res[k][: e.lqr_sizes[k]].cpu().numpy()
        assert not full[:, batch:].any(), k
        assert not full[:, :batch][:, ~good].any(), k
        assert rel_err(full[:, :batch].T[good], ref[k]).max() <= _tol(k), k


@pytest.mark.parametrize("n,m,kw", [(12, 4, {}), (3, 2, {})])
def test_bitwise_repeatable_and_graph_replay(n, m, kw):
    s, host = pg.lqr_benchmark_batch(n, m, 8, 37, seed=9, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    rng = np.random.default_rng(4)
    cot = {k: torch.from_numpy(rng.standard_normal(tuple(pol[k].shape))).to(pol[k].device)
           for k in POLICY_NAMES}
    side = torch.cuda.Stream()
    bufs = lambda: {k: e.empty(e.lqr_sizes[k]) for k in INPUT_NAMES}
    g1, g2 = bufs(), bufs()
    torch.cuda.synchronize()
    _call(lqr, inp, pol, pol["status"], cot, g1, stream=side)
    _call(lqr, inp, pol, pol["status"], cot, g2, stream=side)
    side.synchronize()
    for k in INPUT_NAMES:
        assert torch.equal(g1[k], g2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _call(lqr, inp, pol, pol["status"], cot, g2, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for k in INPUT_NAMES:
        g2[k].fill_(float("nan"))
    torch.cuda.synchronize()
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    for k in INPUT_NAMES:
        assert torch.equal(g1[k], g2[k]), k
    lib.sipoc_graph_destroy(graph)


@pytest.mark.parametrize("n,m,kw", [(6, 2, {}), (5, 3, {})])
def test_directional_finite_difference(n, m, kw):
    s, host = pg.lqr_benchmark_batch(n, m, 5, 9, seed=12, dense_M=True)
    lqr, inp, pol = _forward(s, host, **kw)
    e = lqr.engine
    rng = np.random.default_rng(13)
    cot = {k: torch.from_numpy(rng.standard_normal(tuple(pol[k].shape))).to(pol[k].device)
           for k in POLICY_NAMES}
    grads = lqr.policy_vjp(inp, pol, pol["status"], cot)
    L = {k: e.lqr_sizes[k] for k in INPUT_NAMES}
    direction = {k: torch.randn_like(inp[k]) for k in INPUT_NAMES}
    for key, dims in (("Q", [n] * 6), ("R", [m] * 5)):  # symmetric directions
        d = dims[0]
        t = direction[key][: L[key]].reshape(len(dims), d, d, -1)
        direction[key][: L[key]] = ((t + t.transpose(1, 2)) / 2).reshape(L[key], -1)
    direction["delta"] *= 1e-2 * inp["delta"].abs()

    def loss(t):
        p = lqr.factor_solve_policy({k: inp[k] + t * direction[k] for k in INPUT_NAMES},
                                    lqr.alloc_output())
        return sum((cot[k] * p[k]).sum(0) for k in POLICY_NAMES)

    eps = 1e-6
    fd = ((loss(eps) - loss(-eps)) / (2 * eps))[: lqr.batch]
    dot = sum((grads[k] * direction[k]).sum(0) for k in INPUT_NAMES)[: lqr.batch]
    assert ((dot - fd).abs() <= 1e-6 * (1 + fd.abs().max())).all(), (dot, fd)


def _autograd_case(n=4, m=2, T=3, batch=3):
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=17, dense_M=True)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    return s, lqr, lqr.pack_input(host)


def _sym_blocks(P, d):
    t = P.reshape(-1, d, d, P.shape[1])
    return ((t + t.transpose(1, 2)) / 2).reshape(P.shape)


def test_gradcheck():
    n, m = 4, 2
    s, lqr, inp = _autograd_case(n, m)
    PQ = inp["Q"].clone().requires_grad_(True)
    PR = inp["R"].clone().requires_grad_(True)
    A = inp["A"].clone().requires_grad_(True)
    delta = inp["delta"].clone().requires_grad_(True)
    M = inp["M"].clone().requires_grad_(True)

    def f(PQ, PR, A, delta, M):
        arrays = dict(inp, Q=_sym_blocks(PQ, n), R=_sym_blocks(PR, m), A=A, delta=delta, M=M)
        return autograd.factor_solve_policy(lqr, arrays)[:7]

    assert torch.autograd.gradcheck(f, (PQ, PR, A, delta, M), eps=1e-6, atol=1e-6, rtol=1e-5,
                                    fast_mode=True)


def test_combined_loss_and_forward_outputs():
    s, lqr, inp = _autograd_case(6, 2, 5, 37)
    e = lqr.engine
    leaves = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    outs = autograd.factor_solve_policy(lqr, leaves)
    names = ("x", "u", "y") + POLICY_NAMES
    ref_out = lqr.alloc_output()
    ref_pol = lqr.factor_solve_policy(inp, ref_out)
    for k, t in zip(names, outs[:7]):
        assert torch.equal(t, ref_out[k] if k in "xuy" else ref_pol[k]), k
    assert torch.equal(outs[7], ref_pol["status"])
    cot = {k: torch.randn_like(t) for k, t in zip(names, outs[:7])}
    loss = sum((cot[k] * t).sum() for k, t in zip(names, outs[:7]))
    loss.backward()
    g1 = lqr.vjp(inp, {k: ref_out[k] for k in "xuy"}, {k: cot[k] for k in "xuy"})
    g2 = lqr.policy_vjp(inp, ref_pol, ref_pol["status"], {k: cot[k] for k in POLICY_NAMES})
    for k in INPUT_NAMES:
        want = g1[k] + g2[k]
        assert torch.allclose(leaves[k].grad, want, rtol=1e-13, atol=1e-13 * float(want.abs().max())), k
    # only policy cotangents: the solve VJP does not run
    leaves = {k: v.clone().requires_grad_(True) for k, v in inp.items()}
    outs = autograd.factor_solve_policy(lqr, leaves)
    before = e.launch_count
    (outs[3] * cot["K"]).sum().backward()
    assert e.launch_count - before == 1
    with pytest.raises(RuntimeError):
        with torch.autograd.forward_ad.dual_level():
            dual = {k: torch.autograd.forward_ad.make_dual(v, torch.zeros_like(v))
                    for k, v in inp.items()}
            autograd.factor_solve_policy(lqr, dual)
