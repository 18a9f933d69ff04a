"""sipoc_lqr_factor_solve_policy (the feedback policy K, k, V, v of the LQR solve) against the
CPU reference (policy_reference.py) on every plan family, plus its contract: x, u, y, status
bitwise those of sipoc_lqr_factor_solve, the policy reproduces the device solution, NULL
arrays untouched (and no V rebuild for K, k alone), zeros in failed problems and padding
lanes, bitwise repeatable (eager and graph replay).

Tolerance: REL_TOL (1e-9 relative per problem and array), as for the solution itself."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from oracle.pyoracle import Structure
from policy_reference import POLICY_NAMES, SIZE_OF, lqr_policy, policy_residuals
from sip_optimal_control_b200 import LQR
from sip_optimal_control_b200 import _capi
from sip_optimal_control_b200._capi import lib
from test_gpu_fuzz import random_structure

pytestmark = pytest.mark.gpu


def _unpack_policy(lqr, res):
    e = lqr.engine
    return {k: e.unpack(res[k], e.lqr_sizes[SIZE_OF[k]]) for k in POLICY_NAMES if k in res}


def _check(s, host, family=None, tol=REL_TOL, **kw):
    ref_sol = pyoracle.lqr_factor_solve(s, host)
    assert (ref_sol["status"] == 0).all()
    ref = lqr_policy(s, host)
    dims, topo = to_structs(s)
    batch = host["q"].shape[0]
    lqr = LQR(dims, topo, batch, **kw)
    e = lqr.engine
    if family is not None:
        assert family in e.kernel_variant, e.kernel_variant
    inp = lqr.pack_input(host)
    out0, out = lqr.alloc_output(), lqr.alloc_output()
    st0 = lqr.factor_solve(inp, out0)
    res = lqr.factor_solve_policy(inp, out)
    torch.cuda.synchronize()
    for k in ("x", "u", "y"):
        assert torch.equal(out[k], out0[k]), (k, e.kernel_variant)
    assert torch.equal(res["status"][:batch], st0[:batch])
    assert (res["status"][:batch] == 0).all(), e.kernel_variant
    got = _unpack_policy(lqr, res)
    for k in POLICY_NAMES:
        if got[k].shape[1]:
            err = rel_err(got[k], ref[k]).max()
            assert err <= tol, (k, float(err), e.kernel_variant)
    sol = lqr.unpack_output(out)
    ru, ry = policy_residuals(s, host, got, sol["x"], sol["u"], sol["y"])
    assert ru.max() <= tol and ry.max() <= tol, (ru.max(), ry.max(), e.kernel_variant)
    return lqr, got


@pytest.mark.parametrize("n,m,T,family", [(4, 1, 20, "thread_per_problem"), (4, 3, 7, "thread_per_problem"),
                                          (6, 2, 9, "subwarp4"), (8, 4, 5, "subwarp4"),
                                          (12, 4, 10, "subwarp4"), (16, 4, 6, "cta"),
                                          (64, 24, 3, "cta")])
def test_plan_families_match_reference(n, m, T, family):
    s, host = pg.lqr_benchmark_batch(n, m, T, 37, seed=n + T, dense_M=True)
    _, got = _check(s, host, family)
    for i in range(T + 1):  # V exactly symmetric on the plans that rebuild it
        Vi = got["V"][:, i * n * n:(i + 1) * n * n].reshape(-1, n, n)
        assert np.array_equal(Vi, Vi.transpose(0, 2, 1))


def test_two_kernel_subwarp_pair_large_batch():
    # above 40 960 problems the sub-warp plan runs the sweep and the rollout as two kernels
    n, m, T, batch = 12, 4, 3, 41000
    s = Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    inp = lqr.generate_benchmark(seed=5)
    out = lqr.alloc_output()
    res = lqr.factor_solve_policy(inp, out)
    torch.cuda.synchronize()
    assert (res["status"][:batch] == 0).all()
    idx = torch.from_numpy(np.random.default_rng(7).choice(batch, 48, replace=False)).to(
        e.torch_device())
    sample = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: sample(inp[k], e.lqr_sizes[k]) for k in pyoracle.LQR_INPUT_NAMES}
    ref = lqr_policy(s, host)
    for k in POLICY_NAMES:
        err = rel_err(sample(res[k], e.lqr_sizes[SIZE_OF[k]]), ref[k]).max()
        assert err <= REL_TOL, (k, float(err), e.kernel_variant)


@pytest.mark.parametrize("pad_variable_dims", [False, True])
def test_padded_variable_dims(pad_variable_dims):
    s = Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])
    host = pg.variable_tree_batch(s, 40, seed=4)
    lqr, _ = _check(s, host, pad_variable_dims=pad_variable_dims)
    assert "padded_to_" in lqr.engine.kernel_variant
    assert ("strict" in lqr.engine.kernel_variant) != pad_variable_dims


@pytest.mark.parametrize("n,m,family", [(5, 4, "padded_to_subwarp4_n6_m4"),
                                        (10, 3, "padded_to_subwarp4_n12_m4"),
                                        (20, 4, "padded_to_cta_dmma_n32_m8")])
def test_uniform_shape_padded_to_next_plan(n, m, family):
    s, host = pg.lqr_benchmark_batch(n, m, 6, 33, seed=n, dense_M=True)
    _check(s, host, family)


@pytest.mark.parametrize("builder", [fx.five_node_tree, fx.variable_dim_branch_tree])
def test_force_generic(builder):
    s, p = builder()
    host = {k: np.repeat(v, 5, axis=0) for k, v in fx.pack_problem(**p).items()}
    _check(s, host, "generic", force_generic=True)


@pytest.mark.parametrize("seed", range(8))
def test_random_trees(seed):
    rng = np.random.default_rng(3000 + seed)
    s = random_structure(rng)
    batch = int(rng.integers(1, 71))
    host = pg.variable_tree_batch(s, batch, seed=seed)
    for force_generic in (False, True):
        _check(s, host, "generic" if force_generic else None, force_generic=force_generic)


def test_forced_scan():
    n, m, T, batch = 12, 4, 64, 19
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=T + n, dense_M=True)
    _check(s, host, "scan_", parallel_in_time=True)


def _policy_call(lqr, inp, out, arrays, status, stream=None):
    e = lqr.engine
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in pyoracle.LQR_INPUT_NAMES])
    so = _capi.LqrOutput(*[out[k].data_ptr() for k in ("x", "u", "y")])
    sp = _capi.LqrPolicy(*[arrays[k].data_ptr() if k in arrays else None for k in POLICY_NAMES])
    e._check(lib.sipoc_lqr_factor_solve_policy(
        e._handle, ctypes.byref(si), ctypes.byref(so), ctypes.byref(sp),
        None if status is None else status.data_ptr(), e.stream_ptr(stream)))


def _device_case(n=12, m=4, T=10, batch=37, **kw):
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=9, dense_M=True)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch, **kw)
    return s, host, lqr, lqr.pack_input(host)


def _launches(e):
    launches = {}
    for i in range(lib.sipoc_profile_collect(e._handle)):
        nm, cnt = ctypes.c_char_p(), ctypes.c_int64()
        e._check(lib.sipoc_profile_get(e._handle, i, ctypes.byref(nm), None, ctypes.byref(cnt)))
        launches[nm.value.decode()] = cnt.value
    return launches


@pytest.mark.parametrize("n,m", [(12, 4), (16, 4)])
def test_only_requested_arrays_are_written(n, m):
    s, host, lqr, inp = _device_case(n, m, 6)
    e = lqr.engine
    sentinel = 12345.5
    full = lqr.factor_solve_policy(inp, lqr.alloc_output())
    for want in (("K", "k"), ("V",), ("v", "K")):
        arrays = {k: torch.full_like(full[k], sentinel) for k in POLICY_NAMES}
        _policy_call(lqr, inp, lqr.alloc_output(), {k: arrays[k] for k in want}, None)
        torch.cuda.synchronize()
        for k in POLICY_NAMES:
            if k in want:
                assert torch.equal(arrays[k], full[k]), k
            else:
                assert (arrays[k] == sentinel).all(), k
    # K, k alone: no V rebuild; V: exactly one
    lib.sipoc_profile_enable(e._handle, 1)
    lqr.factor_solve_policy(inp, lqr.alloc_output(), want=("K", "k"))
    launches = _launches(e)
    assert "policy_rebuild_v_kernel" not in launches, launches
    assert launches["policy_gather_kernel"] == 2, launches
    lqr.factor_solve_policy(inp, lqr.alloc_output(), want=("V",))
    assert _launches(e)["policy_rebuild_v_kernel"] == 1
    lib.sipoc_profile_enable(e._handle, 0)
    with pytest.raises(ValueError):
        lqr.factor_solve_policy(inp, lqr.alloc_output(), want=("K", "W"))


@pytest.mark.parametrize("force_generic", [True, False])
def test_failed_problems_and_padding_lanes_are_zero(force_generic):
    n, m, T, batch = 2, 1, 2, 6
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=10, dense_M=True)
    host["delta"][1, T * n + 0] = 0.0
    host["Q"][2, T * n * n:] = (-2.0 * np.eye(n)).flatten()
    host["delta"][2, T * n:] = 1.0
    host["Q"][3, T * n * n:] = 0.0
    host["R"][3, (T - 1) * m * m] = -1.0
    host["delta"][4, 1] = -1.0
    host["R"][4, (T - 1) * m * m] = -50.0
    ref_sol = pyoracle.lqr_factor_solve(s, host)
    assert ref_sol["status"].tolist() == [0, 1, 2, 3, 3, 0]
    ref = lqr_policy(s, host)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch, force_generic=force_generic)
    e = lqr.engine
    assert ("generic" in e.kernel_variant) == force_generic
    inp = lqr.pack_input(host)
    res = lqr.factor_solve_policy(inp, lqr.alloc_output())
    assert res["status"][:batch].cpu().tolist() == [0, 1, 2, 3, 3, 0]
    good = ref_sol["status"] == 0
    for k in POLICY_NAMES:
        full = res[k][: e.lqr_sizes[SIZE_OF[k]]].cpu().numpy()  # [size, batch_stride]
        assert not full[:, batch:].any(), k
        assert not full[:, :batch][:, ~good].any(), k
        assert rel_err(full[:, :batch].T[good], ref[k][good]).max() <= REL_TOL, k


@pytest.mark.parametrize("kw", [{}, dict(parallel_in_time=True)])
def test_bitwise_repeatable_and_graph_replay(kw):
    s, host, lqr, inp = _device_case(12, 4, 64 if kw else 10, 37, **kw)
    e = lqr.engine
    side = torch.cuda.Stream()
    bufs = lambda: {k: e.empty(e.lqr_sizes[SIZE_OF[k]]) for k in POLICY_NAMES}
    p1, p2 = bufs(), bufs()
    o1, o2 = lqr.alloc_output(), lqr.alloc_output()
    status = e.empty_int()
    torch.cuda.synchronize()
    _policy_call(lqr, inp, o1, p1, status, stream=side)
    _policy_call(lqr, inp, o2, p2, status, stream=side)
    side.synchronize()
    for k in POLICY_NAMES:
        assert torch.equal(p1[k], p2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _policy_call(lqr, inp, o2, p2, status, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for k in POLICY_NAMES:
        p2[k].fill_(float("nan"))
    torch.cuda.synchronize()
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    for k in POLICY_NAMES:
        assert torch.equal(p1[k], p2[k]), k
    for k in ("x", "u", "y"):
        assert torch.equal(o1[k], o2[k]), k
    lib.sipoc_graph_destroy(graph)
