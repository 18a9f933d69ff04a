"""sipoc_lqr_vjp (the reverse-mode derivative of the LQR solve) against the CPU reference VJP
(vjp_reference.py) on every plan family, plus its contract: NULL arrays untouched, zeros in
failed problems and padding lanes, bitwise repeatable (eager and graph replay), and the
torch.autograd binding (gradcheck, a composite loss).

Tolerance: REL_TOL (1e-9 relative per problem and array) on q, r, c, which are the adjoint
itself; 2 * REL_TOL on Q, M, R, A, B, delta, each a sum of products of a 1e-9-accurate
solution entry with a 1e-9-accurate adjoint entry."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from oracle.pyoracle import Structure
from sip_optimal_control_b200 import LQR, autograd
from sip_optimal_control_b200 import _capi
from sip_optimal_control_b200._capi import lib
from test_gpu_fuzz import random_structure
from vjp_reference import GRAD_NAMES, lqr_vjp

pytestmark = pytest.mark.gpu

PRODUCTS = ("Q", "M", "R", "A", "B", "delta")


def _tol(k, tol=REL_TOL):
    return 2 * tol if k in PRODUCTS else tol


def _cot(s, batch, seed):
    rng = np.random.default_rng(seed)
    sz = pyoracle.lqr_sizes(s)
    return {k: rng.standard_normal((batch, sz[k])) for k in ("x", "u", "y")}


def _run(s, host, cot, want=None, **kw):
    """Device forward + VJP; returns (solution, gradients, adjoint, status, lqr), host arrays."""
    dims, topo = to_structs(s)
    batch = host["q"].shape[0]
    lqr = LQR(dims, topo, batch, **kw)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    res = lqr.vjp(inp, out, {k: e.pack(cot[k]) for k in cot}, want=want)
    sol = lqr.unpack_output(out)
    grads = {k: e.unpack(res[k], e.lqr_sizes[k]) for k in GRAD_NAMES if k in res}
    adj = lqr.unpack_output(res["adjoint"])
    return sol, grads, adj, res["status"][:batch].cpu().numpy(), lqr


def _check(s, host, cot, tol=REL_TOL, **kw):
    ref_sol = pyoracle.lqr_factor_solve(s, host)
    assert (ref_sol["status"] == 0).all()
    ref = lqr_vjp(s, host, ref_sol, cot)
    sol, grads, adj, status, lqr = _run(s, host, cot, **kw)
    assert (status == 0).all(), lqr.engine.kernel_variant
    for k in ("x", "u", "y"):
        if adj[k].shape[1]:
            assert rel_err(adj[k], ref["adjoint"][k]).max() <= tol, (k, lqr.engine.kernel_variant)
    for k in GRAD_NAMES:
        if grads[k].shape[1]:
            err = rel_err(grads[k], ref[k]).max()
            assert err <= _tol(k, tol), (k, float(err), lqr.engine.kernel_variant)
    return lqr


@pytest.mark.parametrize("n,m,T,family", [(4, 1, 20, "thread"), (12, 4, 10, "subwarp"),
                                          (16, 4, 6, "cta"), (64, 24, 3, "cta")])
def test_plan_families_match_reference(n, m, T, family):
    batch = 37
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=n + T, dense_M=True)
    lqr = _check(s, host, _cot(s, batch, 1))
    assert "generic" not in lqr.engine.kernel_variant, lqr.engine.kernel_variant


def test_two_kernel_subwarp_pair_large_batch():
    # above 40 960 problems the sub-warp plan runs the sweep and the rollout as two kernels
    n, m, T, batch = 12, 4, 3, 41000
    s = Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    inp = lqr.generate_benchmark(seed=5)
    out = lqr.alloc_output()
    lqr.factor_solve(inp, out)
    gen = torch.Generator(device=e.torch_device()).manual_seed(6)
    cot = {k: torch.randn(out[k].shape, generator=gen, dtype=torch.float64,
                          device=e.torch_device()) for k in ("x", "u", "y")}
    res = lqr.vjp(inp, out, cot)
    torch.cuda.synchronize()
    assert (res["status"][:batch] == 0).all()
    idx = torch.from_numpy(np.random.default_rng(7).choice(batch, 64, replace=False)).to(
        e.torch_device())
    sample = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: sample(inp[k], e.lqr_sizes[k]) for k in GRAD_NAMES}
    hcot = {k: sample(cot[k], e.lqr_sizes[k]) for k in ("x", "u", "y")}
    ref = lqr_vjp(s, host, pyoracle.lqr_factor_solve(s, host), hcot)
    for k in GRAD_NAMES:
        err = rel_err(sample(res[k], e.lqr_sizes[k]), ref[k]).max()
        assert err <= _tol(k), (k, float(err), e.kernel_variant)


@pytest.mark.parametrize("pad_variable_dims", [False, True])
def test_padded_variable_dims(pad_variable_dims):
    s = Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])
    host = pg.variable_tree_batch(s, 40, seed=4)
    lqr = _check(s, host, _cot(s, 40, 2), pad_variable_dims=pad_variable_dims)
    assert "generic" not in lqr.engine.kernel_variant


@pytest.mark.parametrize("builder", [fx.five_node_tree, fx.variable_dim_branch_tree])
def test_force_generic(builder):
    s, p = builder()
    host = {k: np.repeat(v, 5, axis=0) for k, v in fx.pack_problem(**p).items()}
    lqr = _check(s, host, _cot(s, 5, 3), force_generic=True)
    assert "generic" in lqr.engine.kernel_variant


@pytest.mark.parametrize("seed", range(8))
def test_random_trees(seed):
    rng = np.random.default_rng(3000 + seed)
    s = random_structure(rng)
    batch = int(rng.integers(1, 71))
    host = pg.variable_tree_batch(s, batch, seed=seed)
    for force_generic in (False, True):
        _check(s, host, _cot(s, batch, seed), force_generic=force_generic)


def test_forced_scan():
    # the scan's own tolerance (test_gpu_scan.py): REL_TOL on (x, u, y)
    n, m, T, batch = 12, 4, 64, 19
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=T + n, dense_M=True)
    lqr = _check(s, host, _cot(s, batch, 4), parallel_in_time=True)
    assert lqr.engine.kernel_variant.startswith("scan_")


def _grad_struct(arrays):
    g = _capi.LqrGrad()
    for k in GRAD_NAMES:
        setattr(g, k, arrays[k].data_ptr() if k in arrays else None)
    return g


def _call(lqr, inp, out, cot, adjoint, grads, status, stream=None):
    e = lqr.engine
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in GRAD_NAMES])
    so = _capi.LqrOutput(*[out[k].data_ptr() for k in ("x", "u", "y")])
    sc = _capi.LqrCotangent(*[cot[k].data_ptr() for k in ("x", "u", "y")])
    sa = _capi.LqrOutput(*[adjoint[k].data_ptr() for k in ("x", "u", "y")])
    sg = _grad_struct(grads)
    e._check(lib.sipoc_lqr_vjp(e._handle, ctypes.byref(si), ctypes.byref(so), ctypes.byref(sc),
                               ctypes.byref(sa), ctypes.byref(sg),
                               None if status is None else status.data_ptr(),
                               e.stream_ptr(stream)))


def _device_case(n=12, m=4, T=10, batch=37, **kw):
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=9, dense_M=True)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch, **kw)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    cot = {k: e.pack(v) for k, v in _cot(s, batch, 8).items()}
    return s, host, lqr, inp, out, cot


def test_only_requested_arrays_are_written():
    s, host, lqr, inp, out, cot = _device_case()
    e = lqr.engine
    sentinel = 12345.5
    full = lqr.vjp(inp, out, cot)
    for want in (("q", "c"), ("Q", "B", "delta"), ("M", "R", "r", "A")):
        arrays = {k: torch.full_like(full[k], sentinel) for k in GRAD_NAMES}
        before = e.launch_count
        _call(lqr, inp, out, cot, lqr.alloc_output(), {k: arrays[k] for k in want}, None)
        torch.cuda.synchronize()
        assert e.launch_count > before
        for k in GRAD_NAMES:
            if k in want:
                assert torch.equal(arrays[k], full[k]), k
            else:
                assert (arrays[k] == sentinel).all(), k
    # no gradient requested: the adjoint alone, and no gradient kernel; one launch of the
    # gradient kernel per call that requests any
    lib.sipoc_profile_enable(e._handle, 1)
    adj = lqr.alloc_output()
    _call(lqr, inp, out, cot, adj, {}, None)
    _call(lqr, inp, out, cot, lqr.alloc_output(), {"r": torch.empty_like(full["r"])}, None)
    launches = {}
    for i in range(lib.sipoc_profile_collect(e._handle)):
        nm, cnt = ctypes.c_char_p(), ctypes.c_int64()
        e._check(lib.sipoc_profile_get(e._handle, i, ctypes.byref(nm), None, ctypes.byref(cnt)))
        launches[nm.value.decode()] = cnt.value
    assert launches["lqr_vjp_kernel"] == 1, launches
    lib.sipoc_profile_enable(e._handle, 0)
    for k in ("x", "u", "y"):
        assert torch.equal(adj[k], full["adjoint"][k]), k


@pytest.mark.parametrize("force_generic", [True, False])
def test_failed_problems_and_padding_lanes_are_zero(force_generic):
    n, m, T, batch = 2, 1, 2, 6
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=10, dense_M=True)
    # the failures of test_status_codes_per_problem (delta = 1 at the leaf keeps F = I - 2 I
    # indefinite on this data, as on that test's identity fixture)
    host["delta"][1, T * n + 0] = 0.0
    host["Q"][2, T * n * n:] = (-2.0 * np.eye(n)).flatten()
    host["delta"][2, T * n:] = 1.0
    host["Q"][3, T * n * n:] = 0.0
    host["R"][3, (T - 1) * m * m] = -1.0
    host["delta"][4, 1] = -1.0
    host["R"][4, (T - 1) * m * m] = -50.0
    ref_sol = pyoracle.lqr_factor_solve(s, host)
    assert ref_sol["status"].tolist() == [0, 1, 2, 3, 3, 0]
    cot = _cot(s, batch, 11)
    ref = lqr_vjp(s, host, ref_sol, cot)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch, force_generic=force_generic)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    res = lqr.vjp(inp, out, {k: e.pack(v) for k, v in cot.items()})
    assert res["status"][:batch].cpu().tolist() == [0, 1, 2, 3, 3, 0]
    good = ref_sol["status"] == 0
    for k in GRAD_NAMES:
        full = res[k][: e.lqr_sizes[k]].cpu().numpy()  # [size, batch_stride]
        assert not full[:, batch:].any(), k            # padding lanes
        assert not full[:, :batch][:, ~good].any(), k  # failed problems
        got = full[:, :batch].T
        assert rel_err(got[good], ref[k][good]).max() <= _tol(k), k


def test_bitwise_repeatable_and_graph_replay():
    s, host, lqr, inp, out, cot = _device_case(12, 4, 10, 37)
    e = lqr.engine
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    bufs = lambda: ({k: e.empty(e.lqr_sizes[k]) for k in GRAD_NAMES}, lqr.alloc_output())
    g1, a1 = bufs()
    g2, a2 = bufs()
    status = e.empty_int()
    torch.cuda.synchronize()
    _call(lqr, inp, out, cot, a1, g1, status, stream=side)
    _call(lqr, inp, out, cot, a2, g2, status, stream=side)
    side.synchronize()
    for k in GRAD_NAMES:
        assert torch.equal(g1[k], g2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _call(lqr, inp, out, cot, a2, g2, status, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for k in GRAD_NAMES:
        g2[k].fill_(float("nan"))
    torch.cuda.synchronize()
    before = e.launch_count
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    assert e.launch_count == before + lib.sipoc_graph_kernel_count(graph)
    for k in GRAD_NAMES:
        assert torch.equal(g1[k], g2[k]), k
    for k in ("x", "u", "y"):
        assert torch.equal(a1[k], a2[k]), k
    lib.sipoc_graph_destroy(graph)


def _block_transpose(sizes):
    """Row permutation of a flat array of square column-major blocks: each block transposed."""
    perm, off = [], 0
    for n in sizes:
        perm += [off + j + i * n for j in range(n) for i in range(n)]
        off += n * n
    return torch.tensor(perm, dtype=torch.long)


def _tiny():
    s, p = fx.variable_dim_branch_tree()
    host = fx.pack_problem(**p)
    batch = 3
    rng = np.random.default_rng(12)
    host = {k: np.repeat(v, batch, axis=0) for k, v in host.items()}
    for k in ("q", "r", "c"):
        host[k] = host[k] + 0.1 * rng.standard_normal(host[k].shape)
    return s, host, batch


def test_gradcheck_through_autograd_binding():
    s, host, batch = _tiny()
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    ld = lqr.engine.batch_stride
    dev = lqr.engine.torch_device()
    permQ = _block_transpose([int(v) for v in s.state_dims]).to(dev)
    permR = _block_transpose([int(v) for v in s.control_dims]).to(dev)
    leaves = [torch.tensor(host[k].T, dtype=torch.float64, device=dev, requires_grad=True)
              for k in GRAD_NAMES]

    def f(*arrays):
        a = dict(zip(GRAD_NAMES, arrays))
        a["Q"] = 0.5 * (a["Q"] + a["Q"].index_select(0, permQ))
        a["R"] = 0.5 * (a["R"] + a["R"].index_select(0, permR))
        # engine layout: [size, batch_stride]; the padding lanes are solved too, on copies of
        # problem 0, and must not leak into the gradients of the live lanes
        inp = {k: torch.cat([v, v[:, :1].expand(-1, ld - batch)], dim=1) for k, v in a.items()}
        x, u, y, status = autograd.factor_solve(lqr, inp)
        return x[:, :batch], u[:, :batch], y[:, :batch]

    assert torch.autograd.gradcheck(f, leaves, eps=1e-6, atol=1e-7, rtol=1e-6)


def test_composite_loss_backward_matches_reference():
    n, m, T, batch = 6, 2, 8, 37
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=13, dense_M=True)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    inp = lqr.pack_input(host)
    for k in inp:
        inp[k].requires_grad_(True)
    x, u, y, status = autograd.factor_solve(lqr, inp)
    assert not status.requires_grad
    # only x and u enter the loss (y's cotangent arrives as None), x through a .sum()
    loss = (x[:, :batch] ** 2).sum() + 3.0 * u[:, :batch].sum()
    loss.backward()
    sol = lqr.unpack_output(dict(x=x.detach(), u=u.detach(), y=y.detach()))
    cot = dict(x=2.0 * sol["x"], u=np.full_like(sol["u"], 3.0), y=np.zeros_like(sol["y"]))
    ref = lqr_vjp(s, host, pyoracle.lqr_factor_solve(s, host), cot)
    for k in GRAD_NAMES:
        got = e.unpack(inp[k].grad, e.lqr_sizes[k])
        assert rel_err(got, ref[k]).max() <= _tol(k), k
        assert not inp[k].grad[:, batch:].any(), k
