"""sipoc_lqr_jvp / sipoc_kkt_jvp (the forward-mode derivatives of the LQR and Newton-KKT solves)
against the CPU reference JVPs (jvp_reference.py) on every plan family, plus their contract:
NULL tangents, zeros in failed problems and padding lanes, bitwise repeatable (eager and graph
replay), no state carried from the forward, the adjoint identity against the VJPs, and the
torch.autograd bindings in forward mode (gradcheck, torch.func.jvp, forward_ad dual tensors).

Three checks per case, split so that a difference is attributed to the right stage:
- rhs (the tangent right-hand side t) against the reference formula evaluated on the GPU's own
  forward solution: no solve in between, so 1e-13 of the magnitude of the terms of each row;
- dsol against the oracle's solve of the GPU's own rhs at REL_TOL, the bar the forward and VJP
  tests hold on the same cases (r2 = 1e9 included);
- dsol against the full CPU reference (its own forward, rhs and solve) at REL_TOL where the
  problem is well conditioned: a reordered rhs moves dsol by the condition number."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
import test_gpu_kkt_vjp as gkv
from gpu_helpers import REL_TOL, rel_err, to_structs
from jvp_reference import kkt_jvp, kkt_tangent_rhs, lqr_jvp, lqr_tangent_rhs
from kkt_vjp_reference import MODEL_NAMES, THETA_NAMES, kkt_solve
from oracle import pyoracle
from oracle.pyoracle import Structure
from sip_optimal_control_b200 import LQR, _capi, autograd
from sip_optimal_control_b200._capi import lib
from sip_optimal_control_b200.kkt import _model_struct
from test_gpu_fuzz import random_structure
from test_gpu_kkt import _uniform_kkt_structure
from vjp_reference import GRAD_NAMES

pytestmark = pytest.mark.gpu

RHS_TOL = 1e-13
XUY = ("x", "u", "y")
QRC = ("q", "r", "c")
REG = gkv.REG


def _assert_rhs(got, ref, mag, what):
    bad = np.abs(got - ref) > RHS_TOL * mag
    assert not bad.any(), (what, float(np.max(np.abs(got - ref) / np.maximum(mag, 1e-300))))


# ---- LQR -----------------------------------------------------------------------------------

def _ltan(s, batch, seed, names=GRAD_NAMES):
    sz = pyoracle.lqr_sizes(s)
    rng = np.random.default_rng(seed)
    return {k: rng.standard_normal((batch, sz[k])) for k in names}


def _lqr_mag(s, sol, tan):
    """Per-row sum of the magnitudes of the terms of t."""
    a = {k: np.abs(v) for k, v in tan.items()}
    if "delta" in a:
        a["delta"] = -a["delta"]  # t_y = dc - ddelta .* y
    return lqr_tangent_rhs(s, {k: np.abs(sol[k]) for k in XUY}, a)


def _lqr(s, batch, **kw):
    dims, topo = to_structs(s)
    return LQR(dims, topo, batch, **kw)


def _lqr_check(s, host, tan, tol=REL_TOL, **kw):
    batch = host["q"].shape[0]
    lqr = _lqr(s, batch, **kw)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    res = lqr.jvp(inp, out, {k: e.pack(v) for k, v in tan.items()})
    assert (res["status"][:batch] == 0).all(), e.kernel_variant
    gsol = lqr.unpack_output(out)
    rhs = {k: e.unpack(res["rhs"][k], e.lqr_sizes[k]) for k in QRC}
    ref_rhs, mag = lqr_tangent_rhs(s, gsol, tan), _lqr_mag(s, gsol, tan)
    for k in QRC:
        _assert_rhs(rhs[k], ref_rhs[k], mag[k], (k, e.kernel_variant))
    dsol = lqr.unpack_output(res)
    own = pyoracle.lqr_factor_solve(s, {**host, **rhs}, residual=False)
    ref = lqr_jvp(s, host, pyoracle.lqr_factor_solve(s, host), tan)
    for k in XUY:
        if dsol[k].shape[1]:
            assert rel_err(dsol[k], own[k]).max() <= tol, (k, e.kernel_variant)
            assert rel_err(dsol[k], ref[k]).max() <= tol, (k, e.kernel_variant)
    return lqr


@pytest.mark.parametrize("n,m,T,family", [(4, 1, 20, "thread"), (12, 4, 10, "subwarp"),
                                          (16, 4, 6, "cta"), (64, 24, 3, "cta")])
def test_lqr_plan_families(n, m, T, family):
    batch = 37
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=n + T, dense_M=True)
    lqr = _lqr_check(s, host, _ltan(s, batch, 1))
    assert "generic" not in lqr.engine.kernel_variant, lqr.engine.kernel_variant


def test_lqr_two_kernel_subwarp_pair_large_batch():
    # above 40 960 problems the sub-warp plan runs the sweep and the rollout as two kernels
    n, m, T, batch = 12, 4, 3, 41000
    s = Structure.chain(T, n, m)
    lqr = _lqr(s, batch)
    e = lqr.engine
    inp = lqr.generate_benchmark(seed=5)
    out = lqr.alloc_output()
    lqr.factor_solve(inp, out)
    gen = torch.Generator(device=e.torch_device()).manual_seed(6)
    tan = {k: torch.randn(inp[k].shape, generator=gen, dtype=torch.float64,
                          device=e.torch_device()) for k in GRAD_NAMES}
    res = lqr.jvp(inp, out, tan)
    torch.cuda.synchronize()
    assert (res["status"][:batch] == 0).all()
    idx = torch.from_numpy(np.random.default_rng(7).choice(batch, 64, replace=False)).to(
        e.torch_device())
    sample = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: sample(inp[k], e.lqr_sizes[k]) for k in GRAD_NAMES}
    htan = {k: sample(tan[k], e.lqr_sizes[k]) for k in GRAD_NAMES}
    ref = lqr_jvp(s, host, pyoracle.lqr_factor_solve(s, host), htan)
    for k in XUY:
        assert rel_err(sample(res[k], e.lqr_sizes[k]), ref[k]).max() <= REL_TOL, k


@pytest.mark.parametrize("pad_variable_dims", [False, True])
def test_lqr_padded_variable_dims(pad_variable_dims):
    s = Structure.chain(6, [2, 1, 3, 2, 1, 3, 2], [1, 2, 1, 2, 1, 2])
    host = pg.variable_tree_batch(s, 40, seed=4)
    lqr = _lqr_check(s, host, _ltan(s, 40, 2), pad_variable_dims=pad_variable_dims)
    assert "generic" not in lqr.engine.kernel_variant


@pytest.mark.parametrize("builder", [fx.five_node_tree, fx.variable_dim_branch_tree])
def test_lqr_force_generic(builder):
    s, p = builder()
    host = {k: np.repeat(v, 5, axis=0) for k, v in fx.pack_problem(**p).items()}
    lqr = _lqr_check(s, host, _ltan(s, 5, 3), force_generic=True)
    assert "generic" in lqr.engine.kernel_variant


@pytest.mark.parametrize("seed", range(8))
def test_lqr_random_trees(seed):
    rng = np.random.default_rng(4000 + seed)
    s = random_structure(rng)
    batch = int(rng.integers(1, 71))
    host = pg.variable_tree_batch(s, batch, seed=seed)
    for force_generic in (False, True):
        _lqr_check(s, host, _ltan(s, batch, seed), force_generic=force_generic)


def test_lqr_forced_scan():
    # the scan's own tolerance (test_gpu_scan.py): REL_TOL on (x, u, y)
    n, m, T, batch = 12, 4, 64, 19
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=T + n, dense_M=True)
    lqr = _lqr_check(s, host, _ltan(s, batch, 4), parallel_in_time=True)
    assert lqr.engine.kernel_variant.startswith("scan_")


def _lqr_call(lqr, inp, out, tan, rhs, dsol, status, stream=None):
    e = lqr.engine
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in GRAD_NAMES])
    st = _capi.LqrInput(*[tan[k].data_ptr() if k in tan else None for k in GRAD_NAMES])
    so, sr, sd = (_capi.LqrOutput(*[d[k].data_ptr() for k in keys])
                  for d, keys in ((out, XUY), (rhs, QRC), (dsol, XUY)))
    e._check(lib.sipoc_lqr_jvp(e._handle, ctypes.byref(si), ctypes.byref(so), ctypes.byref(st),
                               ctypes.byref(sr), ctypes.byref(sd),
                               None if status is None else status.data_ptr(),
                               e.stream_ptr(stream)))


def _lqr_device_case(n=12, m=4, T=10, batch=37, seed=9, **kw):
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=seed, dense_M=True)
    lqr = _lqr(s, batch, **kw)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    tan = {k: e.pack(v) for k, v in _ltan(s, batch, 8).items()}
    return s, host, lqr, inp, out, tan


def test_lqr_null_tangents_equal_zero_tangents():
    s, host, lqr, inp, out, tan = _lqr_device_case()
    for part in (("q", "c"), ("Q", "B", "delta"), ("M", "R", "r", "A")):
        a = lqr.jvp(inp, out, {k: tan[k] for k in part})
        b = lqr.jvp(inp, out, {k: tan[k] if k in part else torch.zeros_like(tan[k])
                               for k in GRAD_NAMES})
        for k in XUY:
            assert torch.equal(a[k], b[k]), (part, k)
        for k in QRC:
            assert torch.equal(a["rhs"][k], b["rhs"][k]), (part, k)
    none = lqr.jvp(inp, out, {})
    for k in XUY:
        assert not none[k].any(), k
    for k in QRC:
        assert not none["rhs"][k].any(), k


@pytest.mark.parametrize("force_generic", [True, False])
def test_lqr_failed_problems_and_padding_lanes_are_zero(force_generic):
    n, m, T, batch = 2, 1, 2, 6
    s, host = pg.lqr_benchmark_batch(n, m, T, batch, seed=10, dense_M=True)
    # the failures of test_gpu_vjp.py's test of the same name
    host["delta"][1, T * n + 0] = 0.0
    host["Q"][2, T * n * n:] = (-2.0 * np.eye(n)).flatten()
    host["delta"][2, T * n:] = 1.0
    host["Q"][3, T * n * n:] = 0.0
    host["R"][3, (T - 1) * m * m] = -1.0
    host["delta"][4, 1] = -1.0
    host["R"][4, (T - 1) * m * m] = -50.0
    ref_sol = pyoracle.lqr_factor_solve(s, host)
    assert ref_sol["status"].tolist() == [0, 1, 2, 3, 3, 0]
    tan = _ltan(s, batch, 11)
    ref = lqr_jvp(s, host, ref_sol, tan)
    lqr = _lqr(s, batch, force_generic=force_generic)
    e = lqr.engine
    inp, out = lqr.pack_input(host), lqr.alloc_output()
    lqr.factor_solve(inp, out)
    dsol = {k: torch.full_like(out[k], float("nan")) for k in XUY}
    res = lqr.jvp(inp, out, {k: e.pack(v) for k, v in tan.items()}, dsol=dsol)
    assert res["status"][:batch].cpu().tolist() == [0, 1, 2, 3, 3, 0]
    good = ref_sol["status"] == 0
    for k in XUY:
        full = res[k][: e.lqr_sizes[k]].cpu().numpy()  # [size, batch_stride]
        assert not full[:, batch:].any(), k            # padding lanes
        assert not full[:, :batch][:, ~good].any(), k  # failed problems
        assert rel_err(full[:, :batch].T[good], ref[k][good]).max() <= REL_TOL, k
    for k in QRC:
        assert not res["rhs"][k][:, batch:].any(), k


def test_lqr_bitwise_repeatable_and_graph_replay():
    s, host, lqr, inp, out, tan = _lqr_device_case()
    e = lqr.engine
    side = torch.cuda.Stream()
    bufs = lambda: ({k: e.empty(e.lqr_sizes[k]) for k in QRC}, lqr.alloc_output())
    (r1, d1), (r2, d2) = bufs(), bufs()
    status = e.empty_int()
    torch.cuda.synchronize()
    _lqr_call(lqr, inp, out, tan, r1, d1, status, stream=side)
    _lqr_call(lqr, inp, out, tan, r2, d2, status, stream=side)
    side.synchronize()
    for k in XUY:
        assert torch.equal(d1[k], d2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _lqr_call(lqr, inp, out, tan, r2, d2, status, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for d in (r2, d2):
        for v in d.values():
            v.fill_(float("nan"))
    torch.cuda.synchronize()
    before = e.launch_count
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    assert e.launch_count == before + lib.sipoc_graph_kernel_count(graph)
    for k in XUY:
        assert torch.equal(d1[k], d2[k]), k
    for k in QRC:
        assert torch.equal(r1[k], r2[k]), k
    lib.sipoc_graph_destroy(graph)


def test_lqr_another_factorization_between_forward_and_jvp():
    s, host, lqr, inp, out, tan = _lqr_device_case()
    first = lqr.jvp(inp, out, tan)
    _, other = pg.lqr_benchmark_batch(12, 4, 10, 37, seed=99, dense_M=True)
    lqr.factor_solve(lqr.pack_input(other), lqr.alloc_output())
    second = lqr.jvp(inp, out, tan)
    for k in XUY:
        assert torch.equal(first[k], second[k]), k


def test_lqr_adjoint_identity_against_vjp():
    s, host, lqr, inp, out, tan = _lqr_device_case(batch=33)  # Q, R tangents not symmetric
    e = lqr.engine
    gen = np.random.default_rng(14)
    cot = {k: e.pack(gen.standard_normal((33, e.lqr_sizes[k]))) for k in XUY}
    fwd = lqr.jvp(inp, out, tan)
    rev = lqr.vjp(inp, out, cot)
    lhs = sum((fwd[k][:, :33] * cot[k][:, :33]).sum(0) for k in XUY)
    terms = [tan[k][:, :33] * rev[k][:, :33] for k in GRAD_NAMES]
    rhs = sum(t.sum(0) for t in terms)
    scale = torch.maximum(lhs.abs(), sum(t.abs().sum(0) for t in terms))
    assert ((lhs - rhs).abs() <= 1e-12 * scale).all(), float(((lhs - rhs).abs() / scale).max())


def _lqr_tiny():
    s, p = fx.variable_dim_branch_tree()
    batch = 3
    rng = np.random.default_rng(12)
    host = {k: np.repeat(v, batch, axis=0) for k, v in fx.pack_problem(**p).items()}
    for k in QRC:
        host[k] = host[k] + 0.1 * rng.standard_normal(host[k].shape)
    return s, host, batch


def _lqr_binding(s, host, batch):
    """f(*leaves) -> (x, u, y) of the live lanes through autograd.factor_solve, Q and R formed
    symmetric from free tensors; the padding lanes solve copies of problem 0."""
    lqr = _lqr(s, batch)
    ld, dev = lqr.engine.batch_stride, lqr.engine.torch_device()
    permQ = gkv._block_transpose([int(v) for v in s.state_dims]).to(dev)
    permR = gkv._block_transpose([int(v) for v in s.control_dims]).to(dev)

    def f(*arrays):
        a = dict(zip(GRAD_NAMES, arrays))
        a["Q"] = 0.5 * (a["Q"] + a["Q"].index_select(0, permQ))
        a["R"] = 0.5 * (a["R"] + a["R"].index_select(0, permR))
        inp = {k: torch.cat([v, v[:, :1].expand(-1, ld - batch)], dim=1) for k, v in a.items()}
        x, u, y, status = autograd.factor_solve(lqr, inp)
        return x[:, :batch], u[:, :batch], y[:, :batch]

    leaves = [torch.tensor(host[k].T, dtype=torch.float64, device=dev) for k in GRAD_NAMES]
    return f, leaves


def test_lqr_gradcheck_forward_and_backward():
    s, host, batch = _lqr_tiny()
    f, leaves = _lqr_binding(s, host, batch)
    leaves = [v.requires_grad_(True) for v in leaves]
    assert torch.autograd.gradcheck(f, leaves, eps=1e-6, atol=1e-7, rtol=1e-6,
                                    check_forward_ad=True, check_backward_ad=True)


def test_lqr_func_jvp_and_dual_tensors_match_reference():
    s, host, batch = _lqr_tiny()
    f, leaves = _lqr_binding(s, host, batch)
    tan = _ltan(s, batch, 15)
    tans = [torch.tensor(tan[k].T, dtype=torch.float64, device=leaves[0].device)
            for k in GRAD_NAMES]
    # the binding symmetrizes Q, R: the reference sees the symmetric parts, which is also what
    # the unsymmetrized tangents give (the convention of sipoc_lqr_jvp)
    ref = lqr_jvp(s, host, pyoracle.lqr_factor_solve(s, host), tan)
    composite = lambda *a: sum((v ** 2).sum(0) for v in f(*a))  # per problem: sum of squares
    _, dc = torch.func.jvp(composite, tuple(leaves), tuple(tans))
    sol = [v.cpu().numpy() for v in f(*leaves)]
    want = sum(2.0 * (sv.T * ref[k]).sum(1) for sv, k in zip(sol, XUY))
    assert np.abs(dc.cpu().numpy() - want).max() <= 1e-9 * max(1.0, np.abs(want).max())
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        duals = [fwAD.make_dual(p, t) for p, t in zip(leaves, tans)]
        outs = f(*duals)
        for o, k in zip(outs, XUY):
            got = fwAD.unpack_dual(o).tangent.cpu().numpy().T
            if got.shape[1]:
                assert rel_err(got, ref[k]).max() <= REL_TOL, k


# ---- Newton-KKT ----------------------------------------------------------------------------

def _ktan(pb, seed, names=None):
    rng = np.random.default_rng(seed)
    names = [k for k in (names or gkv._names(pb.p)) if gkv._size(pb.cp, k)]
    return {k: rng.standard_normal((pb.batch, gkv._size(pb.cp, k))) for k in names}


def _kkt_jvp(pb, tan, **kw):
    e = pb.cp.engine
    return pb.cp.jvp(pb.dm, *(pb.dev[k] for k in REG), pb.sol,
                     {k: e.pack(v) if isinstance(v, np.ndarray) else v for k, v in tan.items()},
                     **kw)


def _kkt_mag(s, p, sol, tan):
    """Per-row sum of the magnitudes of the terms of t."""
    neg = set(MODEL_NAMES) | set(THETA_NAMES) | {"r1"}  # t = db - dK sol: dr1 enters with -
    return kkt_tangent_rhs(s, p, np.abs(sol),
                           {k: -np.abs(v) if k in neg else np.abs(v) for k, v in tan.items()})


def _kkt_check(pb, seed=0, tol=REL_TOL, full=True):
    e, h = pb.cp.engine, pb.host
    kd = h["b"].shape[1]
    tan = _ktan(pb, seed)
    res = _kkt_jvp(pb, tan)
    ok = res["ok"][:pb.batch].cpu().numpy()
    assert (ok == pb.ok[:pb.batch].cpu().numpy()).all()
    good = ok == 1
    gsol = e.unpack(pb.sol, kd)
    rhs = e.unpack(res["rhs"], kd)
    _assert_rhs(rhs[good], kkt_tangent_rhs(pb.s, pb.p, gsol, tan)[good],
                _kkt_mag(pb.s, pb.p, gsol, tan)[good], e.kernel_variant)
    dsol = e.unpack(res["sol"], kd)
    assert not dsol[~good].any()
    reg = [h[k] for k in REG]
    own = kkt_solve(pb.s, pb.p, pb.model, pb.theta, *reg, rhs)
    assert rel_err(dsol[good], own["sol"][good]).max() <= tol, e.kernel_variant
    if full:
        ref_sol = kkt_solve(pb.s, pb.p, pb.model, pb.theta, *reg, h["b"])
        ref = kkt_jvp(pb.s, pb.p, pb.model, pb.theta, *reg, ref_sol["sol"], tan)
        assert (ref["ok"] == ok).all()
        assert rel_err(dsol[good], ref["sol"][good]).max() <= tol, e.kernel_variant
    return res


@pytest.mark.parametrize("case", ["chain", "siblings", "zero_dim_root", "schur"])
@pytest.mark.parametrize("force_generic", [True, False])
def test_kkt_reference_fixtures(case, force_generic):
    if case == "schur":
        pb = gkv._schur_problem(force_generic=force_generic)
    else:
        pb = gkv._fixture_problem(getattr(fx, f"kkt_case_{case}"), force_generic=force_generic)
    assert pb.ok[:pb.batch].all()
    _kkt_check(pb)


@pytest.mark.parametrize("n,m,T", [(4, 1, 16), (12, 4, 12), (6, 2, 20), (8, 3, 9), (16, 4, 6),
                                   (32, 8, 3)])
@pytest.mark.parametrize("force_generic", [True, False])
@pytest.mark.parametrize("r2_max", [1e3, 1e9])
def test_kkt_newton_benchmark_shapes(n, m, T, force_generic, r2_max):
    s = _uniform_kkt_structure(n, m, T)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 33, seed=n * 100 + m, r2_max=r2_max)
    pb = gkv.Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=n, force_generic=force_generic)
    if not force_generic:
        assert "generic" not in pb.cp.engine.kernel_variant, pb.cp.engine.kernel_variant
    _kkt_check(pb, seed=n, full=r2_max < 1e6)


def test_kkt_fused_solve_path_large_batch():
    # above the dispatch threshold the uniform-chain solve runs the fused kernels
    n, m, T, batch = 4, 1, 6, 32768 + 5
    s = _uniform_kkt_structure(n, m, T)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=21, r2_max=1e9)
    pb = gkv.Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=22)
    e = pb.cp.engine
    assert "generic" not in e.kernel_variant
    tan = _ktan(pb, 23)
    res = _kkt_jvp(pb, tan)
    kd = rhs.shape[1]
    sample = np.r_[0:64, batch - 64:batch]
    sub = lambda a: a[sample]
    h = pb.host
    sm = {k: sub(v) for k, v in model.items()}
    reg = [sub(h[k]) for k in REG]
    ok = res["ok"][:batch].cpu().numpy()[sample]
    good = ok == 1
    assert good.sum() >= sample.size - 4
    gsol = sub(e.unpack(pb.sol, kd))
    stan = {k: sub(v) for k, v in tan.items()}
    rhs_g = sub(e.unpack(res["rhs"], kd))
    _assert_rhs(rhs_g[good], kkt_tangent_rhs(s, 0, gsol, stan)[good],
                _kkt_mag(s, 0, gsol, stan)[good], e.kernel_variant)
    dsol = sub(e.unpack(res["sol"], kd))
    own = kkt_solve(s, 0, sm, None, *reg, rhs_g)
    assert rel_err(dsol[good], own["sol"][good]).max() <= REL_TOL
    assert not dsol[~good].any()


@pytest.mark.parametrize("pad_variable_dims,variant", [(False, "padded_to_strict_thread_n3_m2"),
                                                       (True, "padded_to_subwarp4_n6_m2")])
@pytest.mark.parametrize("r2_max", [1e3, 1e9])
def test_kkt_config4_variable_dims(pad_variable_dims, variant, r2_max):
    s = gkv._config4()
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 50, seed=9, r2_max=r2_max)
    pb = gkv.Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=3,
                     pad_variable_dims=pad_variable_dims)
    assert pb.cp.engine.kernel_variant == variant
    _kkt_check(pb, seed=4, full=r2_max < 1e6)


@pytest.mark.parametrize("n,m,T,p", [(4, 1, 16, 4), (12, 4, 10, 8), (6, 2, 12, 4)])
@pytest.mark.parametrize("force_generic", [True, False])
def test_kkt_theta_shapes(n, m, T, p, force_generic):
    c, g = max(1, n // 2), max(1, 2 * m)
    s = Structure.chain(T, n, m, node_c=[0] * T + [c], node_g=[0] * T + [g], edge_c=[c] * T,
                        edge_g=[g] * T)
    model, theta, w, r1, r2, r3, rhs = pg.newton_kkt_theta_batch(s, p, 21, seed=n + p,
                                                                 r2_max=1e9)
    pb = gkv.Problem(s, p, model, theta, w, r1, r2, r3, rhs, seed=p, force_generic=force_generic)
    _kkt_check(pb, seed=p, full=False)


def test_kkt_theta_on_a_variable_dimension_tree():
    s = Structure([0, 0, 1, 1], [1, 2, 3, 4], 0, [3, 1, 2, 4, 2], [2, 1, 3, 1],
                  node_c=[1, 0, 2, 0, 1], node_g=[0, 2, 1, 1, 0], edge_c=[1, 0, 2, 1],
                  edge_g=[2, 1, 0, 1])
    model, theta, w, r1, r2, r3, rhs = pg.newton_kkt_theta_batch(s, 3, 9, seed=5, r2_max=1e3)
    _kkt_check(gkv.Problem(s, 3, model, theta, w, r1, r2, r3, rhs, seed=6))


def test_kkt_null_tangents_equal_zero_tangents():
    pb = gkv._schur_problem(batch=37)
    e = pb.cp.engine
    tan = {k: e.pack(v) for k, v in _ktan(pb, 30).items()}
    for part in (("b", "r1"), ("node_hxx", "edge_A", "node_htt", "w"),
                 ("edge_dynt", "edge_hut", "r2", "r3", "node_jg")):
        part = [k for k in part if k in tan]
        a = _kkt_jvp(pb, {k: tan[k] for k in part})
        b = _kkt_jvp(pb, {k: tan[k] if k in part else torch.zeros_like(v) for k, v in tan.items()})
        assert torch.equal(a["rhs"], b["rhs"]) and torch.equal(a["sol"], b["sol"]), part
    none = _kkt_jvp(pb, {})
    assert not none["rhs"].any() and not none["sol"].any()


@pytest.mark.parametrize("force_generic", [True, False])
def test_kkt_failed_problems_and_padding_lanes_are_zero(force_generic):
    pb = gkv._fixture_problem(fx.kkt_case_chain, batch=4, force_generic=force_generic)
    pb.host["r2"][1, 2] = 0.0  # non-positive r2: the factor rejects the problem
    pb.dev["r2"] = pb.cp.engine.pack(pb.host["r2"])
    e = pb.cp.engine
    dsol = torch.full_like(pb.sol, float("nan"))
    res = _kkt_jvp(pb, _ktan(pb, 31), dsol=dsol)
    assert res["ok"][:pb.batch].cpu().tolist() == [1, 0, 1, 1]
    full = res["sol"].cpu().numpy()
    assert not full[:, pb.batch:].any() and not full[:, 1].any()
    assert full[:, [0, 2, 3]].any(axis=0).all()
    assert not res["rhs"][:, pb.batch:].any()


def _kkt_call(pb, tan, rhs, dsol, ok, stream=None):
    e = pb.cp.engine
    sm = _model_struct(pb.dm, False, [])
    st = _capi.KktTangent()
    for k in _capi.KKT_MODEL_FIELDS:
        setattr(st.model, k, tan[k].data_ptr() if k in tan else None)
    for k in _capi.KKT_VECTOR_GRAD_FIELDS:
        setattr(st, k, tan[k].data_ptr() if k in tan else None)
    tt = _capi.KktThetaModel()
    for k in _capi.KKT_THETA_FIELDS:
        setattr(tt, k, tan[k].data_ptr() if k in tan else None)
    st.model.theta = ctypes.pointer(tt)
    e._check(lib.sipoc_kkt_jvp(e._handle, ctypes.byref(sm),
                               *(pb.dev[k].data_ptr() for k in REG), pb.sol.data_ptr(),
                               ctypes.byref(st), rhs.data_ptr(), dsol.data_ptr(), ok.data_ptr(),
                               e.stream_ptr(stream)))


def test_kkt_bitwise_repeatable_and_graph_replay():
    pb = gkv._schur_problem(batch=37)
    e = pb.cp.engine
    tan = {k: e.pack(v) for k, v in _ktan(pb, 32).items()}
    kd = gkv._size(pb.cp, "b")
    side = torch.cuda.Stream()
    r1, d1, r2, d2 = (e.empty(kd) for _ in range(4))
    ok = e.empty_int()
    torch.cuda.synchronize()
    _kkt_call(pb, tan, r1, d1, ok, stream=side)
    _kkt_call(pb, tan, r2, d2, ok, stream=side)
    side.synchronize()
    assert torch.equal(r1, r2) and torch.equal(d1, d2)
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _kkt_call(pb, tan, r2, d2, ok, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    r2.fill_(float("nan"))
    d2.fill_(float("nan"))
    torch.cuda.synchronize()
    before = e.launch_count
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    assert e.launch_count == before + lib.sipoc_graph_kernel_count(graph)
    assert torch.equal(r1, r2) and torch.equal(d1, d2)
    lib.sipoc_graph_destroy(graph)


def test_kkt_another_factorization_between_forward_and_jvp():
    s = _uniform_kkt_structure(6, 2, 10)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 40, seed=31, r2_max=1e3)
    pb = gkv.Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=32)
    e = pb.cp.engine
    tan = {k: e.pack(v) for k, v in _ktan(pb, 33).items()}
    first = _kkt_jvp(pb, tan)
    other, ow, or1, or2, or3, orhs = pg.newton_kkt_batch(s, 40, seed=33, r2_max=1e3)
    dm2 = pb.cp.pack_model(other)
    pb.cp.factor(dm2, *(e.pack(a) for a in (ow, or1, or2, or3)))
    pb.cp.solve(dm2, e.pack(orhs), e.zeros(rhs.shape[1]))
    second = _kkt_jvp(pb, tan)
    assert torch.equal(first["sol"], second["sol"]) and torch.equal(first["rhs"], second["rhs"])


def test_kkt_adjoint_identity_against_vjp():
    pb = gkv._schur_problem(batch=33)  # Hessian tangents not symmetric
    e = pb.cp.engine
    B = pb.batch
    tan = {k: e.pack(v) for k, v in _ktan(pb, 34).items()}
    fwd = _kkt_jvp(pb, tan)
    rev = pb.vjp()
    lhs = (fwd["sol"][:, :B] * pb.cot[:, :B]).sum(0)
    terms = [tan[k][:, :B] * rev[k][:, :B] for k in tan]
    rhs = sum(t.sum(0) for t in terms)
    scale = torch.maximum(lhs.abs(), sum(t.abs().sum(0) for t in terms))
    assert ((lhs - rhs).abs() <= 1e-12 * scale).all(), float(((lhs - rhs).abs() / scale).max())


def _kkt_binding(pb, names):
    batch = pb.batch
    cp, e = pb.cp, pb.cp.engine
    ld, dev = e.batch_stride, e.torch_device()
    perm = gkv._block_transpose([int(v) for v in pb.s.state_dims]).to(dev)
    const = {**pb.dm, **pb.dev}

    def f(*arrays):
        a = dict(zip(names, arrays))
        if "node_hxx" in a:
            a["node_hxx"] = 0.5 * (a["node_hxx"] + a["node_hxx"].index_select(0, perm))
        full = {k: torch.cat([v, v[:, :1].expand(-1, ld - batch)], dim=1) for k, v in a.items()}
        arg = {**const, **full}
        model = {k: arg[k] for k in MODEL_NAMES + (THETA_NAMES if pb.p else ())}
        sol, ok = autograd.kkt_factor_solve(cp, model, *(arg[k] for k in REG), arg["b"])
        return sol[:, :batch]

    return f, [const[k][:, :batch].clone() for k in names]


def test_kkt_gradcheck_forward_and_backward():
    pb = gkv._schur_problem(batch=2, seed=5)
    names = ("b", "r2", "w", "edge_A", "node_jg", "node_hxx", "edge_dynt")
    f, leaves = _kkt_binding(pb, names)
    leaves = [v.requires_grad_(True) for v in leaves]
    assert torch.autograd.gradcheck(f, leaves, eps=1e-6, atol=1e-7, rtol=1e-6,
                                    check_forward_ad=True, check_backward_ad=True)


def test_kkt_func_jvp_and_dual_tensors_match_reference():
    pb = gkv._schur_problem(batch=3, seed=7)
    names = ("b", "r1", "r3", "edge_B", "node_hxx", "edge_htt", "node_hxt")
    f, leaves = _kkt_binding(pb, names)
    tan = _ktan(pb, 35, names)
    dev = leaves[0].device
    tans = [torch.tensor(tan[k].T, dtype=torch.float64, device=dev) for k in names]
    h = pb.host
    reg = [h[k] for k in REG]
    ref_sol = kkt_solve(pb.s, pb.p, pb.model, pb.theta, *reg, h["b"])
    ref = kkt_jvp(pb.s, pb.p, pb.model, pb.theta, *reg, ref_sol["sol"], tan)["sol"]
    _, dc = torch.func.jvp(lambda *a: (f(*a) ** 2).sum(0), tuple(leaves), tuple(tans))
    want = 2.0 * (ref_sol["sol"] * ref).sum(1)
    assert np.abs(dc.cpu().numpy() - want).max() <= 1e-9 * max(1.0, np.abs(want).max())
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        out = f(*[fwAD.make_dual(p, t) for p, t in zip(leaves, tans)])
        got = fwAD.unpack_dual(out).tangent.cpu().numpy().T
    assert rel_err(got, ref).max() <= REL_TOL
