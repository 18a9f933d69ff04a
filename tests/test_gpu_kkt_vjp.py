"""sipoc_kkt_vjp (the reverse-mode derivative of the Newton-KKT solve) against the CPU reference
VJP (kkt_vjp_reference.py) on the generic and default plans, the benchmark shapes, the fused
solve, padded variable dims and theta, plus its contract: NULL arrays untouched, zeros in
failed problems and padding lanes, bitwise repeatable (eager and graph replay), no state
carried from the forward, and the torch.autograd binding (gradcheck, a composite loss).

Tolerance: REL_TOL (1e-9 relative per problem and array) on the adjoint and b, which is the
adjoint itself; 2 * REL_TOL on every other array, each a sum of products of a 1e-9-accurate
solution entry with a 1e-9-accurate adjoint entry."""
import ctypes

import numpy as np
import pytest
import torch

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err
from kkt_vjp_reference import MODEL_NAMES, THETA_NAMES, VECTOR_NAMES, kkt_solve, kkt_vjp
from oracle import pyoracle
from oracle.pyoracle import Structure
from sip_optimal_control_b200 import CallbackProvider, Dimensions, Topology, _capi, autograd
from sip_optimal_control_b200._capi import lib
from test_gpu_kkt import _uniform_kkt_structure

pytestmark = pytest.mark.gpu

REG = ("w", "r1", "r2", "r3")


def _names(p):
    return MODEL_NAMES + (THETA_NAMES if p else ()) + VECTOR_NAMES


def _tol(k, tol=REL_TOL):
    return tol if k == "b" else 2 * tol


def _provider(s, p, batch, **kw):
    topo = Topology(s.num_edges, s.root, s.parents, s.children)
    dims = Dimensions(p, s.state_dims, s.control_dims, s.node_c, s.node_g, s.edge_c, s.edge_g)
    return CallbackProvider(dims, topo, batch, **kw)


def _size(cp, k):
    z = cp.sizes
    return dict(b=z["kkt_dim"], w=z["z_dim"], r1=z["x_dim"], r2=z["y_dim"],
                r3=z["z_dim"]).get(k, z.get(k))


class Problem:
    """A batch on the device: model, regularization, rhs, the forward's ok and sol, and a
    cotangent."""

    def __init__(self, s, p, model, theta, w, r1, r2, r3, rhs, seed=0, **kw):
        self.s, self.p, self.model, self.theta = s, p, model, theta
        self.host = dict(w=w, r1=r1, r2=r2, r3=r3, b=rhs)
        self.batch = rhs.shape[0]
        self.cp = cp = _provider(s, p, self.batch, **kw)
        e = cp.engine
        self.dm = cp.pack_model({**model, **(theta or {})})
        self.dev = {k: e.pack(v) for k, v in self.host.items()}
        self.ok = cp.factor(self.dm, *(self.dev[k] for k in REG))
        self.sol = e.zeros(rhs.shape[1])
        cp.solve(self.dm, self.dev["b"], self.sol)
        self.hcot = np.random.default_rng(seed).standard_normal(rhs.shape)
        self.cot = e.pack(self.hcot)

    def vjp(self, **kw):
        return self.cp.vjp(self.dm, *(self.dev[k] for k in REG), self.sol, self.cot, **kw)

    def reference(self):
        h = self.host
        ref_sol = kkt_solve(self.s, self.p, self.model, self.theta, h["w"], h["r1"], h["r2"],
                            h["r3"], h["b"])
        return kkt_vjp(self.s, self.p, self.model, self.theta, h["w"], h["r1"], h["r2"],
                       h["r3"], ref_sol["sol"], self.hcot)


def _check(pb: Problem, tol=REL_TOL):
    ref = pb.reference()
    res = pb.vjp()
    e = pb.cp.engine
    ok = res["ok"][:pb.batch].cpu().numpy()
    assert (ok == ref["ok"]).all()
    assert (ok == pb.ok[:pb.batch].cpu().numpy()).all()
    good = ref["ok"] == 1
    adj = e.unpack(res["adjoint"], pb.host["b"].shape[1])
    assert rel_err(adj[good], ref["adjoint"][good]).max() <= tol, e.kernel_variant
    for k in _names(pb.p):
        n = _size(pb.cp, k)
        if n == 0:
            continue
        got = e.unpack(res[k], n)
        assert rel_err(got[good], ref[k][good]).max() <= _tol(k, tol), (k, e.kernel_variant)
        assert not got[~good].any(), k
    return res


def _fixture_problem(build, batch=5, seed=0, **kw):
    s = build()
    sz = pyoracle.kkt_sizes(s)
    rng = np.random.default_rng(seed)
    model = {k: np.repeat(v, batch, axis=0) * (1.0 + 0.1 * rng.standard_normal((batch, 1)))
             for k, v in fx.kkt_model(s).items()}
    w, r1, r2, r3, rhs = (np.repeat(a, batch, axis=0) for a in
                          fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"]))
    return Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=seed, **kw)


def _schur_problem(batch=5, seed=0, **kw):
    s, p, diag = fx.kkt_case_schur()
    sz = pyoracle.kkt_sizes(s)
    rep = lambda a: np.repeat(a, batch, axis=0)
    model = {k: rep(v) for k, v in fx.kkt_model(s).items()}
    theta = {k: rep(v) for k, v in fx.kkt_theta_model(s, p, diag).items()}
    rng = np.random.default_rng(seed)
    w, r1, r2, r3, rhs = (rep(a) for a in
                          fx.kkt_regularization(sz["x_dim"] + p, sz["y_dim"], sz["z_dim"]))
    rhs = rhs + 0.1 * rng.standard_normal(rhs.shape)
    return Problem(s, p, model, theta, w, r1, r2, r3, rhs, seed=seed, **kw)


@pytest.mark.parametrize("case", ["chain", "siblings", "zero_dim_root", "schur"])
@pytest.mark.parametrize("force_generic", [True, False])
def test_reference_fixtures(case, force_generic):
    if case == "schur":
        pb = _schur_problem(force_generic=force_generic)
    else:
        pb = _fixture_problem(getattr(fx, f"kkt_case_{case}"), force_generic=force_generic)
    assert pb.ok[:pb.batch].all()
    _check(pb)


@pytest.mark.parametrize("n,m,T", [(4, 1, 16), (12, 4, 12), (6, 2, 20), (8, 3, 9), (16, 4, 6),
                                   (32, 8, 3)])
@pytest.mark.parametrize("force_generic", [True, False])
@pytest.mark.parametrize("r2_max", [1e3, 1e9])
def test_newton_kkt_benchmark_shapes(n, m, T, force_generic, r2_max):
    s = _uniform_kkt_structure(n, m, T)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 33, seed=n * 100 + m, r2_max=r2_max)
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=n, force_generic=force_generic)
    if not force_generic:
        assert "generic" not in pb.cp.engine.kernel_variant, pb.cp.engine.kernel_variant
    _check(pb)


def test_fused_kkt_solve_path_large_batch():
    # above the dispatch threshold the uniform-chain solve of the adjoint runs the fused kernels
    n, m, T, batch = 4, 1, 6, 32768 + 5
    s = _uniform_kkt_structure(n, m, T)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=21, r2_max=1e9)
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=22)
    e = pb.cp.engine
    assert "generic" not in e.kernel_variant
    res = pb.vjp()
    sample = np.r_[0:64, batch - 64:batch]
    sub = lambda a: a[sample]
    h = pb.host
    sm = {k: sub(v) for k, v in model.items()}
    ref_sol = kkt_solve(s, 0, sm, None, *(sub(h[k]) for k in REG), sub(h["b"]))
    ref = kkt_vjp(s, 0, sm, None, *(sub(h[k]) for k in REG), ref_sol["sol"], sub(pb.hcot))
    good = ref["ok"] == 1
    assert good.sum() >= sample.size - 4
    assert (res["ok"][:batch].cpu().numpy()[sample] == ref["ok"]).all()
    for k in _names(0):
        got = e.unpack(res[k], _size(pb.cp, k))[sample]
        assert rel_err(got[good], ref[k][good]).max() <= _tol(k), k
        assert not got[~good].any(), k


def _config4(reps=6):
    sd = [2, 1, 3] * reps + [2]
    T = len(sd) - 1
    return Structure.chain(T, sd, ([1, 2, 1] * reps)[:T], node_c=([1, 0, 2] * reps + [1])[:T + 1],
                           node_g=([0, 2, 1] * reps + [0])[:T + 1], edge_c=([1, 2, 0] * reps)[:T],
                           edge_g=([2, 1, 1] * reps)[:T])


@pytest.mark.parametrize("pad_variable_dims,variant", [(False, "padded_to_strict_thread_n3_m2"),
                                                       (True, "padded_to_subwarp4_n6_m2")])
@pytest.mark.parametrize("r2_max", [1e3, 1e9])
def test_config4_variable_dims(pad_variable_dims, variant, r2_max):
    s = _config4()
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 50, seed=9, r2_max=r2_max)
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=3,
                 pad_variable_dims=pad_variable_dims)
    assert pb.cp.engine.kernel_variant == variant
    _check(pb)


@pytest.mark.parametrize("n,m,T,p", [(4, 1, 16, 4), (12, 4, 10, 8), (6, 2, 12, 4)])
@pytest.mark.parametrize("force_generic", [True, False])
def test_theta_shapes(n, m, T, p, force_generic):
    c, g = max(1, n // 2), max(1, 2 * m)
    s = Structure.chain(T, n, m, node_c=[0] * T + [c], node_g=[0] * T + [g], edge_c=[c] * T,
                        edge_g=[g] * T)
    model, theta, w, r1, r2, r3, rhs = pg.newton_kkt_theta_batch(s, p, 21, seed=n + p,
                                                                 r2_max=1e9)
    _check(Problem(s, p, model, theta, w, r1, r2, r3, rhs, seed=p, force_generic=force_generic))


def test_theta_on_a_variable_dimension_tree():
    s = Structure([0, 0, 1, 1], [1, 2, 3, 4], 0, [3, 1, 2, 4, 2], [2, 1, 3, 1],
                  node_c=[1, 0, 2, 0, 1], node_g=[0, 2, 1, 1, 0], edge_c=[1, 0, 2, 1],
                  edge_g=[2, 1, 0, 1])
    model, theta, w, r1, r2, r3, rhs = pg.newton_kkt_theta_batch(s, 3, 9, seed=5, r2_max=1e3)
    _check(Problem(s, 3, model, theta, w, r1, r2, r3, rhs, seed=6))


def _call(pb: Problem, grads: dict, adjoint, ok, stream=None):
    """sipoc_kkt_vjp through the C ABI with exactly the arrays of ``grads`` (theta = NULL when
    none of them is a theta block)."""
    from sip_optimal_control_b200.kkt import _model_struct

    e = pb.cp.engine
    keep = []
    m = _model_struct(pb.dm, False, keep)
    sg = _capi.KktGrad()
    for k in MODEL_NAMES + VECTOR_NAMES:
        setattr(sg, k, grads[k].data_ptr() if k in grads else None)
    if any(k in grads for k in THETA_NAMES):
        st = _capi.KktThetaGrad()
        for k in THETA_NAMES:
            setattr(st, k, grads[k].data_ptr() if k in grads else None)
        keep.append(st)
        sg.theta = ctypes.pointer(st)
    e._check(lib.sipoc_kkt_vjp(e._handle, ctypes.byref(m), *(pb.dev[k].data_ptr() for k in REG),
                               pb.sol.data_ptr(), pb.cot.data_ptr(), adjoint.data_ptr(),
                               ctypes.byref(sg), None if ok is None else ok.data_ptr(),
                               e.stream_ptr(stream)))


def _profiled_launches(e):
    launches = {}
    for i in range(lib.sipoc_profile_collect(e._handle)):
        nm, cnt = ctypes.c_char_p(), ctypes.c_int64()
        e._check(lib.sipoc_profile_get(e._handle, i, ctypes.byref(nm), None, ctypes.byref(cnt)))
        launches[nm.value.decode()] = cnt.value
    return launches


def test_only_requested_arrays_are_written():
    pb = _schur_problem(batch=7)
    e = pb.cp.engine
    names = _names(pb.p)
    full = pb.vjp()
    sentinel = 12345.5
    for want in (("b", "r2"), ("node_hxx", "edge_A", "w", "r3"), ("edge_dynt", "node_htt", "r1"),
                 ("edge_jgu", "node_jc", "edge_huu")):  # the last: theta = NULL
        arrays = {k: torch.full_like(full[k], sentinel) for k in names}
        _call(pb, {k: arrays[k] for k in want}, e.empty(_size(pb.cp, "b")), None)
        torch.cuda.synchronize()
        for k in names:
            if k in want:
                assert torch.equal(arrays[k], full[k]), k
            else:
                assert (arrays[k] == sentinel).all(), k
    # no gradient requested: the adjoint alone and no gradient kernel; one launch of it per
    # call that requests any
    lib.sipoc_profile_enable(e._handle, 1)
    adj = e.empty(_size(pb.cp, "b"))
    _call(pb, {}, adj, None)
    _call(pb, {"r2": torch.empty_like(full["r2"])}, e.empty(_size(pb.cp, "b")), None)
    launches = _profiled_launches(e)
    lib.sipoc_profile_enable(e._handle, 0)
    assert launches["kkt_vjp_kernel"] == 1, launches
    assert torch.equal(adj[:, :pb.batch], full["adjoint"][:, :pb.batch])


@pytest.mark.parametrize("force_generic", [True, False])
def test_failed_problems_and_padding_lanes_are_zero(force_generic):
    s = fx.kkt_case_chain()
    sz = pyoracle.kkt_sizes(s)
    batch = 4
    model = {k: np.repeat(v, batch, axis=0) for k, v in fx.kkt_model(s).items()}
    w, r1, r2, r3, rhs = (np.repeat(a, batch, axis=0) for a in
                          fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"]))
    r2[1, 5] = 0.0
    r3[2, 2] = -1.3  # w + r3 < 0
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=4, force_generic=force_generic)
    assert pb.ok[:batch].cpu().tolist() == [1, 0, 0, 1]
    res = _check(pb)
    assert torch.equal(res["ok"][:batch], pb.ok[:batch])
    for k in _names(0):
        n = _size(pb.cp, k)
        full = res[k][:n].cpu().numpy()  # [size, batch_stride]
        assert not full[:, batch:].any(), k           # padding lanes
        assert not full[:, [1, 2]].any(), k           # failed problems
        assert n == 0 or full[:, [0, 3]].any(), k


def test_bitwise_repeatable_and_graph_replay():
    pb = _schur_problem(batch=37)
    e = pb.cp.engine
    names = _names(pb.p)
    side = torch.cuda.Stream()
    bufs = lambda: ({k: e.empty(_size(pb.cp, k)) for k in names}, e.empty(_size(pb.cp, "b")))
    g1, a1 = bufs()
    g2, a2 = bufs()
    ok = e.empty_int()
    torch.cuda.synchronize()
    _call(pb, g1, a1, ok, stream=side)
    _call(pb, g2, a2, ok, stream=side)
    side.synchronize()
    for k in names:
        assert torch.equal(g1[k], g2[k]), k
    graph = ctypes.c_void_p()
    e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
    _call(pb, g2, a2, ok, stream=side)
    e._check(lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(graph)))
    for k in names:
        g2[k].fill_(float("nan"))
    a2.fill_(float("nan"))
    torch.cuda.synchronize()
    before = e.launch_count
    e._check(lib.sipoc_graph_launch(e._handle, graph, int(side.cuda_stream)))
    side.synchronize()
    assert e.launch_count == before + lib.sipoc_graph_kernel_count(graph)
    for k in names:
        assert torch.equal(g1[k], g2[k]), k
    assert torch.equal(a1[:, :pb.batch], a2[:, :pb.batch])
    lib.sipoc_graph_destroy(graph)


def test_another_factorization_between_forward_and_backward():
    s = _uniform_kkt_structure(6, 2, 10)
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 40, seed=31, r2_max=1e3)
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs, seed=32)
    first = pb.vjp()
    # the same provider factors and solves a different model before the backward
    other, ow, or1, or2, or3, orhs = pg.newton_kkt_batch(s, 40, seed=33, r2_max=1e3)
    e = pb.cp.engine
    dm2 = pb.cp.pack_model(other)
    pb.cp.factor(dm2, *(e.pack(a) for a in (ow, or1, or2, or3)))
    pb.cp.solve(dm2, e.pack(orhs), e.zeros(rhs.shape[1]))
    second = pb.vjp()
    for k in _names(0):
        assert torch.equal(first[k], second[k]), k
    _check(pb)


def _block_transpose(sizes):
    """Row permutation of a flat array of square column-major blocks: each block transposed."""
    perm, off = [], 0
    for n in sizes:
        perm += [off + j + i * n for j in range(n) for i in range(n)]
        off += n * n
    return torch.tensor(perm, dtype=torch.long)


def test_gradcheck_through_autograd_binding():
    batch = 2
    pb = _schur_problem(batch=batch, seed=5)
    cp, e = pb.cp, pb.cp.engine
    ld, dev = e.batch_stride, e.torch_device()
    perm = _block_transpose([int(v) for v in pb.s.state_dims]).to(dev)
    names = ("b", "r2", "w", "edge_A", "node_jg", "node_hxx", "edge_dynt")
    const = {**pb.dm, **pb.dev}
    leaves = [const[k][:, :batch].clone().requires_grad_(True) for k in names]

    def f(*arrays):
        a = dict(zip(names, arrays))
        a["node_hxx"] = 0.5 * (a["node_hxx"] + a["node_hxx"].index_select(0, perm))
        # engine layout [size, batch_stride]; the padding lanes are solved too, on copies of
        # problem 0, and must not leak into the gradients of the live lanes
        full = {k: torch.cat([v, v[:, :1].expand(-1, ld - batch)], dim=1) for k, v in a.items()}
        arg = {**const, **full}
        model = {k: arg[k] for k in MODEL_NAMES + THETA_NAMES}
        sol, ok = autograd.kkt_factor_solve(cp, model, *(arg[k] for k in REG), arg["b"])
        return sol[:, :batch]

    assert torch.autograd.gradcheck(f, leaves, eps=1e-6, atol=1e-7, rtol=1e-6)


def test_composite_loss_backward_matches_reference():
    s = _uniform_kkt_structure(6, 2, 8)
    batch = 37
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=13, r2_max=1e3)
    pb = Problem(s, 0, model, None, w, r1, r2, r3, rhs)
    e = pb.cp.engine
    inp = {**pb.dm, **pb.dev}
    for v in inp.values():
        v.requires_grad_(True)
    sol, ok = autograd.kkt_factor_solve(pb.cp, {k: inp[k] for k in MODEL_NAMES},
                                        *(inp[k] for k in REG), inp["b"])
    assert not ok.requires_grad
    xd = pb.cp.sizes["x_dim"]
    # the x rows through a square, the duals through a .sum()
    loss = (sol[:xd, :batch] ** 2).sum() + 3.0 * sol[xd:, :batch].sum()
    loss.backward()
    hsol = e.unpack(sol.detach(), rhs.shape[1])
    cot = np.concatenate([2.0 * hsol[:, :xd], np.full_like(hsol[:, xd:], 3.0)], axis=1)
    ref_sol = kkt_solve(s, 0, model, None, w, r1, r2, r3, rhs)
    ref = kkt_vjp(s, 0, model, None, w, r1, r2, r3, ref_sol["sol"], cot)
    for k in _names(0):
        n = _size(pb.cp, k)
        got = e.unpack(inp[k].grad, n)
        assert n == 0 or rel_err(got, ref[k]).max() <= _tol(k), k
        assert not inp[k].grad[:, batch:].any(), k
