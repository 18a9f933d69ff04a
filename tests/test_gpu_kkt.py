"""GPU parity tests of the Newton-KKT path (CallbackProvider::factor / solve /
add_Kx_to_y with theta_dim == 0), all through the C ABI."""
import numpy as np
import pytest

import problem_gen as pg
import reference_fixtures as fx
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from oracle.pyoracle import Structure
from sip_optimal_control_b200 import CallbackProvider

pytestmark = pytest.mark.gpu


def _gpu_kkt(s, model, w, r1, r2, r3, rhs, force_generic=False, pad_variable_dims=False):
    dims, topo = to_structs(s)
    batch = rhs.shape[0]
    cp = CallbackProvider(dims, topo, batch, force_generic=force_generic,
                          pad_variable_dims=pad_variable_dims)
    e = cp.engine
    dm = cp.pack_model(model)
    dw, dr1, dr2, dr3, db = (e.pack(a) for a in (w, r1, r2, r3, rhs))
    ok = cp.factor(dm, dw, dr1, dr2, dr3)
    sol = e.zeros(cp.sizes["kkt_dim"])
    cp.solve(dm, db, sol)
    norms, stats = cp.residual(dm, dw, dr1, dr2, dr3, sol, db, ok)
    return dict(sol=e.unpack(sol, cp.sizes["kkt_dim"]), ok=ok[:batch].cpu().numpy(),
                residual=norms[:batch].cpu().numpy(), stats=stats.cpu().numpy()), cp, \
        (dm, dw, dr1, dr2, dr3, db)


@pytest.mark.parametrize("case", [fx.kkt_case_chain, fx.kkt_case_siblings,
                                  fx.kkt_case_zero_dim_root])
def test_reference_callback_provider_cases(case):
    # variable_dimensions_test.cpp:265-336 via expect_kkt_solve (:135-181)
    s = case()
    sz = pyoracle.kkt_sizes(s)
    model = fx.kkt_model(s)
    w, r1, r2, r3, rhs = fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"])
    rep = lambda a: np.repeat(a, 3, axis=0)
    model = {k: rep(v) for k, v in model.items()}
    w, r1, r2, r3, rhs = (rep(a) for a in (w, r1, r2, r3, rhs))
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    gpu, cp, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    assert cp.sizes["kkt_dim"] == sz["kkt_dim"]
    assert gpu["ok"].tolist() == [1, 1, 1]
    assert gpu["residual"].max() < 1e-9            # the reference's own bar
    assert rel_err(gpu["sol"], ref["sol"]).max() < 1e-12
    assert {k: v.tolist() for k, v in cp.offsets().items()} == \
        {k: v.tolist() for k, v in pyoracle.kkt_offsets(s).items()}


def _uniform_kkt_structure(n, m, T):
    # newton_kkt_benchmark.cpp:58-80: edge constraints everywhere, node
    # constraints only at the terminal node.
    c, g = max(1, n // 2), max(1, 2 * m)
    node_c = [0] * T + [c]
    node_g = [0] * T + [g]
    return Structure.chain(T, n, m, node_c=node_c, node_g=node_g, edge_c=[c] * T,
                           edge_g=[g] * T)


def _oracle_residual(s, model, w, r1, r2, r3, sol, rhs):
    return np.linalg.norm(pyoracle.kkt_apply(s, model, w, r1, r2, r3, sol, np.zeros_like(sol))
                          - rhs, axis=1)


@pytest.mark.parametrize("n,m,T", [(4, 1, 16), (12, 4, 12), (6, 2, 20), (8, 3, 9), (16, 4, 6),
                                   (32, 8, 3)])
@pytest.mark.parametrize("force_generic", [True, False])
@pytest.mark.parametrize("r2_max", [1e3, 1e9])
def test_newton_kkt_benchmark_shapes(n, m, T, force_generic, r2_max):
    # r2_max = 1e9 is the reference benchmark's own regularization range
    # (newton_kkt_benchmark.cpp:231-233).  The shape-specialised kernels apply
    # (I + D V)^-1 in the reference's F-solve form (lqr.cpp:531-549), so the DEFAULT
    # dispatch stays within 1e-9 of the oracle over the whole range, like the
    # reference-order generic kernels.
    s = _uniform_kkt_structure(n, m, T)
    batch = 33
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=n * 100 + m, r2_max=r2_max)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    good = ref["ok"] == 1
    assert good.sum() >= batch - 2
    gpu, cp, dev = _gpu_kkt(s, model, w, r1, r2, r3, rhs, force_generic=force_generic)
    if not force_generic:
        assert "generic" not in cp.engine.kernel_variant, cp.engine.kernel_variant
    assert (gpu["ok"] == ref["ok"]).all()
    assert rel_err(gpu["sol"][good], ref["sol"][good]).max() < REL_TOL
    scale = np.linalg.norm(rhs, axis=1)
    if r2_max <= 1e3:
        assert (gpu["residual"] / scale)[good].max() < 1e-9
    else:
        # at r2 up to 1e9 the residual is the conditioning of the problem (the reference's
        # own order leaves ~1e-6): the device path must not be worse than the oracle's
        ref_res = _oracle_residual(s, model, w, r1, r2, r3, ref["sol"], rhs)
        assert (gpu["residual"][good] / scale[good]).max() <= 10.0 * (ref_res[good] / scale[good]).max()
    # add_Kx_to_y parity on an arbitrary vector
    dm, dw, dr1, dr2, dr3, _ = dev
    xv = np.random.default_rng(1).standard_normal(rhs.shape)
    y0 = np.random.default_rng(2).standard_normal(rhs.shape)
    dy = cp.engine.pack(y0)
    cp.add_Kx_to_y(dm, dw, dr1, dr2, dr3, cp.engine.pack(xv), dy)
    yref = pyoracle.kkt_apply(s, model, w, r1, r2, r3, xv, y0)
    assert rel_err(cp.engine.unpack(dy, rhs.shape[1]), yref).max() < 1e-12


@pytest.mark.parametrize("n,m", [(4, 1), (6, 2), (8, 3), (12, 4)])
def test_chain_operator_kernel_constraints_on_every_node(n, m):
    # kkt_apply_chain (kkt_fast.cu) reads each model block once and feeds the C x / C' y
    # (G x / G' z) sums from the same register; constraint counts vary per node and per
    # edge here (including none), unlike the benchmark shapes.  Checked against the oracle
    # and against the generic output-driven kernel.
    T = 7
    node_c = [(k * 2 + 1) % 4 for k in range(T + 1)]
    node_g = [(k + 2) % 3 for k in range(T + 1)]
    edge_c = [(k + 1) % 3 for k in range(T)]
    edge_g = [(3 * k) % 4 for k in range(T)]
    s = Structure.chain(T, n, m, node_c=node_c, node_g=node_g, edge_c=edge_c, edge_g=edge_g)
    batch = 37
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=n + m, r2_max=1e3)
    xv = np.random.default_rng(5).standard_normal(rhs.shape)
    y0 = np.random.default_rng(6).standard_normal(rhs.shape)
    yref = pyoracle.kkt_apply(s, model, w, r1, r2, r3, xv, y0)
    dims, topo = to_structs(s)
    got = {}
    for force_generic in (False, True):
        cp = CallbackProvider(dims, topo, batch, force_generic=force_generic)
        e = cp.engine
        dy = e.pack(y0)
        cp.add_Kx_to_y(cp.pack_model(model), *(e.pack(a) for a in (w, r1, r2, r3, xv)), dy)
        got[force_generic] = e.unpack(dy, rhs.shape[1])
        assert rel_err(got[force_generic], yref).max() < 1e-12
    assert rel_err(got[False], got[True]).max() < 1e-12
    # the reduction kernel of the same structure (kkt_reduce_chain: node rows on every node)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    assert (ref["ok"] == 1).all()
    gpu, _, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    assert (gpu["ok"] == 1).all()
    assert rel_err(gpu["sol"], ref["sol"]).max() < REL_TOL
    assert (gpu["residual"] / np.linalg.norm(rhs, axis=1)).max() < 1e-9


@pytest.mark.parametrize("case", [fx.kkt_case_chain, fx.kkt_case_siblings,
                                  fx.kkt_case_zero_dim_root])
def test_operator_blocks(case):
    # add_Hx_to_y / add_Cx_to_y / add_CTx_to_y / add_Gx_to_y / add_GTx_to_y
    # (helpers.hpp:17-21, helpers.cpp:979-1368) against the oracle's operator with the
    # regularization switched off and one slot of [x|y|z] populated at a time.
    s = case()
    sz = pyoracle.kkt_sizes(s)
    xd, yd, zd = sz["x_dim"], sz["y_dim"], sz["z_dim"]
    batch = 5
    rng = np.random.default_rng(4)
    model = {k: np.repeat(v, batch, axis=0) * (1.0 + 0.1 * rng.standard_normal((batch, 1)))
             for k, v in fx.kkt_model(s).items()}
    dims, topo = to_structs(s)
    cp = CallbackProvider(dims, topo, batch)
    e = cp.engine
    dm = cp.pack_model(model)
    zero = lambda n: np.zeros((batch, n))
    vx, vy, vz = (rng.standard_normal((batch, n)) for n in (xd, yd, zd))

    def oracle(x_x, x_y, x_z):  # K with w = r1 = r2 = r3 = 0
        x = np.concatenate([x_x, x_y, x_z], axis=1)
        y = pyoracle.kkt_apply(s, model, zero(zd), zero(xd), zero(yd), zero(zd), x,
                               np.zeros_like(x))
        return y[:, :xd], y[:, xd:xd + yd], y[:, xd + yd:]

    cases = [(cp.add_Hx_to_y, vx, xd, oracle(vx, zero(yd), zero(zd))[0]),
             (cp.add_Cx_to_y, vx, yd, oracle(vx, zero(yd), zero(zd))[1]),
             (cp.add_CTx_to_y, vy, xd, oracle(zero(xd), vy, zero(zd))[0]),
             (cp.add_Gx_to_y, vx, zd, oracle(vx, zero(yd), zero(zd))[2]),
             (cp.add_GTx_to_y, vz, xd, oracle(zero(xd), zero(yd), vz)[0])]
    for fn, vin, nout, want in cases:
        y0 = rng.standard_normal((batch, nout))
        dy = e.pack(y0)
        fn(dm, e.pack(vin), dy)
        got = e.unpack(dy, nout)
        assert got.size == 0 or np.abs(got - (y0 + want)).max() < 1e-12, fn.__name__


def test_full_regularization_range_generic_path():
    # newton_kkt_benchmark.cpp:231-239 as is: r2 log-uniform up to 1e9.  The
    # generic kernels follow the reference's operation order, so they must
    # stay within 1e-9 of the oracle even here, and the residual must meet the
    # reference's bar relative to the rhs.
    s = _uniform_kkt_structure(8, 2, 16)
    batch = 40
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=77, r2_max=1e9)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    good = ref["ok"] == 1
    assert good.sum() >= batch - 2
    gpu, _, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs, force_generic=True)
    assert (gpu["ok"] == ref["ok"]).all()
    assert rel_err(gpu["sol"][good], ref["sol"][good]).max() < REL_TOL


def test_variable_dimension_kkt_tiling():
    # BASELINE config 4: the variable_dimensions_test.cpp:266-271 dims pattern
    # (n in {2,1,3}, m in {1,2}, c/g in {0,1,2}) tiled along the horizon.
    reps = 6
    sd = [2, 1, 3] * reps + [2]
    T = len(sd) - 1
    cd = ([1, 2, 1] * reps)[:T]
    node_c = ([1, 0, 2] * reps + [1])[:T + 1]
    node_g = ([0, 2, 1] * reps + [0])[:T + 1]
    edge_c = ([1, 2, 0] * reps)[:T]
    edge_g = ([2, 1, 1] * reps)[:T]
    s = Structure.chain(T, sd, cd, node_c=node_c, node_g=node_g, edge_c=edge_c, edge_g=edge_g)
    batch = 50
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=9, r2_max=1e3)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    assert (ref["ok"] == 1).all()
    gpu, cp, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    assert cp.engine.kernel_variant == "padded_to_strict_thread_n3_m2", cp.engine.kernel_variant
    assert (gpu["ok"] == 1).all()
    assert rel_err(gpu["sol"], ref["sol"]).max() < REL_TOL
    assert gpu["stats"][3] == batch and gpu["stats"][2] == 0
    # the reference benchmark's full regularization range (r2 log-uniform up to 1e9): the
    # default path keeps the reference's operation order, so it stays within 1e-9 of the
    # oracle even there, like the generic kernels
    fm, fw, fr1, fr2, fr3, frhs = pg.newton_kkt_batch(s, batch, seed=10, r2_max=1e9)
    fref = pyoracle.kkt_factor_solve(s, fm, fw, fr1, fr2, fr3, frhs)
    good = fref["ok"] == 1
    assert good.sum() >= batch - 2
    fgpu, _, _ = _gpu_kkt(s, fm, fw, fr1, fr2, fr3, frhs)
    fgen, _, _ = _gpu_kkt(s, fm, fw, fr1, fr2, fr3, frhs, force_generic=True)
    assert (fgpu["ok"] == fref["ok"]).all()
    assert rel_err(fgpu["sol"][good], fref["sol"][good]).max() < REL_TOL
    assert rel_err(fgpu["sol"][good], fgen["sol"][good]).max() < 1e-11
    # SIPOC_FLAG_PAD_VARIABLE_DIMS: the same chain on the (6, 2) sub-warp kernels through
    # decoupled padding.
    gpu, cp, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs, pad_variable_dims=True)
    assert cp.engine.kernel_variant == "padded_to_subwarp4_n6_m2", cp.engine.kernel_variant
    assert (gpu["ok"] == 1).all()
    assert rel_err(gpu["sol"], ref["sol"]).max() < REL_TOL
    assert gpu["stats"][3] == batch and gpu["stats"][2] == 0
    fpad, _, _ = _gpu_kkt(s, fm, fw, fr1, fr2, fr3, frhs, pad_variable_dims=True)
    assert (fpad["ok"] == fref["ok"]).all()
    assert rel_err(fpad["sol"][good], fref["sol"][good]).max() < REL_TOL


def test_config4_full_horizon_matches_oracle():
    # BASELINE config 4 at the horizon bench.py runs it on (T = 48), r2 up to 1e9.
    reps = 16
    sd = [2, 1, 3] * reps + [2]
    T = len(sd) - 1
    cd = ([1, 2, 1] * reps)[:T]
    s = Structure.chain(T, sd, cd, node_c=([1, 0, 2] * reps + [1])[:T + 1],
                        node_g=([0, 2, 1] * reps + [0])[:T + 1], edge_c=([1, 2, 0] * reps)[:T],
                        edge_g=([2, 1, 1] * reps)[:T])
    assert T == 48
    batch = 64
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=48, r2_max=1e9)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    good = ref["ok"] == 1
    assert good.sum() >= batch - 2
    gpu, cp, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    assert cp.engine.kernel_variant == "padded_to_strict_thread_n3_m2", cp.engine.kernel_variant
    assert (gpu["ok"] == ref["ok"]).all()
    assert rel_err(gpu["sol"][good], ref["sol"][good]).max() < REL_TOL


def test_factor_rejects_nonpositive_regularization_per_problem():
    # helpers.cpp:251-295
    s = fx.kkt_case_chain()
    sz = pyoracle.kkt_sizes(s)
    model = {k: np.repeat(v, 4, axis=0) for k, v in fx.kkt_model(s).items()}
    w, r1, r2, r3, rhs = (np.repeat(a, 4, axis=0) for a in
                          fx.kkt_regularization(sz["x_dim"], sz["y_dim"], sz["z_dim"]))
    r2[1, 5] = 0.0
    r3[2, 2] = -1.3
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    gpu, _, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    assert ref["ok"].tolist() == [1, 0, 0, 1]
    assert gpu["ok"].tolist() == [1, 0, 0, 1]
    assert gpu["stats"][2] == 2


def test_host_buffer_entry_points():
    s = _uniform_kkt_structure(6, 2, 10)
    batch = 17
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=4, r2_max=1e3)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    dims, topo = to_structs(s)
    cp = CallbackProvider(dims, topo, batch)
    ok = cp.factor_host(model, w, r1, r2, r3)
    assert (ok == 1).all()
    sol = cp.solve_host(rhs)
    assert rel_err(sol, ref["sol"]).max() < REL_TOL
    prod = cp.add_Kx_to_y_host(w, r1, r2, r3, sol)
    assert (np.linalg.norm(prod - rhs, axis=1) / np.linalg.norm(rhs, axis=1)).max() < 1e-9


@pytest.mark.parametrize("uniform", [True, False])
def test_captured_step_replays_bit_exact(uniform):
    """CallbackProvider.capture_step: the CUDA-graph replay of factor + solve + residual
    returns exactly what the eager calls return, and follows in-place input updates."""
    import torch

    if uniform:
        s = _uniform_kkt_structure(4, 2, 8)
    else:
        s = fx.kkt_case_chain()
    batch = 96
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, batch, seed=5, r2_max=1e3)
    eager, cp, (dm, dw, dr1, dr2, dr3, db) = _gpu_kkt(s, model, w, r1, r2, r3, rhs)
    e = cp.engine
    sol = e.zeros(cp.sizes["kkt_dim"])
    cap = cp.capture_step(dm, dw, dr1, dr2, dr3, db, sol)
    assert cap.launches >= 3
    launches = e.launch_count
    sol.zero_()
    norms, stats = cap.replay()
    torch.cuda.synchronize()
    assert e.launch_count == launches + cap.launches  # the replay counts what it recorded
    assert np.array_equal(e.unpack(sol, cp.sizes["kkt_dim"]), eager["sol"])
    assert np.array_equal(norms[:batch].cpu().numpy(), eager["residual"])
    # stats[0] is an atomic sum over problems (order not fixed); max / counts are exact
    st = stats.cpu().numpy()
    assert np.array_equal(st[1:], eager["stats"][1:])
    assert abs(st[0] - eager["stats"][0]) <= 1e-12 * eager["stats"][0]
    assert np.array_equal(cap.ok[:batch].cpu().numpy(), eager["ok"])
    # a new right-hand side written in place is what the next replay solves
    rhs2 = rhs[::-1].copy()
    db.copy_(e.pack(rhs2))
    cap.replay()
    torch.cuda.synchronize()
    ref2, *_ = _gpu_kkt(s, model, w, r1, r2, r3, rhs2)
    assert np.array_equal(e.unpack(sol, cp.sizes["kkt_dim"]), ref2["sol"])
