"""Every batch-size path of the shape-specialised LQR and Newton-KKT kernels, element-wise
against the CPU oracle.

Which kernels a call runs depends on its batch as well as its shape (riccati_fast.cu:
kSmallBatch = 37 888, kFusedMaxBatch = 40 960; api.cu: kFusedKktMinBatch = 32 768):

  batch            factor_solve                              factor            solve
  < 37 888         sub-warp: riccati_fused_subwarp           sweep, packed W   affine_backward_staged
                   thread: backward + rollout_forward_staged                   + rollout_forward_staged
  37 888..40 960   sub-warp: fused; thread: + rollout_forward sweep, packed W   affine_backward + rollout_forward
  > 40 960         riccati_backward_subwarp (padded map)      sweep, padded W   affine_backward + rollout_forward
                   + rollout_forward
  KKT solve, batch >= 32 768, unpadded uniform chain: affine_backward_kkt + rollout_forward_kkt

The oracle is too slow for 40 000 problems, so every test draws a pool of POOL = 257 distinct
problems, solves the pool on the CPU once and builds the device batch by column gather:
problem b of the batch is pool problem b % POOL, padding lanes zero.  257 is prime, so every
pool problem lands at every position mod 8 (sub-warp tile), mod 32 (warp, batch stride) and
mod 128 (rollout_forward block), and every problem of the batch is compared with the oracle
result of its source -- a full comparison, not a sample.  The copies also give invariants that
need no tolerance: the copies of one problem agree bit for bit, a failing problem leaves every
other problem bit for bit untouched, and nothing depends on the padding lanes
batch <= b < batch_stride (include/sipoc.h puts no requirement on them).
"""
import ctypes

import numpy as np
import pytest

import problem_gen as pg
from gpu_helpers import REL_TOL, rel_err, to_structs
from oracle import pyoracle
from sip_optimal_control_b200 import LQR, CallbackProvider, Dimensions, Topology, _capi
from sip_optimal_control_b200._capi import lib
from test_gpu_kkt import _oracle_residual, _uniform_kkt_structure

pytestmark = pytest.mark.gpu

POOL = 257
SMALL_BATCH = 148 * 128 * 2      # riccati_fast.cu kSmallBatch
FUSED_MAX_BATCH = 40960          # riccati_fast.cu kFusedMaxBatch
FUSED_KKT_MIN_BATCH = 32768      # api.cu kFusedKktMinBatch
# The threshold edges; the last tile of 40 961 holds one valid problem.
BATCHES = [SMALL_BATCH - 1, SMALL_BATCH, FUSED_MAX_BATCH, FUSED_MAX_BATCH + 1]
KKT_BATCHES = [FUSED_KKT_MIN_BATCH - 1, FUSED_KKT_MIN_BATCH, FUSED_MAX_BATCH + 1]

# Thread per problem (n = 4) and four-lane sub-warp plans: every uniform shape with a plan
# of its own in riccati_fast.cu.
PLANS = [(4, m) for m in (1, 2, 3, 4)] + [(n, m) for n in (6, 8) for m in (1, 2, 3, 4)] + [(12, 4)]
# Uniform shapes without a plan, padded up to a sub-warp one (pad / unpad kernels around it).
PADDED = {(7, 4): (8, 4), (10, 3): (12, 4)}
# T = 7 is not a multiple of the 2-, 3- or 4-stage rotating buffers; T = 1 has no middle.
LQR_CASES = [(n, m, 7) for n, m in PLANS + list(PADDED)] + [(6, 3, 1), (12, 4, 1)]
# Shapes whose Newton-KKT reduction has a chain kernel (kkt_fast.cu select_kkt_reduce).
KKT_REDUCE_CHAIN = {(12, 4), (4, 1), (6, 2), (8, 3)}


def _plan_name(n, m):
    return f"thread_per_problem_n{n}_m{m}" if n == 4 else f"subwarp4_n{n}_m{m}"


def _lqr_paths(n, m, batch, padded):
    """The kernel sets factor_solve, factor and solve run (plan shape n, m)."""
    small = batch < SMALL_BATCH
    rollout = "rollout_forward_staged" if small else "rollout_forward"
    backward = "riccati_backward_thread" if n == 4 else "riccati_backward_subwarp"
    if n != 4 and batch <= FUSED_MAX_BATCH:
        factor_solve = {"riccati_fused_subwarp"}
    else:
        factor_solve = {backward, rollout}
    factor = {backward}
    solve = {"affine_backward_staged" if small else "affine_backward", rollout}
    if padded:
        factor_solve |= {"pad_chain_kernel", "unpad_chain_kernel"}
        factor |= {"pad_chain_kernel"}
        solve |= {"pad_chain_kernel", "unpad_chain_kernel"}
    return factor_solve, factor, solve


def _profiled(engine, call):
    """(call(), the set of kernel names the call launched) via the engine's event profiler."""
    lib.sipoc_profile_enable(engine._handle, 1)
    try:
        result = call()
        names = set()
        for i in range(lib.sipoc_profile_collect(engine._handle)):
            nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
            engine._check(lib.sipoc_profile_get(engine._handle, i, ctypes.byref(nm),
                                                ctypes.byref(ms), ctypes.byref(cnt)))
            names.add(nm.value.decode())
    finally:
        lib.sipoc_profile_enable(engine._handle, 0)
    return result, names


def _src(batch):
    return np.arange(batch) % POOL


def _expand(engine, pool):
    """Pool [POOL, size] (problem-major host) -> engine-layout device tensor of the whole
    batch: column b is pool problem b % POOL, padding lanes zero."""
    import torch

    dev = engine.torch_device()
    full = engine.zeros(pool.shape[1])
    if pool.shape[1]:
        pool_dev = torch.from_numpy(np.ascontiguousarray(pool.T, dtype=np.float64)).to(dev)
        src = torch.from_numpy(_src(engine.batch)).to(dev)
        full[:, :engine.batch] = pool_dev[:, src]
    return full


def _nan_padded(engine, arrays):
    """Copies with NaN in the padding lanes batch <= b < batch_stride."""
    out = {}
    for k, t in arrays.items():
        t = t.clone()
        t[:, engine.batch:] = float("nan")
        out[k] = t
    return out


def _host(t, size, batch):
    return t[:size, :batch].T.cpu().numpy()


def _lanes(idx):
    idx = np.asarray(idx)[:8]
    return (f"problems {idx.tolist()} (mod 8 {sorted(set((idx % 8).tolist()))}, "
            f"mod 32 {sorted(set((idx % 32).tolist()))}, mod 128 {sorted(set((idx % 128).tolist()))})")


def _unpack_lqr(lqr, out, status):
    sz, b = lqr.engine.lqr_sizes, lqr.batch
    got = {k: _host(out[k], sz[k], b) for k in _capi.LQR_OUTPUT_FIELDS}
    got["status"] = status[:b].cpu().numpy()
    return got


def _check_lqr(got, ref, src, what):
    """Status equal to the oracle's for every problem, x/u/y of the solved ones within REL_TOL
    of the oracle, and every copy of a pool problem bitwise equal to its first copy (batch
    index = pool index)."""
    want = ref["status"][src]
    bad = np.flatnonzero(got["status"] != want)
    assert bad.size == 0, (what, "status", _lanes(bad), got["status"][bad[:8]].tolist(),
                           want[bad[:8]].tolist())
    good = want == 0
    for k in _capi.LQR_OUTPUT_FIELDS:
        err = rel_err(got[k], ref[k][src])
        bad = np.flatnonzero(good & ~(err <= REL_TOL))
        assert bad.size == 0, (what, k, float(err[bad].max()), _lanes(bad))
        same = (got[k] == got[k][src]).all(axis=1)
        bad = np.flatnonzero(good & ~same)
        assert bad.size == 0, (what, k, "copies of one problem differ", _lanes(bad))


def _assert_bitwise(a, b, keys, mask, what):
    for k in keys:
        same = (a[k] == b[k]) if a[k].ndim == 1 else (a[k] == b[k]).all(axis=1)
        bad = np.flatnonzero(mask & ~same)
        assert bad.size == 0, (what, k, _lanes(bad))


def _lqr_pool(n, m, T, seed):
    return pg.lqr_benchmark_batch(n, m, T, POOL, seed=seed, dense_M=True)


# --- 1. the LQR path matrix ----------------------------------------------------------------
@pytest.mark.parametrize("batch", BATCHES)
@pytest.mark.parametrize("n,m,T", LQR_CASES)
def test_lqr_batch_paths_match_oracle(n, m, T, batch):
    s, pool = _lqr_pool(n, m, T, seed=1000 + 10 * n + m + T)
    ref = pyoracle.lqr_factor_solve(s, pool)
    assert (ref["status"] == 0).all()
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    padded = (n, m) in PADDED
    pn, pm = PADDED.get((n, m), (n, m))
    assert e.kernel_variant == ("padded_to_" if padded else "") + _plan_name(pn, pm)
    want_fs, want_f, want_s = _lqr_paths(pn, pm, batch, padded)
    src = _src(batch)
    inp = {k: _expand(e, pool[k]) for k in _capi.LQR_INPUT_FIELDS}
    has_padding = e.batch_stride > batch

    # factor + solve in one call
    out = lqr.alloc_output()
    status, names = _profiled(e, lambda: lqr.factor_solve(inp, out))
    assert names == want_fs, names
    fused = _unpack_lqr(lqr, out, status)
    _check_lqr(fused, ref, src, "factor_solve")
    # the KKT residual of every problem at rounding level, on the scale of its right-hand side
    norms, stats = lqr.residual(inp, out, status)
    scale = np.linalg.norm(np.concatenate([pool["q"], pool["r"], pool["c"]], axis=1), axis=1)[src]
    res = norms[:batch].cpu().numpy()
    assert (res / scale).max() < 1e-9, float((res / scale).max())
    st = stats.cpu().numpy()
    assert st[2] == 0 and st[3] == batch and np.isclose(st[1], res.max())
    if has_padding:  # NaN in the padding lanes changes no real problem
        nan_out = lqr.alloc_output()
        nan_status = lqr.factor_solve(_nan_padded(e, inp), nan_out)
        _assert_bitwise(_unpack_lqr(lqr, nan_out, nan_status), fused,
                        ("x", "u", "y", "status"), np.ones(batch, bool), "factor_solve, NaN padding")

    # factor, then solve
    if has_padding:
        nan_inp = _nan_padded(e, inp)
        nan_out = lqr.alloc_output()
        nan_status = lqr.factor_with_status(nan_inp)
        lqr.solve(nan_inp, nan_out)
        nan_split = _unpack_lqr(lqr, nan_out, nan_status)
    out = lqr.alloc_output()
    status, names = _profiled(e, lambda: lqr.factor_with_status(inp))
    assert names == want_f, names
    _, names = _profiled(e, lambda: lqr.solve(inp, out))
    assert names == want_s, names
    split = _unpack_lqr(lqr, out, status)
    _check_lqr(split, ref, src, "factor + solve")
    if has_padding:
        _assert_bitwise(nan_split, split, ("x", "u", "y", "status"), np.ones(batch, bool),
                        "factor + solve, NaN padding")

    # factor once, solve many: new q, r, c against the kept factorization
    rng = np.random.default_rng(T + batch)
    pool2 = dict(pool)
    for k in ("q", "r", "c"):
        pool2[k] = rng.standard_normal(pool[k].shape)
    ref2 = pyoracle.lqr_factor_solve(s, pool2)
    inp2 = dict(inp)
    for k in ("q", "r", "c"):
        inp2[k] = _expand(e, pool2[k])
    out2 = lqr.alloc_output()
    _, names = _profiled(e, lambda: lqr.solve(inp2, out2))
    assert names == want_s, names
    _check_lqr(_unpack_lqr(lqr, out2, status), ref2, src, "re-solve on the kept factor")


# --- 2. failure injection: late pivots, ordering, and what a failure must not touch ---------
def _set(a, problem, block, size, row, col, ld_rows, value):
    """a[problem] holds column-major [rows x cols] blocks of `size` elements each."""
    a[problem, block * size + col * ld_rows + row] = value


def _inject(pool, n, m, T):
    """Each failure into one fixed pool problem (so it appears ~150 times, at every tile,
    warp and block position of a 40 000-problem batch).  Returns {pool index: oracle code}."""
    Q, R, delta = pool["Q"], pool["R"], pool["delta"]
    nn, mm, h = n * n, m * m, T // 2
    want = {}
    # a zero delta at the last state of a middle node (a lane of the partial block at n = 6)
    delta[11, h * n + n - 1] = 0.0
    want[11] = 1
    # F fails at the last pivot only: the leading block is untouched
    _set(Q, 40, T, nn, n - 1, n - 1, n, -1e5)
    want[40] = 2
    # F fails at the first pivot of block 1 (pivot 3 for n = 4)
    p = min(4, n - 1)
    _set(Q, 77, h, nn, p, p, n, -1e5)
    want[77] = 2
    # G fails at its last pivot, and at edge 0
    _set(R, 128, T - 1, mm, m - 1, m - 1, m, -1e5)
    want[128] = 3
    _set(R, 170, 0, mm, 0, 0, m, -1e5)
    want[170] = 3
    # a negative delta at the root AND a G failure deeper: the post-order sweep meets G first
    delta[211, 0] = -1.0
    _set(R, 211, T - 1, mm, 0, 0, m, -1e5)
    want[211] = 3
    # F fails at the root
    _set(Q, 256, 0, nn, 0, 0, n, -1e5)
    want[256] = 2
    return want


@pytest.mark.parametrize("batch", BATCHES)
@pytest.mark.parametrize("n,m", PLANS + list(PADDED))
def test_lqr_failures_set_status_and_touch_nothing_else(n, m, batch):
    T = 7
    s, pool = _lqr_pool(n, m, T, seed=2000 + 10 * n + m)
    bad_pool = {k: v.copy() for k, v in pool.items()}
    want = _inject(bad_pool, n, m, T)
    ref = pyoracle.lqr_factor_solve(s, pool)
    assert (ref["status"] == 0).all()
    bad_ref = pyoracle.lqr_factor_solve(s, bad_pool)
    # the oracle confirms each injection hits the intended case
    assert {p: int(bad_ref["status"][p]) for p in want} == want
    assert (np.delete(bad_ref["status"], list(want)) == 0).all()

    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    src = _src(batch)
    inp = {k: _expand(e, pool[k]) for k in _capi.LQR_INPUT_FIELDS}
    bad_inp = {k: _expand(e, bad_pool[k]) for k in _capi.LQR_INPUT_FIELDS}
    untouched = ~np.isin(src, list(want))

    def fused(i):
        out = lqr.alloc_output()
        return _unpack_lqr(lqr, out, lqr.factor_solve(i, out))

    def split(i):
        out = lqr.alloc_output()
        status = lqr.factor_with_status(i)
        lqr.solve(i, out)
        return _unpack_lqr(lqr, out, status)

    for name, run in (("factor_solve", fused), ("factor + solve", split)):
        clean, bad = run(inp), run(bad_inp)
        _check_lqr(clean, ref, src, name)
        _check_lqr(bad, bad_ref, src, name + ", injected")
        # failed problems: status only (their x, u, y are unspecified); the rest bit for bit
        _assert_bitwise(bad, clean, ("x", "u", "y", "status"), untouched,
                        name + ": a failure changed another problem")
    assert int((bad["status"] != 0).sum()) == int((~untouched).sum())


# --- 3. Newton-KKT ---------------------------------------------------------------------------
def _kkt_paths(n, m, batch):
    small = batch < SMALL_BATCH
    backward = "riccati_backward_thread" if n == 4 else "riccati_backward_subwarp"
    factor = {"kkt_reduce_chain" if (n, m) in KKT_REDUCE_CHAIN else "kkt_reduce_kernel", backward}
    if batch >= FUSED_KKT_MIN_BATCH:
        solve = {"affine_backward_kkt", "rollout_forward_kkt"}
    else:
        solve = {"kkt_build_rhs_kernel", "kkt_recover_kernel",
                 "affine_backward_staged" if small else "affine_backward",
                 "rollout_forward_staged" if small else "rollout_forward"}
    return factor, solve


@pytest.mark.parametrize("batch", KKT_BATCHES)
@pytest.mark.parametrize("n,m", PLANS)
def test_kkt_batch_paths_match_oracle(n, m, batch):
    T = 7
    s = _uniform_kkt_structure(n, m, T)
    # r2 log-uniform up to 1e9: the reference benchmark's own regularization range
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, POOL, seed=3000 + 10 * n + m, r2_max=1e9)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    assert (ref["ok"] == 1).sum() >= POOL - 16
    dims, topo = to_structs(s)
    cp = CallbackProvider(dims, topo, batch)
    e = cp.engine
    assert e.kernel_variant == _plan_name(n, m)
    want_f, want_s = _kkt_paths(n, m, batch)
    src = _src(batch)
    dm = {k: _expand(e, model[k]) for k in _capi.KKT_MODEL_FIELDS}
    dw, dr1, dr2, dr3, db = (_expand(e, a) for a in (w, r1, r2, r3, rhs))
    ok, names = _profiled(e, lambda: cp.factor(dm, dw, dr1, dr2, dr3))
    assert names == want_f, names
    kd = cp.sizes["kkt_dim"]
    sol = e.zeros(kd)
    _, names = _profiled(e, lambda: cp.solve(dm, db, sol))
    assert names == want_s, names

    got_ok = ok[:batch].cpu().numpy()
    want_ok = ref["ok"][src]
    bad = np.flatnonzero(got_ok != want_ok)
    assert bad.size == 0, ("ok", _lanes(bad))
    good = want_ok == 1
    got = _host(sol, kd, batch)
    err = rel_err(got, ref["sol"][src])
    bad = np.flatnonzero(good & ~(err <= REL_TOL))
    assert bad.size == 0, ("sol", float(err[bad].max()), _lanes(bad))
    bad = np.flatnonzero(good & ~(got == got[src]).all(axis=1))
    assert bad.size == 0, ("copies of one problem differ", _lanes(bad))
    # at r2 up to 1e9 the residual is the conditioning of the problem (the reference's own
    # order leaves ~1e-6): the device path must not be worse than the oracle's
    norms, _ = cp.residual(dm, dw, dr1, dr2, dr3, sol, db, ok)
    scale = np.linalg.norm(rhs, axis=1)
    ref_res = _oracle_residual(s, model, w, r1, r2, r3, ref["sol"], rhs) / scale
    res = norms[:batch].cpu().numpy() / scale[src]
    assert res[good].max() <= 10.0 * ref_res[ref["ok"] == 1].max()


# --- 4. the benchmark's own LQR configs at their real batch ----------------------------------
BENCH_SEED = 2026  # bench.py --seed default
BENCH_PATHS = {
    "cartpole": {"riccati_backward_thread", "rollout_forward_staged"},
    "quadrotor": {"riccati_backward_subwarp", "rollout_forward"},
    # CTA per problem: the inputs are transposed to problem-major copies first
    "humanoid": {"unpack_kernel", "riccati_backward_cta", "rollout_forward_cta"},
}


@pytest.mark.parametrize("name", sorted(BENCH_PATHS))
def test_bench_configs_at_full_batch(name):
    import torch

    from bench import WORKLOADS

    wl = WORKLOADS[name]
    n, m, T, batch = wl["n"], wl["m"], wl["T"], wl["batch"]
    lqr = LQR(Dimensions.uniform(T, n, m), Topology.chain(T), batch)
    e = lqr.engine
    sz = e.lqr_sizes
    # inputs + outputs, and as much again for the kept factorization and the solve's scratch
    need = 2 * 8 * e.batch_stride * sum(sz[k] for k in _capi.LQR_INPUT_FIELDS + _capi.LQR_OUTPUT_FIELDS)
    free, _ = torch.cuda.mem_get_info(e.torch_device())
    if free < need:
        pytest.skip(f"{name} needs ~{need / 2**30:.0f} GiB of device memory, "
                    f"{free / 2**30:.0f} GiB free")
    inp = lqr.generate_benchmark(seed=BENCH_SEED)
    out = lqr.alloc_output()
    status, names = _profiled(e, lambda: lqr.factor_solve(inp, out))
    assert names == BENCH_PATHS[name], names
    assert int((status[:batch] != 0).sum().item()) == 0
    # every problem: KKT residual at rounding level on the scale of its right-hand side
    norms, stats = lqr.residual(inp, out, status)
    rhs = torch.cat([inp[k][:sz[k], :batch] for k in ("q", "r", "c")])
    res = (norms[:batch] / torch.linalg.vector_norm(rhs, dim=0)).max().item()
    assert res < 1e-9, res
    assert stats[2].item() == 0 and stats[3].item() == batch
    # a sample against the oracle: the first tile, a rollout block edge, the last tile, and
    # random picks
    count = 64 if n > 16 else 512
    fixed = np.r_[0:8, 127:129, batch - 8:batch]
    rng = np.random.default_rng(5)
    rest = np.setdiff1d(np.arange(batch), fixed)
    idx = np.sort(np.r_[fixed, rng.choice(rest, count - fixed.size, replace=False)])
    tidx = torch.from_numpy(idx).to(e.torch_device())
    host = {k: inp[k][:sz[k]][:, tidx].T.cpu().numpy() for k in _capi.LQR_INPUT_FIELDS}
    ref = pyoracle.lqr_factor_solve(pyoracle.Structure.chain(T, n, m), host)
    assert (ref["status"] == 0).all()
    for k in _capi.LQR_OUTPUT_FIELDS:
        got = out[k][:sz[k]][:, tidx].T.cpu().numpy()
        err = rel_err(got, ref[k])
        assert err.max() <= REL_TOL, (k, float(err.max()), _lanes(idx[err > REL_TOL]))
