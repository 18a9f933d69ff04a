"""Timing of the LQR and Newton-KKT JVPs (sipoc_lqr_jvp, sipoc_kkt_jvp) on the GPU.

Per workload (the LQR rows of tools/bench_vjp.py, the Newton-KKT rows of tools/bench_kkt_vjp.py;
tangents N(0, 1)), with CUDA events after a warm-up:
- the forward (factor_solve / factor + solve);
- the JVP with a tangent of every input, and with the vector tangents alone (dq, dr, dc / db);
- the tangent kernel alone (lqr_jvp_kernel / kkt_jvp_kernel, sipoc_profile_*), with its
  compulsory bytes computed from the sizes -- the tangent arrays read and the solution entries
  they need (live lanes), t written (every lane of batch_stride); the kernel reads no status --
  its bandwidth and share of 7.7 TB/s (the HGX B200 data-sheet HBM3e rate of one GPU), and the
  zeroing pass after the solve (jvp_zero_dead_lanes).
A seeded sample of problems is checked against the CPU reference JVP.  The device name, power
limit and max SM clock are read in the same run.  Usage:
    python tools/bench_jvp.py --out profiles/r05/bench_jvp.json [--workloads quadrotor,...]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from bench import kkt_host_problem  # noqa: E402
from bench_kkt_vjp import REG, dimensions  # noqa: E402
from bench_kkt_vjp import WORKLOADS as KKT_WORKLOADS  # noqa: E402
from bench_vjp import PEAK_TBS, device_info, event_ms  # noqa: E402
from bench_vjp import WORKLOADS as LQR_WORKLOADS  # noqa: E402
from gpu_helpers import rel_err, to_structs  # noqa: E402
from jvp_reference import kkt_jvp, lqr_jvp  # noqa: E402
from kkt_vjp_reference import MODEL_NAMES, VECTOR_NAMES, kkt_solve  # noqa: E402
from oracle import pyoracle  # noqa: E402
from oracle.pyoracle import Structure  # noqa: E402
from sip_optimal_control_b200 import LQR, CallbackProvider, Topology  # noqa: E402
from sip_optimal_control_b200._capi import lib  # noqa: E402
from vjp_reference import GRAD_NAMES  # noqa: E402

# solution vectors the tangent of each LQR input is multiplied with
NEEDS = dict(Q=("x",), M=("x", "u"), R=("u",), q=(), r=(), A=("x", "y"), B=("u", "y"), c=(),
             delta=("y",))


def profiled_ms(eng, fn, iters: int) -> dict:
    """Mean ms per call of every profiled kernel over ``iters`` calls."""
    lib.sipoc_profile_enable(eng._handle, 1)
    for _ in range(iters):
        fn()
    out = {}
    for i in range(lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        eng._check(lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                                         ctypes.byref(cnt)))
        out[nm.value.decode()] = ms.value / iters
    lib.sipoc_profile_enable(eng._handle, 0)
    return out


def kernel_line(ms: float, nbytes: int) -> dict:
    tbs = nbytes / (ms * 1e-3) / 1e12
    return dict(ms=ms, bytes=nbytes, tb_per_s=tbs, share_of_7_7_tb_per_s=tbs / PEAK_TBS)


def run_lqr(name, n, m, T, batch, warmup, iters, sample):
    s = pyoracle.Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    sz, ld = e.lqr_sizes, e.batch_stride
    inp = lqr.generate_benchmark(seed=2026)
    out, dsol = lqr.alloc_output(), lqr.alloc_output()
    rhs = {k: e.empty(sz[k]) for k in ("q", "r", "c")}
    status, jvp_status = e.empty_int(), e.empty_int()
    gen = torch.Generator(device=e.torch_device()).manual_seed(7)
    tan = {k: torch.randn(inp[k].shape, generator=gen, dtype=torch.float64,
                          device=e.torch_device()) for k in GRAD_NAMES}
    forward = lambda: lqr.factor_solve(inp, out, status=status)
    call = lambda t: (lambda: lqr.jvp(inp, out, t, dsol=dsol, rhs=rhs, status=jvp_status))
    vec = {k: tan[k] for k in ("q", "r", "c")}
    jvp_all, jvp_vec = call(tan), call(vec)
    forward()
    line = dict(workload=name, n=n, m=m, T=T, batch=batch, batch_stride=ld,
                kernel_variant=e.kernel_variant, iters=iters)
    line["forward_ms"] = event_ms(forward, warmup, iters)
    line["jvp_all_ms"] = event_ms(jvp_all, warmup, iters)
    line["jvp_vectors_ms"] = event_ms(jvp_vec, warmup, iters)
    rhs_bytes = 8 * ld * (sz["q"] + sz["r"] + sz["c"])
    for tag, fn, want in (("all", jvp_all, GRAD_NAMES), ("vectors", jvp_vec, ("q", "r", "c"))):
        prof = profiled_ms(e, fn, iters)
        read = set().union(*(NEEDS[k] for k in want))
        nbytes = 8 * batch * (sum(sz[k] for k in want) + sum(sz[v] for v in read)) + rhs_bytes
        line[f"kernel_{tag}"] = kernel_line(prof["lqr_jvp_kernel"], nbytes)
        line[f"zero_pass_{tag}_ms"] = prof.get("jvp_zero_dead_lanes")
    forward()
    jvp_all()
    torch.cuda.synchronize()
    idx = torch.from_numpy(np.sort(np.random.default_rng(11).choice(batch, min(sample, batch),
                                                                    replace=False)))
    idx = idx.to(e.torch_device())
    pick = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: pick(inp[k], sz[k]) for k in GRAD_NAMES}
    ref = lqr_jvp(s, host, pyoracle.lqr_factor_solve(s, host),
                  {k: pick(tan[k], sz[k]) for k in GRAD_NAMES})
    line["sample_problems"] = int(idx.numel())
    line["sample_max_rel_err"] = {k: float(rel_err(pick(dsol[k], sz[k]), ref[k]).max())
                                  for k in ("x", "u", "y")}
    return line


def run_kkt(name, kind, batch, warmup, iters, sample, seed):
    T, dims = dimensions(kind)
    cp = CallbackProvider(dims, Topology.chain(T), batch, device=0)
    e = cp.engine
    z, ld = cp.sizes, e.batch_stride
    size = {k: z[k] for k in MODEL_NAMES}
    size.update(b=z["kkt_dim"], w=z["z_dim"], r1=z["x_dim"], r2=z["y_dim"], r3=z["z_dim"])
    model_h, w_h, r1_h, r2_h, r3_h, b_h = kkt_host_problem(dims, batch, seed, 1e9)
    reg_h = dict(w=w_h, r1=r1_h, r2=r2_h, r3=r3_h)
    model = cp.pack_model(model_h)
    reg = {k: e.pack(v) for k, v in reg_h.items()}
    b = e.pack(b_h)
    del b_h
    kd = z["kkt_dim"]
    sol, dsol, rhs = e.zeros(kd), e.empty(kd), e.empty(kd)
    ok, jvp_ok = e.empty_int(), e.empty_int()
    gen = torch.Generator(device=e.torch_device()).manual_seed(7)
    tan = {k: torch.randn((max(size[k], 1), ld), generator=gen, dtype=torch.float64,
                          device=e.torch_device()) for k in MODEL_NAMES + VECTOR_NAMES}

    def forward():
        cp.factor(model, *(reg[k] for k in REG), ok=ok)
        cp.solve(model, b, sol)

    call = lambda t: (lambda: cp.jvp(model, *(reg[k] for k in REG), sol, t, dsol=dsol, rhs=rhs,
                                     ok=jvp_ok))
    vec = {k: tan[k] for k in VECTOR_NAMES}
    jvp_all, jvp_vec = call(tan), call(vec)
    forward()
    line = dict(workload=name, T=T, batch=batch, batch_stride=ld,
                kernel_variant=e.kernel_variant, iters=iters)
    line["forward_ms"] = event_ms(forward, warmup, iters)
    line["jvp_all_ms"] = event_ms(jvp_all, warmup, iters)
    line["jvp_vectors_ms"] = event_ms(jvp_vec, warmup, iters)
    for tag, fn, want in (("all", jvp_all, MODEL_NAMES + VECTOR_NAMES),
                          ("vectors", jvp_vec, VECTOR_NAMES)):
        prof = profiled_ms(e, fn, iters)
        nbytes = 8 * batch * (sum(size[k] for k in want) + kd) + 8 * ld * kd
        line[f"kernel_{tag}"] = kernel_line(prof["kkt_jvp_kernel"], nbytes)
        line[f"zero_pass_{tag}_ms"] = prof.get("jvp_zero_dead_lanes")
    forward()
    jvp_all()
    torch.cuda.synchronize()
    idx_h = np.sort(np.random.default_rng(11).choice(batch, min(sample, batch), replace=False))
    idx = torch.from_numpy(idx_h).to(e.torch_device())
    pick = lambda t, n: t[:n].index_select(1, idx).T.contiguous().cpu().numpy()
    s = Structure.chain(T, dims.state_dims, dims.control_dims, node_c=dims.node_c_dims,
                        node_g=dims.node_g_dims, edge_c=dims.edge_c_dims,
                        edge_g=dims.edge_g_dims)
    hm = {k: v[idx_h] for k, v in model_h.items()}
    hr = [reg_h[k][idx_h] for k in REG]
    ref_sol = kkt_solve(s, 0, hm, None, *hr, pick(b, kd))
    htan = {k: pick(tan[k], size[k]) for k in tan}
    ref = kkt_jvp(s, 0, hm, None, *hr, ref_sol["sol"], htan)
    good = ref["ok"] == 1
    assert (jvp_ok[:batch].index_select(0, idx).cpu().numpy() == ref["ok"]).all()
    line["sample_problems"] = int(idx.numel())
    line["sample_ok"] = int(good.sum())
    line["sample_max_rel_err"] = float(rel_err(pick(dsol, kd)[good], ref["sol"][good]).max())
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(list(LQR_WORKLOADS) + list(KKT_WORKLOADS)))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sample", type=int, default=16)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_jvp.py needs a CUDA device")
    torch.cuda.set_device(0)
    result = dict(tool="tools/bench_jvp.py", **device_info(), peak_tb_per_s=PEAK_TBS, runs=[])
    for name in args.workloads.split(","):
        if name in LQR_WORKLOADS:
            line = run_lqr(name, *LQR_WORKLOADS[name], args.warmup, args.iters, args.sample)
        else:
            kind, batch = KKT_WORKLOADS[name]
            line = run_kkt(name, kind, batch, args.warmup, args.iters, args.sample, args.seed)
        print(json.dumps(line), flush=True)
        result["runs"].append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
