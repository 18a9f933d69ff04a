"""Timing of the LQR VJP (sipoc_lqr_vjp) on the GPU.

Per workload (inputs from sipoc_generate_lqr_benchmark, cotangents N(0, 1)), with CUDA
events after a warm-up:
- the forward factor_solve;
- sipoc_lqr_vjp with all nine gradients, and with only (q, c);
- the gradient kernel alone (lqr_vjp_kernel, sipoc_profile_*), with its bytes computed from
  the sizes -- the requested gradients written (every lane of batch_stride), the x, u, y and
  mu entries they need read, and the status -- its bandwidth and share of 7.7 TB/s (the
  HGX B200 data-sheet HBM3e rate of one GPU).
A seeded sample of problems is checked against the CPU reference VJP.  The device name, power
limit and max SM clock are read in the same run.  Usage:
    python tools/bench_vjp.py --out profiles/r03/bench_vjp.json [--workloads quadrotor,...]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from gpu_helpers import rel_err, to_structs  # noqa: E402
from oracle import pyoracle  # noqa: E402
from sip_optimal_control_b200 import LQR, _capi  # noqa: E402
from sip_optimal_control_b200._capi import lib  # noqa: E402
from vjp_reference import GRAD_NAMES, lqr_vjp  # noqa: E402

PEAK_TBS = 7.7
WORKLOADS = {  # name: (n, m, T, batch)
    "quadrotor": (12, 4, 50, 65536),
    "cartpole": (4, 1, 100, 65536),
    "humanoid": (64, 24, 32, 4096),
    "long_horizon": (12, 4, 4096, 64),  # runs on the parallel-in-time scan
}
# solution / adjoint vectors each gradient array is built from
NEEDS = dict(Q=("x", "mx"), M=("x", "mx", "u", "mu"), R=("u", "mu"), q=("mx",), r=("mu",),
             A=("x", "mx", "y", "my"), B=("y", "my", "u", "mu"), c=("my",), delta=("y", "my"))


def device_info() -> dict:
    info = dict(device=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (v.strip() for v in q.split(","))
        info.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:  # the numbers are still reported, without these fields
        info["smi_error"] = repr(exc)
    return info


def kernel_bytes(sizes: dict, want, batch: int, ld: int) -> int:
    vec = dict(x=sizes["x"], mx=sizes["x"], u=sizes["u"], mu=sizes["u"], y=sizes["y"],
               my=sizes["y"])
    read = set().union(*(NEEDS[k] for k in want))
    return (8 * ld * sum(sizes[k] for k in want) + 8 * batch * sum(vec[v] for v in read)
            + 4 * batch)


def event_ms(fn, warmup: int, iters: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def profiled_kernel_ms(eng, fn, iters: int) -> float:
    lib.sipoc_profile_enable(eng._handle, 1)
    for _ in range(iters):
        fn()
    total, count = 0.0, 0
    for i in range(lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        eng._check(lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                                         ctypes.byref(cnt)))
        if nm.value.decode() == "lqr_vjp_kernel":
            total, count = ms.value, cnt.value
    lib.sipoc_profile_enable(eng._handle, 0)
    assert count == iters, count
    return total / count


def run(name, n, m, T, batch, warmup, iters, sample):
    s = pyoracle.Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    sz = e.lqr_sizes
    inp = lqr.generate_benchmark(seed=2026)
    out, adj = lqr.alloc_output(), lqr.alloc_output()
    status = e.empty_int()
    gen = torch.Generator(device=e.torch_device()).manual_seed(7)
    cot = {k: torch.randn(out[k].shape, generator=gen, dtype=torch.float64,
                          device=e.torch_device()) for k in ("x", "u", "y")}
    grads = {k: e.empty(sz[k]) for k in GRAD_NAMES}
    stream = e.stream_ptr()
    si = _capi.LqrInput(*[inp[k].data_ptr() for k in GRAD_NAMES])
    so = _capi.LqrOutput(*[out[k].data_ptr() for k in ("x", "u", "y")])
    sc = _capi.LqrCotangent(*[cot[k].data_ptr() for k in ("x", "u", "y")])
    sa = _capi.LqrOutput(*[adj[k].data_ptr() for k in ("x", "u", "y")])

    def vjp_call(want):
        sg = _capi.LqrGrad(*[grads[k].data_ptr() if k in want else None for k in GRAD_NAMES])
        return lambda: e._check(lib.sipoc_lqr_vjp(
            e._handle, ctypes.byref(si), ctypes.byref(so), ctypes.byref(sc), ctypes.byref(sa),
            ctypes.byref(sg), status.data_ptr(), stream))

    forward = lambda: lqr.factor_solve(inp, out, status=status)
    forward()
    vjp_all, vjp_qc = vjp_call(GRAD_NAMES), vjp_call(("q", "c"))
    line = dict(workload=name, n=n, m=m, T=T, batch=batch, batch_stride=e.batch_stride,
                kernel_variant=e.kernel_variant, iters=iters)
    line["forward_ms"] = event_ms(forward, warmup, iters)
    line["vjp_all_ms"] = event_ms(vjp_all, warmup, iters)
    line["vjp_qc_ms"] = event_ms(vjp_qc, warmup, iters)
    for tag, fn, want in (("all", vjp_all, GRAD_NAMES), ("qc", vjp_qc, ("q", "c"))):
        ms = profiled_kernel_ms(e, fn, iters)
        nbytes = kernel_bytes(sz, want, batch, e.batch_stride)
        tbs = nbytes / (ms * 1e-3) / 1e12
        line[f"kernel_{tag}"] = dict(ms=ms, bytes=nbytes, tb_per_s=tbs,
                                     share_of_7_7_tb_per_s=tbs / PEAK_TBS)
    # seeded sample against the CPU reference, from the last (all-gradient) call
    vjp_all()
    torch.cuda.synchronize()
    assert bool((status[:batch] == 0).all())
    idx = torch.from_numpy(np.random.default_rng(11).choice(batch, min(sample, batch),
                                                            replace=False)).to(e.torch_device())
    pick = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: pick(inp[k], sz[k]) for k in GRAD_NAMES}
    hcot = {k: pick(cot[k], sz[k]) for k in ("x", "u", "y")}
    ref = lqr_vjp(s, host, pyoracle.lqr_factor_solve(s, host, residual=False), hcot)
    line["sample_problems"] = int(idx.numel())
    line["sample_max_rel_err"] = {k: float(rel_err(pick(grads[k], sz[k]), ref[k]).max())
                                  for k in GRAD_NAMES}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sample", type=int, default=16)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_vjp.py needs a CUDA device")
    torch.cuda.set_device(0)
    result = dict(tool="tools/bench_vjp.py", **device_info(), peak_tb_per_s=PEAK_TBS, runs=[])
    for name in args.workloads.split(","):
        line = run(name, *WORKLOADS[name], args.warmup, args.iters, args.sample)
        print(json.dumps(line), flush=True)
        result["runs"].append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
