"""Timing of the LQR policy export (sipoc_lqr_factor_solve_policy) on the GPU.

Per workload (inputs from sipoc_generate_lqr_benchmark), with CUDA events after a warm-up:
- factor_solve alone;
- factor_solve_policy with all four arrays (K, k, V, v), and with K, k only;
- the export kernels alone (sipoc_profile_*): the gathers of K, k, v (policy_gather_kernel)
  and the V rebuild (policy_rebuild_v_kernel), each with its bytes computed from the sizes --
  what it must read per problem and the lanes of batch_stride it writes -- its bandwidth and
  share of 7.7 TB/s (the HGX B200 data-sheet HBM3e rate of one GPU).
A seeded sample of problems is checked against the CPU reference (policy_reference.py).  The
device name, power limit and max SM clock are read in the same run.  Usage:
    python tools/bench_policy.py --out profiles/r07/bench_policy.json [--workloads quadrotor,...]
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

from bench_vjp import device_info, event_ms  # noqa: E402
from gpu_helpers import rel_err, to_structs  # noqa: E402
from oracle import pyoracle  # noqa: E402
from policy_reference import POLICY_NAMES, SIZE_OF, lqr_policy  # noqa: E402
from sip_optimal_control_b200 import LQR  # noqa: E402
from sip_optimal_control_b200._capi import lib  # noqa: E402

PEAK_TBS = 7.7
WORKLOADS = {  # name: (n, m, T, batch)
    "quadrotor": (12, 4, 50, 65536),
    "cartpole": (4, 1, 100, 65536),
    "humanoid": (64, 24, 32, 4096),
    "long_horizon": (12, 4, 4096, 64),  # runs on the parallel-in-time scan
}


def tri(n):
    return n * (n + 1) // 2


def gather_bytes(n, m, T, batch, ld, want):
    """K, k, v: each element read once per problem and written once per lane."""
    count = dict(K=T * n * m, k=T * m, v=(T + 1) * n)
    return sum(8 * (batch + ld) * count[k] for k in want) + 4 * ld * len(want)


def rebuild_bytes(n, m, T, batch, ld):
    """V: per edge Q (lower), M, A, B, delta of the child, P of the child (packed), K read once;
    the terminal Q (lower); every V entry written once per lane."""
    per_edge = tri(n) + n * m + n * n + n * m + n + tri(n) + n * m
    return 8 * batch * (T * per_edge + tri(n)) + 8 * ld * (T + 1) * n * n + 4 * ld


def profiled_ms(eng, fn, iters):
    lib.sipoc_profile_enable(eng._handle, 1)
    for _ in range(iters):
        fn()
    got = {}
    for i in range(lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        eng._check(lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                                         ctypes.byref(cnt)))
        got[nm.value.decode()] = (ms.value / iters, cnt.value)
    lib.sipoc_profile_enable(eng._handle, 0)
    return got


def run(name, n, m, T, batch, warmup, iters, sample):
    s = pyoracle.Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    sz = e.lqr_sizes
    inp = lqr.generate_benchmark(seed=2026)
    out = lqr.alloc_output()
    status = e.empty_int()
    pol = {k: e.empty(sz[SIZE_OF[k]]) for k in POLICY_NAMES}
    forward = lambda: lqr.factor_solve(inp, out, status=status)
    policy_all = lambda: lqr.factor_solve_policy(inp, out, policy=pol, status=status)
    policy_kk = lambda: lqr.factor_solve_policy(inp, out, want=("K", "k"), policy=pol,
                                                status=status)
    line = dict(workload=name, n=n, m=m, T=T, batch=batch, batch_stride=e.batch_stride,
                kernel_variant=e.kernel_variant, iters=iters)
    line["factor_solve_ms"] = event_ms(forward, warmup, iters)
    line["policy_all_ms"] = event_ms(policy_all, warmup, iters)
    line["policy_K_k_ms"] = event_ms(policy_kk, warmup, iters)
    prof = profiled_ms(e, policy_all, iters)
    ld = e.batch_stride
    g_ms, g_cnt = prof["policy_gather_kernel"]
    gb = gather_bytes(n, m, T, batch, ld, ("K", "k", "v"))
    line["gather_K_k_v"] = dict(ms=g_ms, launches_per_call=g_cnt / iters, bytes=gb,
                                tb_per_s=gb / (g_ms * 1e-3) / 1e12,
                                share_of_7_7_tb_per_s=gb / (g_ms * 1e-3) / 1e12 / PEAK_TBS)
    r_ms, _ = prof["policy_rebuild_v_kernel"]
    rb = rebuild_bytes(n, m, T, batch, ld)
    line["rebuild_V"] = dict(ms=r_ms, bytes=rb, tb_per_s=rb / (r_ms * 1e-3) / 1e12,
                             share_of_7_7_tb_per_s=rb / (r_ms * 1e-3) / 1e12 / PEAK_TBS)
    # seeded sample against the CPU reference, from a last all-array call
    policy_all()
    torch.cuda.synchronize()
    assert bool((status[:batch] == 0).all())
    idx = torch.from_numpy(np.random.default_rng(11).choice(batch, min(sample, batch),
                                                            replace=False)).to(e.torch_device())
    pick = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: pick(inp[k], sz[k]) for k in pyoracle.LQR_INPUT_NAMES}
    ref = lqr_policy(s, host)
    line["sample_problems"] = int(idx.numel())
    line["sample_max_rel_err"] = {k: float(rel_err(pick(pol[k], sz[SIZE_OF[k]]), ref[k]).max())
                                  for k in POLICY_NAMES}
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
        sys.exit("bench_policy.py needs a CUDA device")
    torch.cuda.set_device(0)
    result = dict(tool="tools/bench_policy.py", **device_info(), peak_tb_per_s=PEAK_TBS, runs=[])
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
