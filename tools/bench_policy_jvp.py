"""Timing of the policy JVP (sipoc_lqr_policy_jvp, the tangent Riccati sweep) on the GPU.

Per workload (inputs from sipoc_generate_lqr_benchmark, tangents seeded), with CUDA events
after a warm-up:
- the forward factor_solve_policy with all four arrays (K, k, V, v);
- the policy_jvp call with all nine tangents, and with the vector tangents (q, r, c) only;
- the policy_vjp call with all four cotangents and all nine gradients, for comparison;
- the JVP kernel alone (sipoc_profile_*), with its compulsory bytes and FP64 FMAs computed
  from the shapes below, the achieved rates, and the kernel's share of whichever bound applies
  (7.7 TB/s, the HGX B200 data-sheet HBM3e rate of one GPU; 64 FP64 FMA/clk/SM x 148 SMs at
  the max SM clock read in the same run, DESIGN.md 2.5).
Every working set is larger than the 126 MB L2 except long_horizon's (64 problems).  A seeded
sample of problems is checked against the CPU sweep (policy_jvp_reference.py).  The device
name, power limit and max SM clock are read in the same run.  Usage:
    python tools/bench_policy_jvp.py --out profiles/r09/bench_policy_jvp.json [--workloads ...]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from bench_policy import profiled_ms, tri  # noqa: E402
from bench_vjp import device_info, event_ms  # noqa: E402
from gpu_helpers import rel_err, to_structs  # noqa: E402
from oracle import pyoracle  # noqa: E402
from policy_reference import POLICY_NAMES, SIZE_OF  # noqa: E402
from policy_jvp_reference import policy_jvp  # noqa: E402
from policy_vjp_reference import INPUT_NAMES  # noqa: E402
from sip_optimal_control_b200 import LQR  # noqa: E402

PEAK_TBS = 7.7
FMA_PER_CLK_SM = 64
SMS = 148
WORKLOADS = {  # name: (n, m, T, batch)
    "quadrotor": (12, 4, 50, 65536),
    "cartpole": (4, 1, 100, 65536),
    "humanoid": (64, 24, 32, 4096),
    "long_horizon": (12, 4, 4096, 64),  # forward on the parallel-in-time scan
}


def compulsory_bytes(n, m, T, batch, ld):
    """Read once per problem: per edge R (lower), M, r, A, B and the child's c, delta, V (lower),
    v, and the tangents of M, R, r, A, B, the child's c, delta, and the parent's Q, q; the last
    node's tangents of Q, q.  Written once per lane of batch_stride: dK, dk, dV, dv.  Plus the
    status word."""
    per_edge = tri(m) + n * m + m + n * n + n * m + n + n + tri(n) + n \
        + n * m + m * m + m + n * n + n * m + n + n + n * n + n
    reads = T * per_edge + n * n + n
    writes = T * (n * m + m) + (T + 1) * (n * n + n)
    return 8 * batch * reads + 8 * ld * writes + 4 * batch


def sweep_fmas(n, m):
    """FP64 FMAs of one edge of the sweep as written in policy_jvp.cu (n = n_p = n_c): the
    primal recompute (Cholesky factor and inverse of F, W, G and its factor, Y, K, f, g, h, k),
    then T = dV_c S, dW, dW B, dW A, dG, df, dY, dg, dH, dh, dG K, the solves with G for dK and
    dk, and the lower triangle of dV_p and dv_p."""
    n3, n2m, nm2 = n ** 3, n * n * m, n * m * m
    primal = n3 / 6 + n3 + 2 * n * n + n2m + nm2 / 2 + m ** 3 / 6 + n3 + n2m + nm2 + 2 * n * n \
        + n * m + m * m
    tangent = n3 + 2 * n3 + n2m + n3 + 3 * nm2 + n + n3 + 2 * n * n + 2 * n2m + 2 * n * m \
        + nm2 + m * m + nm2 + m * m + (3 * n3 + 3 * n2m) / 2 + 2 * n * n + 2 * n * m
    return primal + tangent


def run(name, n, m, T, batch, warmup, budget_s, sample):
    s = pyoracle.Structure.chain(T, n, m)
    dims, topo = to_structs(s)
    lqr = LQR(dims, topo, batch)
    e = lqr.engine
    sz = e.lqr_sizes
    inp = lqr.generate_benchmark(seed=2026)
    out = lqr.alloc_output()
    status = e.empty_int()
    pol = {k: e.empty(sz[SIZE_OF[k]]) for k in POLICY_NAMES}
    gen = torch.Generator(device=e.torch_device()).manual_seed(7)
    rand = lambda t: torch.randn(tuple(t.shape), dtype=torch.float64, device=e.torch_device(),
                                 generator=gen)
    tan = {k: rand(inp[k]) for k in INPUT_NAMES}
    vec_tan = {k: tan[k] for k in ("q", "r", "c")}
    cot = {k: rand(pol[k]) for k in POLICY_NAMES}
    dpol = {k: e.empty(sz[SIZE_OF[k]]) for k in POLICY_NAMES}
    grads = {k: e.empty(sz[k]) for k in INPUT_NAMES}
    forward = lambda: lqr.factor_solve_policy(inp, out, policy=pol, status=status)
    jvp = lambda: lqr.policy_jvp(inp, pol, status, tan, dpolicy=dpol)
    jvp_vec = lambda: lqr.policy_jvp(inp, pol, status, vec_tan, dpolicy=dpol)
    vjp = lambda: lqr.policy_vjp(inp, pol, status, cot, grad=grads)
    forward()
    once = max(event_ms(jvp, 1, 1), event_ms(vjp, 1, 1))  # warms the modules, sizes the window
    iters = int(max(2, min(20, budget_s * 1e3 / max(once, 1e-3))))
    line = dict(workload=name, n=n, m=m, T=T, batch=batch, batch_stride=e.batch_stride,
                forward_variant=e.kernel_variant, iters=iters)
    line["forward_policy_ms"] = event_ms(forward, warmup, iters)
    forward()
    line["policy_jvp_ms"] = event_ms(jvp, warmup, iters)
    line["policy_jvp_vector_tangents_ms"] = event_ms(jvp_vec, warmup, iters)
    line["policy_vjp_ms"] = event_ms(vjp, warmup, iters)
    prof = profiled_ms(e, jvp, iters)
    (kname, (k_ms, k_cnt)), = prof.items()
    ld = e.batch_stride
    nbytes = compulsory_bytes(n, m, T, batch, ld)
    fmas = sweep_fmas(n, m) * T * batch
    line["kernel"] = dict(name=kname, ms=k_ms, launches_per_call=k_cnt / iters,
                          compulsory_bytes=nbytes, fp64_fmas=fmas,
                          tb_per_s=nbytes / (k_ms * 1e-3) / 1e12,
                          tfma_per_s=fmas / (k_ms * 1e-3) / 1e12)
    # seeded sample against the CPU sweep
    jvp()
    torch.cuda.synchronize()
    assert bool((status[:batch] == 0).all())
    idx = torch.from_numpy(np.random.default_rng(11).choice(batch, min(sample, batch),
                                                            replace=False)).to(e.torch_device())
    pick = lambda t, size: t[:size].index_select(1, idx).T.contiguous().cpu().numpy()
    host = {k: pick(inp[k], sz[k]) for k in INPUT_NAMES}
    ref = policy_jvp(s, host, {k: pick(tan[k], sz[k]) for k in INPUT_NAMES})
    line["sample_problems"] = int(idx.numel())
    line["sample_max_rel_err"] = {k: float(rel_err(pick(dpol[k], sz[SIZE_OF[k]]), ref[k]).max())
                                  for k in POLICY_NAMES}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--budget-s", type=float, default=1.0, help="timed window per measurement")
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_policy_jvp.py needs a CUDA device")
    torch.cuda.set_device(0)
    info = device_info()
    clock = info.get("max_sm_clock", "")
    ghz = float(clock.split()[0]) / 1e3 if clock else None
    result = dict(tool="tools/bench_policy_jvp.py", **info, peak_tb_per_s=PEAK_TBS,
                  peak_fp64_tfma_per_s=SMS * FMA_PER_CLK_SM * ghz / 1e3 if ghz else None, runs=[])
    for name in args.workloads.split(","):
        line = run(name, *WORKLOADS[name], args.warmup, args.budget_s, args.sample)
        k = line["kernel"]
        bw = k["tb_per_s"] / PEAK_TBS
        fp = k["tfma_per_s"] / result["peak_fp64_tfma_per_s"] if ghz else None
        k["share_of_7_7_tb_per_s"] = bw
        k["share_of_fp64_fma_peak"] = fp
        k["bound"] = "fp64" if fp is not None and fp > bw else "bytes"
        print(json.dumps(line), flush=True)
        result["runs"].append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
