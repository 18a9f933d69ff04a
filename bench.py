#!/usr/bin/env python
"""Headline benchmark: batched regularized-LQR factor + solve, solves/sec in FP64.

One *step* = one pass of the hot path over one batch of synthetic problems:
the factor + solve of every problem of the batch (reference loop body of
BM_LQRFactorSolve, benchmarks/lqr_benchmark.cpp:653-663) followed by the
failure-flag reduction a Newton iteration all-reduces.  Inputs are resident in
HBM in the engine layout when the timed region starts (``value``); ``e2e`` is
the same metric through the host-buffer C-ABI call with the host<->device
copies inside the timed region.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --steps K --warmup W     # CPU reference arm

For N > 1 launch under torch.distributed.run (one rank per GPU); the batch is
sharded with no data-path collective, the only traffic being the all-reduce of
the 4-double statistics vector per step.  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs: (state dim n, control dim m, horizon T, batch).
WORKLOADS = {
    "cartpole": dict(n=4, m=1, T=100, batch=16384),
    "quadrotor": dict(n=12, m=4, T=50, batch=65536),
    "humanoid": dict(n=64, m=24, T=32, batch=4096),
    # Config 5's long-horizon, small-batch case at both dims SURVEY section 8d names.  The
    # parallel-in-time scan is not built: these run the sequential-in-time kernels above.
    "long_horizon_quadrotor": dict(n=12, m=4, T=4096, batch=64),
    "long_horizon_humanoid": dict(n=64, m=24, T=4096, batch=64),
}
# Config 4: Newton-KKT with inequality constraints and variable per-stage dims — the
# pattern of tests/variable_dimensions_test.cpp:266-271 tiled along the horizon.
KKT_WORKLOAD = dict(T=48, batch=8192, state=(2, 1, 3), control=(1, 2), node_c=(1, 0, 2),
                    node_g=(0, 2, 1), edge_c=(1, 2), edge_g=(2, 1))
# The uniform newton_kkt_benchmark.cpp shape (:58-93): c = max(1, n/2), g = max(1, 2m) on
# every edge, node constraints only at the terminal node; quadrotor dims.
KKT_UNIFORM = dict(T=50, batch=8192, n=12, m=4)
DEFAULT_WORKLOAD = "quadrotor"  # the config north_star quotes its target on
METRIC = "batched LQR factor+solve solves/sec (FP64)"
UNIT = "solves/s"
FP64_PEAK_TFLOPS = 36.8  # DFMA peak measured on this pool (profiles/microbench)


def algorithmic_bytes(n, m, T):
    """SURVEY.md 8(d): compulsory in + out bytes of one factor+solve."""
    inb = 8 * ((T + 1) * (n * n + 3 * n) + T * (n * n + 2 * n * m + m * m + m))
    outb = 8 * ((T + 1) * 2 * n + T * m)
    return inb, outb


def algorithmic_flops(n, m, T):
    """SURVEY.md 8(d): the reference's operation count of one factor+solve."""
    factor = T * (19 * n ** 3 / 3 + 6 * m * n * n + 4 * m * m * n + m ** 3 / 3) \
        + n ** 3 / 3 + 2 * (T + 1) * n * n
    solve = T * (10 * n * n + 8 * n * m + 2 * m * m) + 4 * n * n
    return factor + solve


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# --------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks DURING the timed region")
# --------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, gpu_index: int):
        self.samples = []  # (host time, sm MHz, max MHz, [reasons])
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50", "-i", str(gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm, mx = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            reasons = [n for n, v in zip(self.NAMES, parts[2:6]) if v.lower().startswith("active")]
            self.samples.append((time.time(), sm, mx, reasons))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float):
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        window = "timed region"
        if not inside:  # region shorter than the sampling period
            inside = [s for s in self.samples if t0 - 0.5 <= s[0] <= t1 + 0.2]
            window = "timed region +-0.5 s"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({r for s in inside for r in s[3]})
        return {"sm_mhz": float(np.median([s[1] for s in inside])),
                "sm_max_mhz": float(max(s[2] for s in inside)), "reasons": reasons,
                "samples": len(inside), "window": window}


# --------------------------------------------------------------------------
# host-side synthetic problems (reference arm / cpu baseline): the distribution
# of benchmarks/lqr_benchmark.cpp:61-96, numpy stream.
# --------------------------------------------------------------------------
def host_problems(n, m, T, batch, seed):
    rng = np.random.default_rng(seed)

    def spd(count, d, shift):
        Z = rng.standard_normal((batch, count, d, d))
        return np.einsum("bckj,bcki->bcij", Z, Z) + shift * np.eye(d)

    def cm(x):
        return np.ascontiguousarray(np.swapaxes(x, -1, -2)).reshape(batch, -1)

    return dict(
        Q=cm(spd(T + 1, n, 1e-3)), M=np.zeros((batch, T * n * m)), R=cm(spd(T, m, 1.01)),
        q=rng.standard_normal((batch, (T + 1) * n)), r=rng.standard_normal((batch, T * m)),
        A=cm(0.05 * rng.standard_normal((batch, T, n, n)) + np.eye(n)),
        B=cm(0.1 * rng.standard_normal((batch, T, n, m))),
        c=rng.standard_normal((batch, (T + 1) * n)),
        delta=1e-3 + 1e-1 * rng.random((batch, (T + 1) * n)))


def cpu_time_sample(wl, sample, nthreads, repeats=1, host=None):
    """Seconds for the oracle to factor+solve `sample` problems, `repeats` times."""
    from oracle import pyoracle

    s = pyoracle.Structure.chain(wl["T"], wl["n"], wl["m"])
    if host is None:
        host = host_problems(wl["n"], wl["m"], wl["T"], sample, seed=1234)
    out = pyoracle.lqr_factor_solve(s, host, solve=True, residual=False, repeats=repeats,
                                    nthreads=nthreads)
    assert (out["status"] == 0).all()
    return out["seconds"], host


def host_threads():
    """All the host threads this process may use.  Not omp_get_max_threads(): torchrun exports
    OMP_NUM_THREADS=1 to every rank, which would leave the CPU arm on one core at N > 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(wl, target_seconds=10.0):
    """Oracle (port of the reference) across all host cores on a bounded sample."""
    from oracle import pyoracle

    cores = host_threads()
    sample = max(cores * 8, 64)
    _, host = cpu_time_sample(wl, sample, cores)  # warm-up: page in, spin up the threads
    total, reps = 0.0, 0
    while total < target_seconds and reps < 100000:
        secs, _ = cpu_time_sample(wl, sample, cores, host=host)
        total += secs
        reps += 1
    value = sample * reps / total
    return {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{sample} problems of the workload x {reps} passes "
                      f"({total:.1f} s), one problem per OpenMP thread, oracle/liboracle.so"}


# --------------------------------------------------------------------------
def run_reference(args, wl, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import pyoracle

    cores = host_threads()
    # One step = the workload's whole batch (the GPU arm's config: same_config), as
    # `passes` sweeps over a pool of distinct problems: 65 536 quadrotor problems would be
    # 11.6 GB of host arrays, the pool (<= 2 048 problems, 360 MB, far beyond the CPU caches) keeps
    # the arm's set-up to seconds.  Warm-up is bounded to what half a minute allows.
    batch = wl["batch"]
    pool = min(batch, 2048)
    while batch % pool:
        pool -= 1
    passes = batch // pool
    host = host_problems(wl["n"], wl["m"], wl["T"], pool, seed=1234)
    secs, _ = cpu_time_sample(wl, pool, cores, host=host)  # warm-up pass, sizes the warm-up
    step_s = secs * passes
    steps = args.steps
    warm = max(0, min(args.warmup, int(30.0 / max(step_s, 1e-9))))
    for _ in range(warm):
        cpu_time_sample(wl, pool, cores, repeats=passes, host=host)
    total = 0.0
    for _ in range(steps):
        s, _ = cpu_time_sample(wl, pool, cores, repeats=passes, host=host)
        total += s
    value = batch * steps / total
    sample = batch
    desc = (f"{batch} problems per step ({passes} passes over {pool} distinct problems), {steps} timed "
            f"steps, one problem per OpenMP thread over {cores} threads; "
            "Eigen-free port of lqr.cpp (the reference itself needs Eigen, absent here)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * total / steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": name, **wl, "batch": sample, "global_batch": sample,
                   "note": "host CPU arm: the workload's whole batch per step; warm-up bounded "
                           "to half a minute of CPU time"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------
def load_traffic(name, kernels, batch):
    """DRAM traffic (dram__bytes_read + dram__bytes_write) of the hot-path kernels of one step
    on this rank, from the committed ncu captures: profiles/traffic.json holds bytes per
    problem for every kernel of a workload; the kernels that ran this step are summed."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            per_problem = json.load(f).get(name, {})
        known = [per_problem[k] for k in kernels if k in per_problem]
        if not known or len(known) < sum(1 for k in kernels if k != "status_stats_kernel"):
            return None
        return float(sum(known)) * batch
    except Exception:
        return None


# --dump-outputs keeps the whole dump under DUMP_BYTES: when every problem does not fit, it writes
# the rows np.sort(np.random.default_rng(DUMP_SEED).choice(batch, k, replace=False)) of every
# per-problem array, so two builds run with the same arguments write the same problems.
DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 0


def dump_outputs(directory, batch, per_problem, whole):
    """Writes DIR/<name>.npy for the arrays the timed call returned in its last step.

    per_problem: name -> device tensor, either [size, batch_stride] (engine layout, written as
    [problems, size]) or [batch_stride] (one value per problem); whole: name -> device tensor
    written as it is.  Floating arrays keep their precision, integer ones are written as float64.
    """
    import torch

    def itemsize(t):
        return t.element_size() if t.is_floating_point() else 8

    fixed = sum(t.numel() * itemsize(t) for t in whole.values())
    per_row = sum((t.shape[0] if t.dim() == 2 else 1) * itemsize(t) for t in per_problem.values())
    headers = 256 * (len(per_problem) + len(whole))
    k = min(batch, (DUMP_BYTES - headers - fixed) // per_row)
    rows = np.arange(batch)
    if k < batch:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(batch, k, replace=False))
    os.makedirs(directory, exist_ok=True)
    arrays = dict(whole)
    for name, t in per_problem.items():
        idx = torch.from_numpy(rows).to(t.device)
        arrays[name] = t[:, idx].T if t.dim() == 2 else t[idx]
    for name, t in arrays.items():
        t = t if t.is_floating_point() else t.to(torch.float64)
        np.save(os.path.join(directory, f"{name}.npy"), t.contiguous().cpu().numpy())
    print(f"bench: wrote {len(arrays)} arrays of the last timed step to {directory} "
          f"({k} of {batch} problems)", file=sys.stderr)


def run_ours(args, wl, name):
    import torch
    import torch.distributed as dist

    from sip_optimal_control_b200 import LQR, Dimensions, Topology, _capi
    from sip_optimal_control_b200._capi import lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one process: run it with --gpus 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's banner ("NCCL version ...") belongs on stderr: stdout carries the JSON line and
        # nothing else.  NCCL_DEBUG_FILE does not catch it on every build, so file descriptor 1
        # points at stderr while the communicator comes up (init + the first collective).
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(4, dtype=torch.float64, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    assert world == args.gpus, (world, args.gpus)

    from sip_optimal_control_b200.sharding import Communicator, shard_range

    n, m, T = wl["n"], wl["m"], wl["T"]
    # weak: every GPU gets the workload's batch; strong: the workload's batch is
    # cut into contiguous shards (sharding.shard_range).
    total_batch = wl["batch"] * (world if args.scaling == "weak" else 1)
    first, last = shard_range(total_batch, rank, world)
    batch = last - first
    sampler = ClockSampler(local_rank) if rank == 0 else None

    lqr = LQR(Dimensions.uniform(T, n, m), Topology.chain(T), batch, device=local_rank,
              force_generic=args.force_generic,
              parallel_in_time=False if args.serial_in_time else None)
    eng = lqr.engine
    inp = lqr.generate_benchmark(seed=args.seed, problem_offset=first)
    out = lqr.alloc_output()
    status = eng.empty_int()
    stats = torch.zeros(4, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev)
    sp = eng.stream_ptr(stream)
    comm = None
    if world > 1:
        # The per-iteration exchange belongs to the engine: with its communicator attached
        # (include/sipoc.h, sipoc_attach_comm) sipoc_status_stats ends with the all-reduce of
        # the 4 statistics -- one NCCL all-gather + a one-warp fold kernel on the step's stream.
        comm = Communicator(device=local_rank)
        comm.attach(eng)

    inp_pm = None
    if args.input_layout == "problem_major":
        # The same inputs, problem-major on the device (sipoc_lqr_factor_solve_pm): transposed
        # once here, outside the timed region -- they are resident in HBM in the layout the call takes.
        inp_pm = {}
        for k in _capi.LQR_INPUT_FIELDS:
            size = inp[k].numel() // eng.batch_stride
            dst = torch.empty((batch, size), dtype=torch.float64, device=dev)
            eng._check(lib.sipoc_unpack(eng._handle, inp[k].data_ptr(), dst.data_ptr(), size, sp))
            inp_pm[k] = dst
        torch.cuda.synchronize(dev)

    inp32 = out32 = None
    if args.fp32:
        # Optional FP32 mode (north_star; sipoc_lqr_factor_solve_f32): every array in single
        # precision, narrowed once outside the timed region.  Reported as its own line
        # (dtype f32, the algorithmic bytes halve), never mixed with the FP64 numbers.
        if not lqr.f32_supported:
            raise SystemExit("--fp32: the FP32 mode covers uniform chains with n = 4, m = 1..4 "
                             "(workload cartpole)")
        inp32, out32 = lqr.narrow_f32(inp), lqr.alloc_output_f32()

    def step():
        if inp32 is not None:
            lqr.factor_solve_f32(inp32, out32, status=status, stream=stream)
        elif inp_pm is not None:
            lqr.factor_solve_pm(inp_pm, out, status=status, stream=stream)
        else:
            lqr.factor_solve(inp, out, status=status, stream=stream)
        # (all-reduced over the ranks inside the call when world > 1)
        eng._check(lib.sipoc_status_stats(eng._handle, status.data_ptr(), stats.data_ptr(), sp))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = eng.launch_count
    lib.sipoc_profile_enable(eng._handle, 1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    t1 = time.time()
    ms_total = ev0.elapsed_time(ev1)
    gpu_launches = eng.launch_count - launches0
    failed_total, count_total = float(stats[2].item()), float(stats[3].item())

    # per-kernel device time over the same timed region
    kernels = {}
    for i in range(lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                              ctypes.byref(cnt))
        kernels[nm.value.decode()] = {"ms_per_launch": ms.value / max(cnt.value, 1),
                                      "launches_per_step": cnt.value / args.steps,
                                      "ms_per_step": ms.value / args.steps}
    lib.sipoc_profile_enable(eng._handle, 0)

    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = total_batch / (ms_per_step * 1e-3)

    if args.dump_outputs:
        sizes = eng.lqr_sizes
        last = out32 if out32 is not None else out
        dump_outputs(args.dump_outputs, batch,
                     {**{k: last[k][:sizes[k]] for k in _capi.LQR_OUTPUT_FIELDS}, "status": status},
                     {"stats": stats})

    # correctness outside the timed region: KKT residual of every problem
    if inp32 is not None:
        # FP32 mode: the residual of the single-precision solution, evaluated in FP64 against
        # the float-rounded problem it solved
        inp = {k: v.double() for k, v in inp32.items()}
        out = {k: v.double() for k, v in out32.items()}
    norms, rstats = lqr.residual(inp, out, status)  # (all-reduced inside the call too)
    max_residual = float(rstats[1].item())

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region ----
    # One call solves the GPU's whole shard (65 536 problems at N = 1: 11.6 GB of pinned
    # host inputs); --e2e-batch caps the call size.  The call is PCIe-bound (189 KB cross
    # the bus per problem).
    e2e = None
    if not args.no_e2e and not args.fp32:
        hb = min(batch, args.e2e_batch) if args.e2e_batch > 0 else batch
        lqr_h = lqr if hb == batch else LQR(Dimensions.uniform(T, n, m), Topology.chain(T), hb,
                                            device=local_rank, force_generic=args.force_generic)
        eng_h = lqr_h.engine
        inp_h = inp if hb == batch else lqr_h.generate_benchmark(seed=args.seed,
                                                                 problem_offset=first)
        sizes = eng_h.lqr_sizes
        host_in, keep = {}, []
        for k in _capi.LQR_INPUT_FIELDS:
            pinned = torch.empty((hb, max(sizes[k], 1)), dtype=torch.float64, pin_memory=True)
            tmp = torch.empty((hb, max(sizes[k], 1)), dtype=torch.float64, device=dev)
            eng_h._check(lib.sipoc_unpack(eng_h._handle, inp_h[k].data_ptr(), tmp.data_ptr(),
                                          sizes[k], sp))
            pinned.copy_(tmp)
            del tmp
            host_in[k] = pinned.numpy()
            keep.append(pinned)
        host_out = {}
        for k in _capi.LQR_OUTPUT_FIELDS:
            pinned = torch.empty((hb, max(sizes[k], 1)), dtype=torch.float64, pin_memory=True)
            host_out[k] = pinned.numpy()
            keep.append(pinned)
        torch.cuda.synchronize(dev)
        e2e_steps = max(1, args.e2e_steps)
        res = lqr_h.factor_solve_host(host_in, host_out)  # warm-up: allocates resident buffers
        barrier()
        te0 = time.perf_counter()
        for _ in range(e2e_steps):
            res = lqr_h.factor_solve_host(host_in, host_out)
        torch.cuda.synchronize(dev)
        te = torch.tensor([time.perf_counter() - te0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        assert (res["status"] == 0).all()
        h2d = sum(hb * sizes[k] * 8 for k in _capi.LQR_INPUT_FIELDS)
        d2h = sum(hb * sizes[k] * 8 for k in _capi.LQR_OUTPUT_FIELDS) + hb * 4
        e2e = {"value": hb * world * e2e_steps / float(te.item()), "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
               "problems_per_call_per_gpu": hb,
               "call": "sipoc_lqr_factor_solve_host (pinned host buffers, problem-major)"}
        if args.e2e_packed and n < 16:
            # The same call through sipoc_lqr_factor_solve_host_packed: Q / R as packed lower
            # triangles, M not sent (the reference benchmark's M is zero, lqr_benchmark.cpp:61-96).
            # NOT the reference's dense interface: an extra key, never the headline e2e.
            packed_in = dict(host_in)
            for k, dim in (("Q", n), ("R", m)):
                tri = LQR.pack_symmetric(host_in[k], dim)
                pinned = torch.empty(tri.shape, dtype=torch.float64, pin_memory=True)
                pinned.numpy()[...] = tri
                packed_in[k] = pinned.numpy()
                keep.append(pinned)
            packed_in["M"] = None
            res = lqr_h.factor_solve_host_packed(packed_in, host_out)
            barrier()
            tp0 = time.perf_counter()
            for _ in range(e2e_steps):
                res = lqr_h.factor_solve_host_packed(packed_in, host_out)
            torch.cuda.synchronize(dev)
            tp = torch.tensor([time.perf_counter() - tp0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            assert (res["status"] == 0).all()
            h2dp = sum(hb * packed_in[k].shape[1] * 8 for k in _capi.LQR_INPUT_FIELDS
                       if packed_in[k] is not None)
            e2e["packed"] = {"value": hb * world * e2e_steps / float(tp.item()), "unit": UNIT,
                             "h2d_bytes_per_step": h2dp, "d2h_bytes_per_step": d2h,
                             "call": "sipoc_lqr_factor_solve_host_packed (Q, R packed lower "
                                     "triangles, M = NULL; not the reference's dense interface)"}

    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(t0, t1)
        inb, outb = algorithmic_bytes(n, m, T)
        if args.fp32:
            inb, outb = inb // 2, outb // 2  # the same element counts, four bytes each
        flops = algorithmic_flops(n, m, T)
        peak, peak_kind = measured_peaks()
        hot = {k: v for k, v in kernels.items() if k != "status_stats_kernel"}
        # The roofline uses the step's device time (kernels + launch gaps), not the sum of
        # the per-kernel times: conservative, and valid if kernels ever overlap.
        hot_sum = sum(v["ms_per_step"] for v in hot.values())
        hot_ms = ms_per_step
        dominant = max(hot, key=lambda k: hot[k]["ms_per_step"]) if hot else None
        t_hbm = (inb + outb) * batch / (peak * 1e9)
        t_f64 = flops * batch / (FP64_PEAK_TFLOPS * 1e12)
        if t_hbm >= t_f64:
            achieved = (inb + outb) * batch / (hot_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak}
        else:
            achieved = flops * batch / (hot_ms * 1e-3) / 1e12
            roof = {"bound": "fp64", "achieved": achieved, "peak": FP64_PEAK_TFLOPS,
                    "unit": "TFLOP/s", "frac": achieved / FP64_PEAK_TFLOPS}
        roof.update({
            "peak_source": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs; FP64 = DFMA microbench)",
            "traffic": load_traffic(name, hot, batch),
            "algorithmic_bytes_per_solve": inb + outb,
            "algorithmic_flops_per_solve": flops,
            "basis": "algorithmic bytes of one factor+solve x problems per step / device time of "
                     "the step (CUDA events around the timed region); kernels lists the per-launch "
                     "CUDA-event times of the same region",
            "dominant_kernel": dominant,
            "dominant_share": (hot[dominant]["ms_per_step"] / hot_sum) if dominant else None,
            "kernels": kernels,
        })
        line = {
            "metric": METRIC.replace("FP64", "FP32 mode, reported separately") if args.fp32
            else METRIC,
            "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if args.fp32 else "f64", "data": "synthetic",
            "config": {"workload": name, "n": n, "m": m, "T": T, "batch_per_gpu": batch,
                       "global_batch": total_batch, "parallelism": f"batch-sharded x{world}",
                       "kernel_variant": eng.kernel_variant, "input_layout": args.input_layout,
                       "l2": "inputs larger than L2 (no flush needed)"
                       if (inb * batch > 2 * 126e6) else "inputs smaller than L2",
                       "generator": "lqr_benchmark.cpp:61-96 distribution, counter-based RNG"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches),
            "roofline": roof,
            "check": {"failed_problems": failed_total, "problems": count_total,
                      "max_kkt_residual": max_residual},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wl)
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def kkt_host_problem(dims, batch, seed, r2_max=1e9):
    """newton_kkt_benchmark.cpp:171-240 distribution on a chain with the given dims."""
    rng = np.random.default_rng(seed)
    sd, cd = dims.state_dims, dims.control_dims
    N, E = len(sd), len(cd)

    def cm(x):
        return np.ascontiguousarray(np.swapaxes(x, -1, -2)).reshape(batch, -1)

    def spd(d, shift):
        Z = rng.standard_normal((batch, d, d))
        return np.einsum("bkj,bki->bij", Z, Z) + shift * np.eye(d)

    m = {k: [] for k in ("node_hxx", "node_jc", "node_jg", "edge_hxx", "edge_hxu", "edge_huu",
                         "edge_A", "edge_B", "edge_jcx", "edge_jcu", "edge_jgx", "edge_jgu")}
    for i in range(N):
        n = int(sd[i])
        m["node_jc"].append(cm(0.1 * rng.standard_normal((batch, int(dims.node_c_dims[i]), n))))
        m["node_jg"].append(cm(0.1 * rng.standard_normal((batch, int(dims.node_g_dims[i]), n))))
        m["node_hxx"].append(cm(spd(n, 1e-3)))
    for e in range(E):
        npar, nch, mm = int(sd[e]), int(sd[e + 1]), int(cd[e])
        c, g = int(dims.edge_c_dims[e]), int(dims.edge_g_dims[e])
        A = 0.05 * rng.standard_normal((batch, nch, npar))
        if nch == npar:
            A = A + np.eye(nch)
        m["edge_A"].append(cm(A))
        m["edge_B"].append(cm(0.1 * rng.standard_normal((batch, nch, mm))))
        m["edge_jcx"].append(cm(0.1 * rng.standard_normal((batch, c, npar))))
        m["edge_jcu"].append(cm(0.1 * rng.standard_normal((batch, c, mm))))
        m["edge_jgx"].append(cm(0.1 * rng.standard_normal((batch, g, npar))))
        m["edge_jgu"].append(cm(0.1 * rng.standard_normal((batch, g, mm))))
        m["edge_hxx"].append(np.zeros((batch, npar * npar)))
        m["edge_hxu"].append(cm(0.01 * rng.standard_normal((batch, npar, mm))))
        m["edge_huu"].append(cm(spd(mm, 1.0)))
    model = {k: np.concatenate(v, axis=1) for k, v in m.items()}
    x_dim, y_dim, z_dim = dims.get_x_dim(E), dims.get_y_dim(E), dims.get_z_dim(E)

    def logu(shape, lo, hi):
        return np.exp(np.log(lo) + (np.log(hi) - np.log(lo)) * rng.random(shape))

    return (model, logu((batch, z_dim), 1e-2, 1e3), np.full((batch, x_dim), 1e-8),
            logu((batch, y_dim), 1e-3, r2_max), logu((batch, z_dim), 1e-3, 1e1),
            rng.standard_normal((batch, x_dim + y_dim + z_dim)))


def run_kkt(args):
    """Config 4: KKT factor + KKT solve + KKT residual per step, variable per-stage dims."""
    import torch

    from sip_optimal_control_b200 import CallbackProvider, Dimensions, Topology
    from sip_optimal_control_b200._capi import lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    uniform = args.workload == "newton_kkt_uniform"
    wl = dict(KKT_UNIFORM if uniform else KKT_WORKLOAD)
    if args.batch:
        wl["batch"] = args.batch
    T, batch = wl["T"], wl["batch"]
    if uniform:
        n, m = wl["n"], wl["m"]
        c, g = max(1, n // 2), max(1, 2 * m)
        term = lambda v: np.array([0] * T + [v], np.int32)
        dims = Dimensions(0, np.full(T + 1, n, np.int32), np.full(T, m, np.int32), term(c),
                          term(g), np.full(T, c, np.int32), np.full(T, g, np.int32))
    else:
        tile = lambda pat, count: np.array([pat[i % len(pat)] for i in range(count)], np.int32)
        dims = Dimensions(0, tile(wl["state"], T + 1), tile(wl["control"], T),
                          tile(wl["node_c"], T + 1), tile(wl["node_g"], T + 1),
                          tile(wl["edge_c"], T), tile(wl["edge_g"], T))
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    sampler = ClockSampler(0)
    cp = CallbackProvider(dims, Topology.chain(T), batch, device=0,
                          force_generic=getattr(args, "force_generic", False),
                          pad_variable_dims=getattr(args, "pad_variable_dims", False))
    eng = cp.engine
    # The reference benchmark's full regularization range (newton_kkt_benchmark.cpp:231-233) on
    # both workloads: the rollout of the shape-specialised kernels applies (I + D V)^-1 in the
    # reference's F-solve form, so the default path holds 1e-9 against the oracle up to
    # r2 = 1e9 (tests/test_gpu_kkt.py::test_newton_kkt_benchmark_shapes).
    r2_max = 1e9
    model_h, w_h, r1_h, r2_h, r3_h, b_h = kkt_host_problem(dims, batch, args.seed, r2_max)
    model = cp.pack_model(model_h)
    w, r1, r2, r3, b = (eng.pack(a) for a in (w_h, r1_h, r2_h, r3_h, b_h))
    sol = eng.zeros(b_h.shape[1])
    ok = eng.empty_int()
    stream = torch.cuda.current_stream(dev)

    captured = None
    if getattr(args, "graph", False):
        # the step recorded once as a CUDA graph, replayed with one driver call per step
        captured = cp.capture_step(model, w, r1, r2, r3, b, sol, ok=ok)

    def step():
        if captured is not None:
            return captured.replay()
        cp.factor(model, w, r1, r2, r3, ok=ok, stream=stream)
        cp.solve(model, b, sol, stream=stream)
        return cp.residual(model, w, r1, r2, r3, sol, b, ok=ok, stream=stream)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize(dev)
    launches0 = eng.launch_count
    if captured is None:
        lib.sipoc_profile_enable(eng._handle, 1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        norms, stats = step()
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    t1 = time.time()
    ms_per_step = ev0.elapsed_time(ev1) / args.steps
    gpu_launches = eng.launch_count - launches0
    kernels = {}
    if captured is not None:
        # no per-kernel events inside a graph: the step's device time is attributed as a whole
        # (sipoc_graph_launch adds the recorded kernels to the launch count)
        kernels["captured_step"] = {"ms_per_launch": ms_per_step, "ms_per_step": ms_per_step}
    for i in range(0 if captured is not None else lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                              ctypes.byref(cnt))
        kernels[nm.value.decode()] = {"ms_per_launch": ms.value / max(cnt.value, 1),
                                      "ms_per_step": ms.value / args.steps}
    lib.sipoc_profile_enable(eng._handle, 0)
    sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch,
                     {"sol": sol[:b_h.shape[1]], "ok": ok, "residual_norm": norms},
                     {"stats": stats})
    st = stats.cpu().numpy()
    # relative residual: ||K sol - b|| / ||b|| (r2 up to 1e9 scales the rows)
    rel = (norms[:batch].cpu().numpy() / np.linalg.norm(b_h, axis=1)).max()
    in_elems = sum(v.shape[1] for v in model_h.values()) + w_h.shape[1] + r1_h.shape[1] \
        + r2_h.shape[1] + r3_h.shape[1] + b_h.shape[1]
    alg_bytes = 8 * (in_elems + b_h.shape[1])
    peak, peak_kind = measured_peaks()
    hot_ms = sum(v["ms_per_step"] for v in kernels.values())
    achieved = alg_bytes * batch / (hot_ms * 1e-3) / 1e9
    dominant = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
    line = {
        "metric": "batched Newton-KKT factor+solve+residual solves/sec (FP64)",
        "value": batch / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "r2_max": r2_max, **{k: (list(v) if isinstance(v, tuple) else v)
                                                for k, v in wl.items()},
                   "kkt_dim": int(b_h.shape[1]), "kernel_variant": eng.kernel_variant,
                   "launch": "cuda_graph" if captured is not None else "eager",
                   "generator": "newton_kkt_benchmark.cpp:171-240 distribution"},
        "clocks": sampler.summary(t0, t1), "e2e": None, "gpu_launches": int(gpu_launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_kind, "traffic": None,
                     "algorithmic_bytes_per_solve": alg_bytes, "dominant_kernel": dominant,
                     "kernels": kernels},
        "check": {"failed_problems": float(st[2]), "problems": float(st[3]),
                  "max_relative_kkt_residual": float(rel)},
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS) + ["newton_kkt", "newton_kkt_uniform"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--horizon", type=int, default=0, help="override the horizon T")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default, BASELINE's config): the workload's batch is sharded over "
                         "the GPUs; weak: every GPU gets the workload's batch")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--force-generic", action="store_true")
    ap.add_argument("--input-layout", default="interleaved", choices=["interleaved", "problem_major"],
                    help="device layout of the inputs the timed call takes (LQR workloads)")
    ap.add_argument("--pad-variable-dims", action="store_true",
                    help="newton_kkt: SIPOC_FLAG_PAD_VARIABLE_DIMS (shape-specialised kernels through "
                         "decoupled padding instead of the strict-order generic kernels)")
    ap.add_argument("--graph", action="store_true",
                    help="newton_kkt workloads: replay the step as one CUDA graph "
                         "(CallbackProvider.capture_step) instead of launching its kernels eagerly")
    ap.add_argument("--fp32", action="store_true",
                    help="the optional FP32 mode (sipoc_lqr_factor_solve_f32; workload cartpole): "
                         "a separate line with dtype f32, tolerance 5e-4 against the FP64 oracle")
    ap.add_argument("--serial-in-time", action="store_true",
                    help="long-horizon workloads: forbid the parallel-in-time scan "
                         "(SIPOC_FLAG_SERIAL_IN_TIME), i.e. time the serial sweep + rollout")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-batch", type=int, default=0,
                    help="problems per host-buffer call per GPU (0 = the GPU's whole shard)")
    ap.add_argument("--e2e-packed", action="store_true",
                    help="also time sipoc_lqr_factor_solve_host_packed (e2e.packed: Q / R as packed "
                         "lower triangles, M not sent)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the timed call returned in its "
                         "last step as DIR/<name>.npy (float32 / float64, under 64 MB in all: a "
                         "fixed sample of the problems when the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload in ("newton_kkt", "newton_kkt_uniform"):
        return run_kkt(args)
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
    if args.horizon:
        wl["T"] = args.horizon
    if args.impl == "reference":
        return run_reference(args, wl, args.workload)
    return run_ours(args, wl, args.workload)


if __name__ == "__main__":
    sys.exit(main())
