"""Timing of the Newton-KKT VJP (sipoc_kkt_vjp) on the GPU.

Per workload (inputs from bench.py's kkt_host_problem, r2 up to 1e9; cotangents N(0, 1)), with
CUDA events after a warm-up:
- the forward factor + solve;
- sipoc_kkt_vjp with every gradient, and with b alone;
- the gradient kernel alone (kkt_vjp_kernel, sipoc_profile_*), with its bytes computed from
  the sizes -- the requested gradients written (every lane of batch_stride), the sol and lam
  entries they need read, and ok -- its bandwidth and share of 7.7 TB/s (the HGX B200
  data-sheet HBM3e rate of one GPU).
A seeded sample of problems is checked against the CPU reference VJP.  The device name, power
limit and max SM clock are read in the same run.  Usage:
    python tools/bench_kkt_vjp.py --out profiles/r04/bench_kkt_vjp.json [--workloads ...]
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

from bench import KKT_UNIFORM, KKT_WORKLOAD, kkt_host_problem  # noqa: E402
from bench_vjp import PEAK_TBS, device_info, event_ms  # noqa: E402
from gpu_helpers import rel_err  # noqa: E402
from kkt_vjp_reference import MODEL_NAMES, VECTOR_NAMES, kkt_solve, kkt_vjp  # noqa: E402
from oracle.pyoracle import Structure  # noqa: E402
from sip_optimal_control_b200 import CallbackProvider, Dimensions, Topology, _capi  # noqa: E402
from sip_optimal_control_b200._capi import lib  # noqa: E402

GRAD_NAMES = MODEL_NAMES + VECTOR_NAMES
REG = ("w", "r1", "r2", "r3")
WORKLOADS = {  # name: (bench.py workload, batch)
    "newton_kkt_uniform": ("uniform", 8192),
    "newton_kkt_uniform_fused": ("uniform", 32768),  # the fused solve (batch >= 32 768)
    "newton_kkt_config4": ("config4", 8192),
}


def dimensions(kind: str):
    if kind == "uniform":
        T, n, m = KKT_UNIFORM["T"], KKT_UNIFORM["n"], KKT_UNIFORM["m"]
        c, g = max(1, n // 2), max(1, 2 * m)
        term = lambda v: np.array([0] * T + [v], np.int32)
        return T, Dimensions(0, np.full(T + 1, n, np.int32), np.full(T, m, np.int32), term(c),
                             term(g), np.full(T, c, np.int32), np.full(T, g, np.int32))
    wl = KKT_WORKLOAD
    T = wl["T"]
    tile = lambda pat, count: np.array([pat[i % len(pat)] for i in range(count)], np.int32)
    return T, Dimensions(0, tile(wl["state"], T + 1), tile(wl["control"], T),
                         tile(wl["node_c"], T + 1), tile(wl["node_g"], T + 1),
                         tile(wl["edge_c"], T), tile(wl["edge_g"], T))


def profiled_kernel_ms(eng, fn, iters: int) -> float:
    lib.sipoc_profile_enable(eng._handle, 1)
    for _ in range(iters):
        fn()
    total, count = 0.0, 0
    for i in range(lib.sipoc_profile_collect(eng._handle)):
        nm, ms, cnt = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_int64()
        eng._check(lib.sipoc_profile_get(eng._handle, i, ctypes.byref(nm), ctypes.byref(ms),
                                         ctypes.byref(cnt)))
        if nm.value.decode() == "kkt_vjp_kernel":
            total, count = ms.value, cnt.value
    lib.sipoc_profile_enable(eng._handle, 0)
    assert count == iters, count
    return total / count


def kernel_bytes(size: dict, want, batch: int, ld: int) -> int:
    # b alone is lam alone; every other gradient reads both sol and lam
    vectors = 1 if set(want) == {"b"} else 2
    return 8 * ld * sum(size[k] for k in want) + 8 * batch * vectors * size["b"] + 4 * batch


def run(name, kind, batch, warmup, iters, sample, seed):
    T, dims = dimensions(kind)
    cp = CallbackProvider(dims, Topology.chain(T), batch, device=0)
    e = cp.engine
    z = cp.sizes
    size = {k: z[k] for k in MODEL_NAMES}
    size.update(b=z["kkt_dim"], w=z["z_dim"], r1=z["x_dim"], r2=z["y_dim"], r3=z["z_dim"])
    model_h, w_h, r1_h, r2_h, r3_h, b_h = kkt_host_problem(dims, batch, seed, 1e9)
    reg_h = dict(w=w_h, r1=r1_h, r2=r2_h, r3=r3_h)
    model = cp.pack_model(model_h)
    reg = {k: e.pack(v) for k, v in reg_h.items()}
    b = e.pack(b_h)
    del b_h
    sol, adj = e.zeros(z["kkt_dim"]), e.empty(z["kkt_dim"])
    ok, vjp_ok = e.empty_int(), e.empty_int()
    gen = torch.Generator(device=e.torch_device()).manual_seed(7)
    cot = torch.randn(sol.shape, generator=gen, dtype=torch.float64, device=e.torch_device())
    grads = {k: e.empty(size[k]) for k in GRAD_NAMES}
    stream = e.stream_ptr()
    from sip_optimal_control_b200.kkt import _model_struct

    keep = []
    sm = _model_struct(model, False, keep)

    def vjp_call(want):
        sg = _capi.KktGrad()
        for k in GRAD_NAMES:
            setattr(sg, k, grads[k].data_ptr() if k in want else None)
        keep.append(sg)
        return lambda: e._check(lib.sipoc_kkt_vjp(
            e._handle, ctypes.byref(sm), *(reg[k].data_ptr() for k in REG), sol.data_ptr(),
            cot.data_ptr(), adj.data_ptr(), ctypes.byref(sg), vjp_ok.data_ptr(), stream))

    def forward():
        cp.factor(model, *(reg[k] for k in REG), ok=ok)
        cp.solve(model, b, sol)

    forward()
    vjp_all, vjp_b = vjp_call(GRAD_NAMES), vjp_call(("b",))
    line = dict(workload=name, T=T, batch=batch, batch_stride=e.batch_stride,
                kernel_variant=e.kernel_variant, iters=iters,
                model_bytes=8 * e.batch_stride * sum(size[k] for k in MODEL_NAMES))
    line["forward_ms"] = event_ms(forward, warmup, iters)
    line["vjp_all_ms"] = event_ms(vjp_all, warmup, iters)
    line["vjp_b_ms"] = event_ms(vjp_b, warmup, iters)
    for tag, fn, want in (("all", vjp_all, GRAD_NAMES), ("b", vjp_b, ("b",))):
        ms = profiled_kernel_ms(e, fn, iters)
        nbytes = kernel_bytes(size, want, batch, e.batch_stride)
        tbs = nbytes / (ms * 1e-3) / 1e12
        line[f"kernel_{tag}"] = dict(ms=ms, bytes=nbytes, tb_per_s=tbs,
                                     share_of_7_7_tb_per_s=tbs / PEAK_TBS)
    # seeded sample against the CPU reference, from the last (all-gradient) call
    forward()
    vjp_all()
    torch.cuda.synchronize()
    idx_h = np.sort(np.random.default_rng(11).choice(batch, min(sample, batch), replace=False))
    idx = torch.from_numpy(idx_h).to(e.torch_device())
    pick = lambda t, n: t[:n].index_select(1, idx).T.contiguous().cpu().numpy()
    s = Structure.chain(T, dims.state_dims, dims.control_dims, node_c=dims.node_c_dims,
                        node_g=dims.node_g_dims, edge_c=dims.edge_c_dims,
                        edge_g=dims.edge_g_dims)
    hm = {k: v[idx_h] for k, v in model_h.items()}
    hr = {k: v[idx_h] for k, v in reg_h.items()}
    hb = pick(b, size["b"])
    ref_sol = kkt_solve(s, 0, hm, None, *(hr[k] for k in REG), hb)
    ref = kkt_vjp(s, 0, hm, None, *(hr[k] for k in REG), ref_sol["sol"], pick(cot, size["b"]))
    good = ref["ok"] == 1
    line["sample_problems"] = int(idx.numel())
    line["sample_ok"] = int(good.sum())
    assert (vjp_ok[:batch].index_select(0, idx).cpu().numpy() == ref["ok"]).all()
    line["sample_max_rel_err"] = {k: float(rel_err(pick(grads[k], size[k])[good],
                                                   ref[k][good]).max()) for k in GRAD_NAMES}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sample", type=int, default=16)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_kkt_vjp.py needs a CUDA device")
    torch.cuda.set_device(0)
    result = dict(tool="tools/bench_kkt_vjp.py", **device_info(), peak_tb_per_s=PEAK_TBS,
                  runs=[])
    for name in args.workloads.split(","):
        kind, batch = WORKLOADS[name]
        line = run(name, kind, batch, args.warmup, args.iters, args.sample, args.seed)
        print(json.dumps(line), flush=True)
        result["runs"].append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
