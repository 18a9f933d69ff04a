"""Timing of the reference's VariableLQRProblem benchmark shapes (lqr_benchmark.cpp:209-310: heterogeneous
chain, star, binary tree) on the reference-order padded plans against the generic kernels."""
import os, sys, time, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import problem_gen as pg
from gpu_helpers import *
from oracle import pyoracle
for shape, base_n, T in (("chain", 4, 63), ("chain", 5, 63), ("star", 4, 63), ("binary", 4, 63)):
    sd = [max(1, base_n + (i % 3) - 1) for i in range(T + 1)]
    cd = [max(1, 2 + (e % 3) - 1) for e in range(T)]
    children = list(range(1, T + 1))
    parents = {"chain": list(range(T)), "star": [0] * T, "binary": [(c - 1) // 2 for c in children]}[shape]
    s = pyoracle.Structure(parents, children, 0, sd, cd)
    batch = 8192
    host = pg.variable_tree_batch(s, 64, seed=1)
    host = {k: np.tile(v, (batch // 64, 1)) for k, v in host.items()}
    dims, topo = to_structs(s)
    for gen in (True, False):
        lqr = LQR(dims, topo, batch, force_generic=gen)
        inp, out = lqr.pack_input(host), lqr.alloc_output()
        for _ in range(3): lqr.factor_solve(inp, out)
        torch.cuda.synchronize(); t0 = time.time()
        for _ in range(10): lqr.factor_solve(inp, out)
        torch.cuda.synchronize(); dt = (time.time() - t0) / 10
        print(shape, max(sd), max(cd), lqr.engine.kernel_variant, f"{dt*1e3:.3f} ms", f"{batch/dt/1e6:.2f} M solves/s")
