import os, sys, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import problem_gen as pg
from gpu_helpers import *
from test_gpu_kkt import _gpu_kkt, rel_err
import test_gpu_kkt as t
from oracle import pyoracle
from oracle.pyoracle import Structure
reps = 6
sd = [2, 1, 3] * reps + [2]; T = len(sd) - 1
cd = ([1, 2, 1] * reps)[:T]
node_c = ([1, 0, 2] * reps + [1])[:T + 1]; node_g = ([0, 2, 1] * reps + [0])[:T + 1]
edge_c = ([1, 2, 0] * reps)[:T]; edge_g = ([2, 1, 1] * reps)[:T]
s = Structure.chain(T, sd, cd, node_c=node_c, node_g=node_g, edge_c=edge_c, edge_g=edge_g)
for r2max in (1e3, 1e6, 1e9):  # default = reference-order strict plan; flag = reordered padded plan
    model, w, r1, r2, r3, rhs = pg.newton_kkt_batch(s, 200, seed=9, r2_max=r2max)
    ref = pyoracle.kkt_factor_solve(s, model, w, r1, r2, r3, rhs)
    good = ref["ok"] == 1
    for pad, gen in ((False, True), (False, False), (True, False)):
        gpu, cp, _ = _gpu_kkt(s, model, w, r1, r2, r3, rhs, pad_variable_dims=pad, force_generic=gen)
        scale = np.linalg.norm(rhs, axis=1)
        print(r2max, cp.engine.kernel_variant, 'rel_err max', rel_err(gpu["sol"][good], ref["sol"][good]).max(),
              'rel residual max', (gpu["residual"][good] / scale[good]).max(), 'ok match', (gpu["ok"] == ref["ok"]).all())
