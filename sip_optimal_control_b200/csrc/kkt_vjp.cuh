// Reverse-mode derivative (vector-Jacobian product) of the batched Newton-KKT solve.
//
// The solve is sol = K^-1 b with K = [H + diag(r1), C', G'; C, -diag(r2), 0;
// G, 0, -diag(w + r3)] symmetric, so for a cotangent g = dL/dsol the adjoint lam = K^-1 g is
// one more solve of the same system with b := g, and dL = lam' db - lam' dK sol.  A model
// block B at K[R, C] (and B' at K[C, R]) gets
//   dB = -(lam_R s_C' + s_R lam_C')                off-diagonal blocks
//   dB = -(lam_R s_R' + s_R lam_R') / 2            symmetric Hessian blocks (R == C)
// and the vectors db = lam, dr1 = -lam_x .* s_x, dr2 = lam_y .* s_y, dw = dr3 = lam_z .* s_z
// (DESIGN.md, "Differentiating the Newton-KKT solve"; include/sipoc.h, sipoc_kkt_vjp).
#pragma once

#include <cuda_runtime.h>

#include "generic_kernels.cuh"
#include "kkt_theta.cuh"
#include "structure.hpp"

namespace sipoc {

// Gradient arrays in the layout of the arrays they belong to; any may be nullptr (neither
// computed nor written).  w and r3 share one formula and may be the same array.
struct KktGrad {
  double *node_hxx, *node_jc, *node_jg;
  double *edge_hxx, *edge_hxu, *edge_huu, *edge_A, *edge_B;
  double *edge_jcx, *edge_jcu, *edge_jgx, *edge_jgu;
  double *node_hxt, *node_jct, *node_jgt, *node_htt;
  double *edge_hxt, *edge_hut, *edge_dynt, *edge_jct, *edge_jgt, *edge_htt;
  double *b, *w, *r1, *r2, *r3;
};

// One launch.  Any tree, any dims, theta included: it works on the structure's own
// (unpadded) arrays.  sol and lam are full [x | y | z] vectors.  Every lane b < ld of every
// requested array is written; lanes b >= batch and problems with ok[b] == 0 get zeros.
// ok: int[batch], not nullptr.
void launch_kkt_vjp(const DevTables &t, const double *sol, const double *lam, const int *ok,
                    const KktGrad &grad, int64_t batch, int64_t ld, cudaStream_t stream);

}  // namespace sipoc
