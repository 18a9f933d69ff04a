// Reverse-mode derivative (vector-Jacobian product) of the batched LQR solve.
//
// The solve is K z = -h with z = (x, u, y), h = (q, r, c) and K symmetric, so for a
// cotangent g = dL/dz the adjoint mu = -K^-1 g is one more solve of the same LQR with
// (q, r, c) := g, and dL = mu^T (dK z + dh).  This kernel turns (z, mu) into the gradients
// of every input array (DESIGN.md, "Differentiating the LQR solve"):
//   q, r, c   mu_x, mu_u, mu_y              delta_i   -mu_y_i * y_i
//   Q_i       (mu_x_i x_i' + x_i mu_x_i') / 2     R_e   (mu_u_e u_e' + u_e mu_u_e') / 2
//   M_e       mu_x_p u_e' + x_p mu_u_e'            A_e   y_c mu_x_p' + mu_y_c x_p'
//   B_e       y_c mu_u_e' + mu_y_c u_e'            (p, c: the parent / child node of edge e)
#pragma once

#include <cuda_runtime.h>

#include "generic_kernels.cuh"
#include "structure.hpp"

namespace sipoc {

// Gradient arrays in the layout of the input arrays they belong to; any may be nullptr
// (neither computed nor written).
struct LqrGrad {
  double *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
};

// One launch.  Any tree and any dims: it works on the structure's own (unpadded) arrays.
// Every lane b < ld of every requested array is written; lanes b >= batch and problems with
// status[b] != 0 get zeros.  status: int[batch], not nullptr.
void launch_lqr_vjp(const DevTables &t, const LqrOut &sol, const LqrOut &adjoint,
                    const int *status, const LqrGrad &grad, int64_t batch, int64_t ld,
                    cudaStream_t stream);

}  // namespace sipoc
