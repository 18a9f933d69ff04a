// Forward-mode derivatives (Jacobian-vector products) of the batched LQR and Newton-KKT solves.
//
// LQR: the solve is K z = -h with z = (x, u, y), h = (q, r, c), so for tangents (dK, dh) of
// the inputs dz = -K^-1 (dK z + dh): the same LQR solved with (q, r, c) := t = dK z + dh,
//   t_x_i = dQ_i x_i + dq_i + sum_{e: parent(e) = i} (dM_e u_e + dA_e' y_c(e))
//   t_u_e = dR_e u_e + dr_e + dM_e' x_p + dB_e' y_c
//   t_y_c = dA_e x_p + dB_e u_e - ddelta_c .* y_c + dc_c     (root: -ddelta_r .* y_r + dc_r)
// KKT: sol = K^-1 b, so d sol = K^-1 (db - dK sol): the same KKT solve with b := t = db - dK sol,
// dK holding the tangent model blocks where kkt_blocks.cuh places them, diag(dr1) on the x
// rows, -diag(dr2) on the y rows and -diag(dw + dr3) on the z rows.
// Symmetric blocks (Q, R, the Hessian blocks) enter through their symmetric part
// (dB + dB') / 2, the transpose of the VJPs' symmetric-gradient convention
// (DESIGN.md, "Forward-mode derivatives").
#pragma once

#include <cuda_runtime.h>

#include "generic_kernels.cuh"
#include "kkt_theta.cuh"
#include "structure.hpp"

namespace sipoc {

// Tangents of the nine LQR inputs; any may be nullptr (a zero tangent, not read).
struct LqrTangent {
  const double *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
};

// Tangents of the Newton-KKT inputs, named after the blocks; any may be nullptr.
struct KktTangent {
  const double *node_hxx, *node_jc, *node_jg;
  const double *edge_hxx, *edge_hxu, *edge_huu, *edge_A, *edge_B;
  const double *edge_jcx, *edge_jcu, *edge_jgx, *edge_jgu;
  const double *node_hxt, *node_jct, *node_jgt, *node_htt;
  const double *edge_hxt, *edge_hut, *edge_dynt, *edge_jct, *edge_jgt, *edge_htt;
  const double *b, *w, *r1, *r2, *r3;
};

// One launch each.  Any tree and any dims (theta included): they work on the structure's own
// (unpadded) arrays.  Every lane b < ld of the right-hand side is written: t by the formula
// for b < batch, zeros in the padding lanes.  sol: the forward's solution (LQR: x, u, y;
// KKT: the full [x | y | z] vector); rhs: LQR (q, r, c)-shaped arrays, KKT an [x | y | z]
// vector.
void launch_lqr_jvp(const DevTables &t, const LqrOut &sol, const LqrTangent &tan,
                    const LqrOut &rhs, int64_t batch, int64_t ld, cudaStream_t stream);
void launch_kkt_jvp(const DevTables &t, const double *sol, const KktTangent &tan, double *rhs,
                    int64_t batch, int64_t ld, cudaStream_t stream);

// a[r * ld + b] = 0 for every row r < rows of the lanes b < ld that are padding (b >= batch)
// or whose flag marks a failed problem: flag[b] != 0 for an LQR status, flag[b] == 0 for a
// KKT ok.
void launch_zero_dead_lanes(double *a, int64_t rows, const int *flag, bool flag_is_ok,
                            int64_t batch, int64_t ld, cudaStream_t stream);

}  // namespace sipoc
