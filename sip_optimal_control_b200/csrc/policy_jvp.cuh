// Forward-mode derivative of the feedback policy of the LQR solve (sipoc_lqr_policy_jvp): the
// tangent of the Riccati recursion that produces K, k, V, v (policy.cuh), one sweep from the
// leaves to the root (post-order), the direction of the factorization itself.  Per edge e with
// parent p and child c:
//   primal (recomputed from the inputs and the forward's V_c, v_c as policy_vjp.cuh does):
//     P = (I + D^1/2 V_c D^1/2)^-1   W = D^-1/2 (I - P) D^-1/2   S = D^1/2 P D^-1/2 = (I + D V_c)^-1
//     G = R + B' W B   Y = W A   H = M' + B' Y   K = -G^-1 H                  (D = diag delta_c)
//     f = delta_c .* v_c - c_c   g = v_c - W f   h = r + B' g   k = -G^-1 h
//   tangent, with dV_c, dv_c of the child complete (sym(dQ_c), dq_c plus what c's own child
//   edges added):
//     dW = S' dV_c S - W dD W                                  (dD = diag ddelta_c)
//     dG = sym(dR) + dB' W B + B' W dB + B' dW B
//     dY = dW A + W dA   dH = dM' + dB' Y + B' dY   dK = -G^-1 (dH + dG K)
//     df = ddelta_c .* v_c + delta_c .* dv_c - dc_c
//     dg = dv_c - dW f - W df   dh = dr + dB' g + B' dg   dk = -G^-1 (dh + dG k)
//     dV_p += dA' Y + Y' dA + A' dW A + dH' K + K' dH + K' dG K  (one triangle, mirrored)
//     dv_p += dA' g + A' dg + dK' h + K' dh
// Every node starts from dV_i = sym(dQ_i), dv_i = dq_i.  Each convention is the transpose of
// one of sipoc_lqr_policy_vjp, so <cot, JVP(t)> = <t, VJP(cot)> holds for every tangent: dQ
// and dR enter through their symmetric parts, and the root's dc and ddelta are not read.
// Tangents of q, r, c alone give dK = 0 and dV = 0 exactly.
//
// Kernels (policy_jvp.cu):
// - policy_jvp_subwarp<N, M>: uniform chains at the shapes of the thread and four-lane plans.
//   A sub-warp of lanes per problem, several problems per warp; each edge's operands are
//   staged global -> shared for the warp's problems with cp.async, every matrix of the edge
//   lives in shared memory, and a lane owns a cyclic set of the elements (or columns, for the
//   triangular solves) of each result.  dV, dv of the current node stay on chip.
// - policy_jvp_generic_kernel: every other structure, one thread per problem with runtime dims
//   on an engine-layout workspace.  A parent sums its child edges in child_offsets order.
// Lanes b >= batch and problems whose forward status != 0 get zeros in every requested output.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "generic_kernels.cuh"
#include "policy.cuh"
#include "policy_vjp.cuh"
#include "structure.hpp"

namespace sipoc {

// Element count of the per-problem workspace of the generic kernel: the edge scratch for
// state dims <= nx and controls <= mx, then dV, dv of every node (nn_off[N] + n_off[N]).
int64_t policy_jvp_generic_ws_elems(const HostStructure &h);

// Whether launch_policy_jvp_subwarp has an instance for (n, m).
bool policy_jvp_subwarp_shape(int n, int m);

// Uniform chain of E edges with (n, m) in {4, 6, 8} x {1..4} or (12, 4).  in: the forward's
// inputs (R, M, r, A, B, c, delta) and V (lower), v.  tan: any array may be nullptr (zeros,
// not read).  out: any array may be nullptr (not written).  Returns false when (n, m) has no
// instance or the launch could not be configured.
bool launch_policy_jvp_subwarp(int n, int m, int E, const PolicyVjpIn &in, const LqrIn &tan,
                               const LqrPolicy &out, const int *status, int64_t batch,
                               int64_t ld, cudaStream_t stream);

// Any tree and any dims; ws: policy_jvp_generic_ws_elems(h) elements per problem.
void launch_policy_jvp_generic(const DevTables &t, const HostStructure &h, const PolicyVjpIn &in,
                               const LqrIn &tan, const LqrPolicy &out, double *ws,
                               const int *status, int64_t batch, int64_t ld, cudaStream_t stream);

}  // namespace sipoc
