// Reverse-mode derivative of the feedback policy of the LQR solve (sipoc_lqr_policy_vjp):
// the adjoint of the Riccati recursion that produces K, k, V, v (policy.cuh), one sweep from
// the root to the leaves (pre-order), per edge e with parent p and child c:
//   forward (recomputed from the inputs and the forward's V_c, v_c; nothing is kept):
//     P_c = (I + D^1/2 V_c D^1/2)^-1   W_c = D^-1/2 (I - P_c) D^-1/2   (D = diag(delta_c))
//     G = R + B' W_c B   Y = W_c A   H = M' + B' Y   K = -G^-1 H
//     f = delta_c .* v_c - c_c   g = v_c - W_c f   h = r + B' g   k = -G^-1 h
//   adjoint, with Vb_p, vb_p the cotangents of V_p, v_p (the caller's, symmetrised, plus what
//   p's parent edge sent down), Qb_p = Vb_p and qb_p = vb_p:
//     Kb = cot K + h vb_p'   kb = cot k
//     hb = K vb_p - G^-1 kb   Hb = 2 K Vb_p - G^-1 Kb
//     Gb = sym(K Vb_p K' - G^-1 Kb K' - G^-1 kb k')
//     gb = A vb_p + B hb   Yb = B Hb   fb = -W_c gb
//     rb = hb   Mb = Hb'   Rb = Gb
//     Ab = g vb_p' + 2 Y Vb_p + W_c Yb      Bb = g hb' + Y Hb' + 2 W_c B Gb
//     Wb = sym(A Vb_p A' + Yb A' + B Gb B' - gb f')
//     cb_c = -fb   deltab_c = fb .* v_c - diag(W_c Wb W_c)
//     sent down to c: Vb_c += S Wb S' (S = (I + D V_c)^-1 = D^1/2 P_c D^-1/2),
//                     vb_c += gb + delta_c .* fb
// The root's c and delta get zero gradient.  Q and R get the gradient with respect to the
// symmetric matrix (the same values in both triangles), as in sipoc_lqr_vjp.
//
// Mapping: one thread per problem on the engine layout X[flat * ld + b].  Lanes b >= batch and
// problems whose forward status != 0 get zeros in every requested gradient.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "generic_kernels.cuh"
#include "lqr_vjp.cuh"
#include "structure.hpp"

namespace sipoc {

// Cotangents of the policy, in the engine layout of M, r, Q, q; any may be nullptr (zeros).
struct LqrPolicyCot {
  const double *K, *k, *V, *v;
};

// The forward's policy arrays the sweep reads (V through its lower triangle), and the inputs.
struct PolicyVjpIn {
  LqrIn in;  // R, M, r, A, B, c, delta are read; Q, q are not
  const double *V, *v;
};

// Element counts of the per-problem scratch of one edge for state dims <= nx, controls <= mx.
int64_t policy_vjp_scratch_elems(int nx, int mx);

// Whether launch_policy_vjp_chain has an instance for (n, m).
bool policy_vjp_chain_shape(int n, int m);

// Uniform chain of E edges with (n, m) in the shapes of the thread-per-problem and four-lane
// plans ({4, 6, 8} x {1..4} and (12, 4)): scratch in each thread's local memory.  Returns
// false when (n, m) has no instance.
bool launch_policy_vjp_chain(int n, int m, int E, const PolicyVjpIn &in, const LqrPolicyCot &cot,
                             const LqrGrad &grad, const int *status, int64_t batch, int64_t ld,
                             cudaStream_t stream);

// Any tree and any dims.  ws: engine-layout workspace of
// policy_vjp_scratch_elems(max_n, max_m) + nn_off[N] + n_off[N] elements per problem (the
// edge scratch, then Vb and vb of every node).
void launch_policy_vjp_generic(const DevTables &t, const HostStructure &h, const PolicyVjpIn &in,
                               const LqrPolicyCot &cot, const LqrGrad &grad, double *ws,
                               const int *status, int64_t batch, int64_t ld, cudaStream_t stream);

}  // namespace sipoc
