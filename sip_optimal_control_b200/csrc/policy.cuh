// Export of the feedback policy an LQR solve computes (sipoc_lqr_factor_solve_policy):
//   u_e = K_e x_parent(e) + k_e   per edge,      y_i = V_i x_i + v_i   per node,
// the reference's K, k, V, v after factor_with_status + solve (lqr.cpp:658, :707-719,
// :744, :785-794).  Every plan keeps K, k and v of every block; the reference-order plans
// (generic, strict) keep V too, the others keep P = F^-1 instead and V is rebuilt per edge.
//
// Mapping, as lqr_vjp_kernel: threads go across problems (engine layout X[flat * ld + b]),
// each grid row (blockIdx.y, grid-stride) owns one node or edge.  Every lane b < ld of a
// requested array is written; lanes b >= batch and problems with status[b] != 0 get zeros.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "generic_kernels.cuh"
#include "structure.hpp"

namespace sipoc {

struct LqrPolicy {
  double *K, *k, *V, *v;  // each in the engine layout of M, r, Q, q; any may be nullptr
};

// Where a plan keeps one array of blocks.  Block j (edge for K / k, node for V / v, P) starts
// at flat element off + j * block of the problem's store; entry (r, c) of a matrix block sits
// at r + c * rows (the plan's possibly padded leading dimension).
//   element-major (pm_stride == 0): src[flat * ld + b];  problem-major: src[b * pm_stride + flat]
//   segments (seg_len > 0, parallel in time): block j lives in segment s = min(j / seg_len,
//     segs - 1) at local index j - s seg_len, and segment s's region starts at s * seg_stride.
//     So node s seg_len comes from segment s, the last node from the last segment.
//   same_as_out: the source uses the output's own offsets (the generic workspace).
struct PolicySrc {
  const double *p = nullptr;
  int64_t pm_stride = 0;
  int64_t off = 0, block = 0;
  int rows = 1;
  int seg_len = 0, segs = 1;
  int64_t seg_stride = 0;
  bool same_as_out = false;
};

enum class PolicyArray { K, k, V, v };

// Blocks of `which` -> dst (the structure's own unpadded layout).  One launch.
void launch_policy_gather(const DevTables &t, PolicyArray which, const PolicySrc &src,
                          double *dst, const int *status, int64_t batch, int64_t ld,
                          cudaStream_t stream);

// V of every node of a uniform chain of E edges with n states and m controls, rebuilt from
// the inputs and the plan's kept P = F^-1 (node blocks of tri(n), packed lower) and K (edge
// blocks of n m):  W_c = D_c^-1/2 (I - P_c) D_c^-1/2,  H = M' + B' W_c A,
// V_p = Q_p + A' W_c A + K' H;  V_E = Q_E.  Q is read through its lower triangle and both
// triangles of V are written from the lower one.  `in` holds Q, M, A, B, delta in the
// engine layout of the (n, m) chain; V gets node i at flat i n n.  For segments, P and K of
// edge e are read from the edge's own segment.  Returns false when (n, m) has no instance.
bool launch_policy_rebuild_v(int n, int m, const LqrIn &in, const PolicySrc &P,
                             const PolicySrc &K, double *V, const int *status, int E,
                             int64_t batch, int64_t ld, cudaStream_t stream);

// Where the shape-specialised plans keep K, k, v, P (or V), for (n, m) and T edges.
enum class PolicyStore { FAST, CTA, STRICT };
struct PolicySources {
  PolicySrc K, k, v, V_or_P;  // V_or_P: V for STRICT, P = F^-1 otherwise
};
PolicySources policy_sources(PolicyStore kind, int n, int m, int T, const double *store,
                             const double *scratch);

}  // namespace sipoc
