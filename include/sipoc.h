/*
 * sipoc.h — C ABI of the B200-native batched regularized-LQR / Newton-KKT engine.
 *
 * Drop-in boundary for the Newton-KKT linear-solve path of
 * joaospinto/sip_optimal_control.  One engine handle owns ONE problem
 * structure (Topology + Dimensions, reference lqr.hpp:5-64) and a batch of B
 * numerically independent problems of that structure, all resident on one
 * CUDA device.  Every entry point is extern "C" with plain pointers and
 * sizes; nothing here depends on PyTorch, Eigen or sip.
 *
 * Reference interfaces each group of entry points replaces (file:line are
 * relative to the reference repository):
 *
 *   sipoc_create / sipoc_destroy      LQR::LQR + LQR::compile_topology
 *                                     (lqr.hpp:189-191, lqr.cpp:563-643) and
 *                                     CallbackProvider::CallbackProvider +
 *                                     validate_input (helpers.cpp:11-26,
 *                                     types.cpp:68-134)
 *   sipoc_lqr_factor                  LQR::factor_with_status / LQR::factor
 *                                     (lqr.hpp:192-193, lqr.cpp:645-733)
 *   sipoc_lqr_solve                   LQR::solve (lqr.hpp:194, lqr.cpp:735-871)
 *   sipoc_lqr_factor_solve            factor_with_status + solve back to back,
 *                                     the loop body of BM_LQRFactorSolve
 *                                     (benchmarks/lqr_benchmark.cpp:653-663)
 *   sipoc_lqr_residual                compute_residual_norm
 *                                     (tests/lqr_test.cpp:152-186, :371-409)
 *   sipoc_kkt_apply_block             CallbackProvider::add_Hx_to_y / add_Cx_to_y /
 *                                     add_CTx_to_y / add_Gx_to_y / add_GTx_to_y
 *                                     (helpers.hpp:17-21, helpers.cpp:979-1368)
 *   sipoc_kkt_factor                  CallbackProvider::factor
 *                                     (helpers.hpp:11-12, helpers.cpp:190-407)
 *   sipoc_kkt_solve                   CallbackProvider::solve
 *                                     (helpers.hpp:13, helpers.cpp:749-951)
 *   sipoc_kkt_apply                   CallbackProvider::add_Kx_to_y
 *                                     (helpers.hpp:14-16, helpers.cpp:953-977)
 *   sipoc_kkt_residual                the ||K sol - rhs|| harness
 *                                     (tests/variable_dimensions_test.cpp:159-180,
 *                                     benchmarks/newton_kkt_benchmark.cpp:106-120)
 *   sipoc_*_sizes / sipoc_kkt_offsets Dimensions::get_*_dim (lqr.cpp:146-180),
 *                                     populate_workspace_metadata (types.cpp:24-64)
 *   *_host variants                   the same calls on HOST buffers in the
 *                                     reference's own memory order (what a
 *                                     thin C++ shim behind LQR / CallbackProvider
 *                                     passes), including host<->device copies.
 *
 * DATA LAYOUT
 *   "flat per-problem index": for each array the column-major blocks of all
 *   nodes (resp. edges) concatenated in node (edge) index order — exactly the
 *   memory a reference caller reaches through the double** tables of
 *   LQR::Input (lqr.hpp:76-89) when the blocks are stored back to back.
 *     Q: sum n_i*n_i   q,c,delta,x,y: sum n_i     (per node i)
 *     M: n_parent*m_e  R: m_e*m_e  r,u: m_e  A: n_child*n_parent  B: n_child*m_e
 *   HOST ("problem-major"):   X_host[b * size + flat]            b < batch
 *   DEVICE ("engine layout"): X_dev[flat * batch_stride + b]     batch innermost,
 *     batch_stride = sipoc_batch_stride() (batch rounded up to 32), so the
 *     lanes that work on neighbouring problems read neighbouring addresses.
 *   Q and R must be symmetric; like the reference's tests
 *   (selfadjointView<Lower>, tests/lqr_test.cpp:159,164) the fast kernels read
 *   only their lower triangles.
 *
 * ERRORS
 *   Every call returns a sipoc_error; nothing throws across the ABI.  Numerical
 *   failure is reported per problem with the reference's LQR::FactorStatus
 *   values (lqr.hpp:68-74), first failure in post-order wins
 *   (lqr.cpp:696-700,722-727).  x/u/y (sol) of a failed problem are unspecified.
 *   There is no CPU fallback: without a CUDA device sipoc_create fails with
 *   SIPOC_CUDA_ERROR.
 *
 * THREADING  A handle is not thread-safe; use one per host thread / stream.
 */
#ifndef SIPOC_H_
#define SIPOC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIPOC_VERSION 200

typedef struct sipoc_engine sipoc_engine;

typedef enum sipoc_error {
  SIPOC_OK = 0,
  SIPOC_INVALID_ARGUMENT = 1,
  SIPOC_CUDA_ERROR = 2,
  SIPOC_OUT_OF_MEMORY = 3,
  SIPOC_INVALID_TOPOLOGY = 4,   /* InputValidationStatus::INVALID_TOPOLOGY   */
  SIPOC_INVALID_DIMENSIONS = 5, /* InputValidationStatus::INVALID_DIMENSIONS */
  SIPOC_UNSUPPORTED = 6,
  SIPOC_NOT_FACTORED = 7
} sipoc_error;

/* Per-problem factor status == LQR::FactorStatus (lqr.hpp:68-74). */
typedef enum sipoc_factor_status {
  SIPOC_FACTOR_SUCCESS = 0,
  SIPOC_FACTOR_INVALID_DELTA = 1,
  SIPOC_FACTOR_F_FACTORIZATION_FAILURE = 2,
  SIPOC_FACTOR_G_FACTORIZATION_FAILURE = 3,
  SIPOC_FACTOR_INVALID_TOPOLOGY = 4
} sipoc_factor_status;

/* Topology (lqr.hpp:5-22) + Dimensions (lqr.hpp:24-33), shared by the batch.
 * The four constraint-dimension arrays may be NULL (= all zero, lqr.cpp:98-112).
 * theta_dim (global / Schur variables, at most 32) closes the x vector. */
typedef struct sipoc_structure {
  int num_edges;
  int root;
  const int *edge_parents;  /* [num_edges]     */
  const int *edge_children; /* [num_edges]     */
  const int *state_dims;    /* [num_edges + 1] */
  const int *control_dims;  /* [num_edges]     */
  const int *node_c_dims;   /* [num_edges + 1] or NULL */
  const int *node_g_dims;   /* [num_edges + 1] or NULL */
  const int *edge_c_dims;   /* [num_edges]     or NULL */
  const int *edge_g_dims;   /* [num_edges]     or NULL */
  int theta_dim;            /* 0 .. 32 */
  int64_t batch;            /* number of problems on this device */
  int device;               /* CUDA ordinal, -1 = current device */
  int flags;                /* SIPOC_FLAG_* */
} sipoc_structure;

#define SIPOC_FLAG_FORCE_GENERIC 1 /* never pick a shape-specialised kernel */
/* Chains whose dims vary from stage to stage run, padded to a uniform shape with
 * decoupled states / controls, on reference-order register kernels (same operations in
 * the same order as the generic kernels, hence the same parity at any regularization).
 * This flag picks the reordered shape-specialised kernels for them instead: faster
 * still, but a correct FP64 solve in another order, which drifts from the reference on
 * ill-conditioned regularization (r2 up to 1e9). */
#define SIPOC_FLAG_PAD_VARIABLE_DIMS 2
/* Parallel-in-time factor + solve (sipoc_lqr_factor_solve on uniform chains with a
 * sub-warp plan): the horizon is cut into segments whose conditional value functions are
 * combined by an associative scan, then every (problem, segment) tile is swept and rolled out
 * at once -- depth 2 (L + S) stage times instead of 2 N.  Chosen automatically for long
 * horizons with small batches (N >= 512 edges, batch <= 512); _PARALLEL_IN_TIME forces it,
 * _SERIAL_IN_TIME forbids it.  It needs R > 0 (a non-positive pivot of R reports
 * G_FACTORIZATION_FAILURE) and agrees with the serial recursion to rounding times the
 * conditioning of the segments, not bit for bit; the factorization it keeps is per segment,
 * so a later sipoc_lqr_solve needs its own sipoc_lqr_factor. */
#define SIPOC_FLAG_PARALLEL_IN_TIME 4
#define SIPOC_FLAG_SERIAL_IN_TIME 8

/* validate_input (types.cpp:68-134) on its own: SIPOC_OK, SIPOC_INVALID_DIMENSIONS or
 * SIPOC_INVALID_TOPOLOGY, dimension checks first.  Needs no device (batch is ignored). */
sipoc_error sipoc_validate(const sipoc_structure *structure);
sipoc_error sipoc_create(const sipoc_structure *structure, sipoc_engine **out);
void sipoc_destroy(sipoc_engine *engine);
int sipoc_version(void);
/* Message of the last failing call on this handle ("" if none). */
const char *sipoc_last_error(const sipoc_engine *engine);
/* Name of the kernel variant the handle dispatches LQR calls to. */
const char *sipoc_kernel_variant(const sipoc_engine *engine);
/* Compiled traversal orders (lqr.cpp:563-631); arrays sized E+2, E, E+1, E+1. */
sipoc_error sipoc_get_topology(const sipoc_engine *engine, int *child_offsets,
                               int *child_edges, int *preorder, int *postorder);
/* Kernels launched by this handle so far (each launch of one of OUR kernels). */
int64_t sipoc_launch_count(const sipoc_engine *engine);

/* Per-kernel device timing (bench tooling).  While enabled, every launch of one
 * of OUR kernels through this handle is bracketed by CUDA events on the
 * launching stream.  sipoc_profile_collect synchronises on them, folds the
 * spans by kernel name and returns the number of distinct names;
 * sipoc_profile_get reads entry `index` of that summary (name stays valid until
 * the next enable / collect).  Enabling or disabling clears recorded spans. */
sipoc_error sipoc_profile_enable(sipoc_engine *engine, int on);
int sipoc_profile_collect(sipoc_engine *engine);
sipoc_error sipoc_profile_get(const sipoc_engine *engine, int index, const char **name,
                              double *total_ms, int64_t *launches);

/* ---- CUDA graphs --------------------------------------------------------
 * The device entry points below only enqueue kernels on the caller's stream, so
 * any sequence of them -- e.g. one Newton-KKT iteration, sipoc_kkt_factor +
 * sipoc_kkt_solve + sipoc_kkt_residual (sip_optimal_control.cpp:129-145) -- can
 * be recorded once and relaunched with a single driver call.  Run the sequence
 * eagerly once first (workspaces are sized on first use, which may not happen
 * under capture); `stream` must be a non-default stream; the arrays the recorded
 * calls were given must stay allocated, their contents may change between
 * launches.  sipoc_graph_launch adds the recorded kernels to sipoc_launch_count.
 * While recording nothing executes: the handle's "a factorization exists" state is what it
 * was at sipoc_graph_begin again after sipoc_graph_end, and a call that would have to
 * allocate a workspace fails with SIPOC_INVALID_ARGUMENT (and a message saying so) instead
 * of breaking the capture.  A graph belongs to the handle it was recorded on (its kernels
 * point into that handle's workspaces): sipoc_destroy(engine) invalidates the engine's
 * graphs -- destroy them first, or at least never launch them afterwards. */
typedef struct sipoc_graph sipoc_graph;
sipoc_error sipoc_graph_begin(sipoc_engine *engine, void *stream);
sipoc_error sipoc_graph_end(sipoc_engine *engine, void *stream, sipoc_graph **out);
sipoc_error sipoc_graph_launch(sipoc_engine *engine, sipoc_graph *graph, void *stream);
int64_t sipoc_graph_kernel_count(const sipoc_graph *graph);
void sipoc_graph_destroy(sipoc_graph *graph);

/* ---- sizes ------------------------------------------------------------- */
typedef struct sipoc_lqr_sizes {
  int64_t Q, M, R, q, r, A, B, c, delta; /* inputs, elements per problem  */
  int64_t x, u, y;                       /* outputs, elements per problem */
} sipoc_lqr_sizes;
sipoc_error sipoc_lqr_get_sizes(const sipoc_engine *engine, sipoc_lqr_sizes *out);
int64_t sipoc_batch(const sipoc_engine *engine);
int64_t sipoc_batch_stride(const sipoc_engine *engine);

/* ---- LQR, device buffers in engine layout ------------------------------- */
typedef struct sipoc_lqr_input {
  const double *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
} sipoc_lqr_input;
typedef struct sipoc_lqr_output {
  double *x, *u, *y;
} sipoc_lqr_output;

/* stream: a cudaStream_t passed as void* (NULL = default stream).
 * status: device int[batch_stride], or NULL. */
sipoc_error sipoc_lqr_factor(sipoc_engine *engine, const sipoc_lqr_input *in,
                             int *status, void *stream);
/* Uses q, r, c (and A, B, delta) of `in` plus the stored factorization. */
sipoc_error sipoc_lqr_solve(sipoc_engine *engine, const sipoc_lqr_input *in,
                            const sipoc_lqr_output *out, void *stream);
/* One fused launch: factor + solve, keeping only what the rollout needs. */
sipoc_error sipoc_lqr_factor_solve(sipoc_engine *engine, const sipoc_lqr_input *in,
                                   const sipoc_lqr_output *out, int *status,
                                   void *stream);
/* The same three calls with the INPUT arrays problem-major on the device,
 * X[problem * size + flat] -- the layout of the *_host entry points, i.e. what a
 * caller holding one set of matrices per problem (LQR::Input's tables,
 * lqr.hpp:76-89) has after a plain copy.  Outputs and status stay in the engine
 * layout.  Native for the CTA-per-problem plans (state dimension >= 16), which
 * would otherwise transpose every call's inputs; every other plan packs the
 * arrays into the engine layout first.  Arrays must be 16-byte aligned. */
sipoc_error sipoc_lqr_factor_pm(sipoc_engine *engine, const sipoc_lqr_input *in,
                                int *status, void *stream);
sipoc_error sipoc_lqr_solve_pm(sipoc_engine *engine, const sipoc_lqr_input *in,
                               const sipoc_lqr_output *out, void *stream);
sipoc_error sipoc_lqr_factor_solve_pm(sipoc_engine *engine, const sipoc_lqr_input *in,
                                      const sipoc_lqr_output *out, int *status,
                                      void *stream);
/* residual_norm: device double[batch_stride] or NULL.  stats: device double[4]
 * or NULL, overwritten with {sum of squared norms, max norm, #failed problems
 * (status != 0; status may be NULL), #problems} over this device's batch —
 * the 4 numbers a multi-GPU driver all-reduces. */
sipoc_error sipoc_lqr_residual(sipoc_engine *engine, const sipoc_lqr_input *in,
                               const sipoc_lqr_output *out, const int *status,
                               double *residual_norm, double *stats, void *stream);

/* stats: device double[4], overwritten with {0, 0, #problems with status != 0,
 * #problems}: the failure / convergence flags of one Newton iteration in the
 * same 4-slot form as sipoc_lqr_residual, ready for an all-reduce(sum). */
sipoc_error sipoc_status_stats(sipoc_engine *engine, const int *status, double *stats,
                               void *stream);

/* ---- reverse-mode derivative of the LQR solve ------------------------------------------
 * The solve is K z = -h with z = (x, u, y), h = (q, r, c) and K symmetric.  For a cotangent
 * g = (g_x, g_u, g_y) = dL/d(x, u, y), sipoc_lqr_vjp writes the adjoint mu = -K^-1 g (the same
 * LQR solved with (q, r, c) := g) and, from dL = mu' (dK z + dh), the gradient of L with
 * respect to every input array, per problem, in that array's own layout:
 *   q, r, c : mu_x, mu_u, mu_y          delta_i : -mu_y_i .* y_i  (every node, root included)
 *   Q_i : (mu_x_i x_i' + x_i mu_x_i') / 2          R_e : (mu_u_e u_e' + u_e mu_u_e') / 2
 *   M_e : mu_x_p u_e' + x_p mu_u_e'                A_e : y_c mu_x_p' + mu_y_c x_p'
 *   B_e : y_c mu_u_e' + mu_y_c u_e'                (p / c: parent / child node of edge e)
 * Q and R get the gradient of the solve as a function of the SYMMETRIC matrices (the same
 * values in both triangles), although the kernels read only lower triangles: it is what a
 * caller who forms Q = (P + P') / 2 receives as dL/dQ.
 *   in      : Q, M, R, A, B, delta of the forward; q, r, c are not read and may be NULL.
 *   sol     : the forward's x, u, y.
 *   cot     : required, all three arrays.
 *   adjoint : caller-owned, receives mu (unspecified where status != 0).
 *   grad    : required; any of its arrays may be NULL, and is then neither computed nor
 *             written (a caller who wants dq / dc alone pays no matrix writes).
 *   status  : device int[batch_stride] receiving the adjoint factorization's per-problem
 *             FactorStatus, or NULL (an engine-owned buffer is used).
 * Every requested gradient array is written in full: zeros in problems whose status != 0
 * and in the padding lanes batch <= b < batch_stride, so every entry has a defined value.
 * All arrays in the engine layout, 16-byte aligned as for the other device entry points.
 * FP64 only.  The factorization is recomputed (the call keeps no state from the forward) on
 * the plan the forward uses, and it replaces the handle's kept LQR factorization the way
 * sipoc_lqr_factor_solve does.  The call only enqueues work on `stream`, so it can be
 * recorded in a graph under the rules above. */
typedef struct sipoc_lqr_cotangent {
  const double *x, *u, *y;
} sipoc_lqr_cotangent;
typedef struct sipoc_lqr_grad {
  double *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
} sipoc_lqr_grad;
sipoc_error sipoc_lqr_vjp(sipoc_engine *engine, const sipoc_lqr_input *in,
                          const sipoc_lqr_output *sol, const sipoc_lqr_cotangent *cot,
                          const sipoc_lqr_output *adjoint, const sipoc_lqr_grad *grad,
                          int *status, void *stream);

/* ---- forward-mode derivative of the LQR solve ------------------------------------------
 * From K z = -h, tangents (dK, dh) of the inputs move the solution by dz = -K^-1 (dK z + dh):
 * the same LQR solved with (q, r, c) := t = dK z + dh.  sipoc_lqr_jvp builds t per problem
 *   t_x_i = dQ_i x_i + dq_i + sum over the edges e with parent(e) = i of (dM_e u_e + dA_e' y_c)
 *   t_u_e = dR_e u_e + dr_e + dM_e' x_p + dB_e' y_c
 *   t_y_c = dA_e x_p + dB_e u_e - ddelta_c .* y_c + dc_c      (root: -ddelta_r .* y_r + dc_r)
 * (p / c: parent / child node of edge e) and solves for dz = (dx, du, dy).  dQ and dR enter
 * through their symmetric parts (dQ + dQ') / 2, read as full matrices: the exact transpose of
 * the symmetric gradient of sipoc_lqr_vjp, so <JVP(t), g> = <t, VJP(g)> for every tangent.
 *   in      : Q, M, R, A, B, delta of the forward; q, r, c are not read and may be NULL.
 *   sol     : the forward's x, u, y.
 *   tangent : required; any of its nine arrays may be NULL (a zero tangent: not read).
 *   rhs     : caller-owned (q, r, c)-shaped arrays, required, receiving t (zeros in the
 *             padding lanes batch <= b < batch_stride).
 *   dsol    : caller-owned, required, receives (dx, du, dy).
 *   status  : as for sipoc_lqr_vjp (the factorization's per-problem FactorStatus, or NULL).
 * dsol is written in full: zeros in problems whose status != 0 and in the padding lanes.
 * Everything else as for sipoc_lqr_vjp: engine layout, FP64, the factorization recomputed on
 * the forward's plan (replacing the handle's kept one), graph-capturable. */
sipoc_error sipoc_lqr_jvp(sipoc_engine *engine, const sipoc_lqr_input *in,
                          const sipoc_lqr_output *sol, const sipoc_lqr_input *tangent,
                          const sipoc_lqr_output *rhs, const sipoc_lqr_output *dsol,
                          int *status, void *stream);

/* ---- feedback policy of the LQR solve --------------------------------------------------
 * sipoc_lqr_factor_solve_policy does exactly what sipoc_lqr_factor_solve does, on the same
 * plan (x, u, y and status are bitwise the same, and the handle's kept factorization is
 * replaced the same way), then writes the policy the Riccati recursion computed, per problem:
 *   u_e = K_e x_p + k_e   (p: parent node of edge e)       y_i = V_i x_i + v_i
 * These are the reference's K, k, V, v after factor_with_status + solve (lqr.cpp:658,
 * :707-719, :744, :785-794).  V is the Hessian of the cost-to-go BEFORE the delta
 * regularization, so y_i = v_i + V_i x_i holds for the solution.  Layouts, per problem, in the
 * flat index of this header (each array reuses the element count of an input):
 *   K : per edge, m_e x n_p column-major (the element count of M)
 *   k : per edge, m_e                     (the element count of r)
 *   V : per node, n_i x n_i, both triangles, exactly symmetric on the shape-specialised
 *       plans (the element count of Q)
 *   v : per node, n_i                     (the element count of q)
 *   policy : required; any of its four arrays may be NULL, and is then neither computed nor
 *            written (K, k alone do not pay for V, which the plans that keep F^-1 instead
 *            rebuild per edge from Q, M, A, B, delta, F^-1 and K).
 *   status : as for sipoc_lqr_factor_solve, or NULL (an engine-owned buffer is used).
 * Every requested array is written in full: zeros in problems whose status != 0 and in the
 * padding lanes batch <= b < batch_stride.  FP64, device engine layout only, 16-byte aligned
 * arrays; the call only enqueues work on `stream` and can be recorded in a graph once it has
 * run eagerly (its workspaces are sized on the first call).  On the parallel-in-time plan a
 * node shared by two segments takes its values from the later one (node s L from segment s),
 * and the last node from the last segment. */
typedef struct sipoc_lqr_policy {
  double *K, *k, *V, *v;
} sipoc_lqr_policy;
sipoc_error sipoc_lqr_factor_solve_policy(sipoc_engine *engine, const sipoc_lqr_input *in,
                                          const sipoc_lqr_output *out,
                                          const sipoc_lqr_policy *policy, int *status,
                                          void *stream);

/* ---- reverse-mode derivative of the feedback policy -------------------------------------
 * For cotangents (Kb, kb, Vb, vb) = dL/d(K, k, V, v) of the policy sipoc_lqr_factor_solve_policy
 * returned, sipoc_lqr_policy_vjp writes the gradient of L with respect to the inputs, per
 * problem, in each input array's own layout.  It is the adjoint of the Riccati recursion, one
 * sweep from the root to the leaves: K_e and V_i are sensitivities of tail subproblems, not
 * functions of one solution, so they have no cheaper route through sipoc_lqr_vjp.  Per edge
 * the recursion is recomputed from the inputs and the forward's V, v (W_c from the Cholesky
 * factor of I + D^1/2 V_c D^1/2, K and k from that of G), so the call keeps no state from the
 * forward and works the same whichever plan ran it.  K and V do not depend on q, r, c: with
 * only Kb and Vb given, the gradients of q, r, c are exactly zero.
 *   in     : R, M, r, A, B, c, delta of the forward are read; Q and q are not and may be NULL.
 *   V, v   : the forward's policy arrays, required.  Only the lower triangle of V is read.
 *   status : the forward's per-problem FactorStatus, required.
 *   cot    : required; any of its four arrays may be NULL, which is bitwise the same as zeros.
 *   grad   : required; any of its arrays may be NULL, and is then neither computed nor
 *            written.  Q and R get the gradient with respect to the SYMMETRIC matrices (the
 *            same values in both triangles), as for sipoc_lqr_vjp.  The root's c and delta get
 *            zero gradient.
 * Every requested gradient array is written in full: zeros in problems whose status != 0 and
 * in the padding lanes batch <= b < batch_stride.  Any structure sipoc_lqr_factor_solve_policy
 * accepts.  FP64, engine layout, 16-byte aligned arrays.  Trees and shapes without a
 * specialised kernel use an engine-owned workspace sized on the first call, so the call can
 * be recorded in a graph once it has run eagerly. */
typedef struct sipoc_lqr_policy_cotangent {
  const double *K, *k, *V, *v;
} sipoc_lqr_policy_cotangent;
sipoc_error sipoc_lqr_policy_vjp(sipoc_engine *engine, const sipoc_lqr_input *in,
                                 const double *V, const double *v, const int *status,
                                 const sipoc_lqr_policy_cotangent *cot,
                                 const sipoc_lqr_grad *grad, void *stream);

/* ---- forward-mode derivative of the feedback policy -------------------------------------
 * For tangents (dQ, dM, dR, dq, dr, dA, dB, dc, ddelta) of the inputs, sipoc_lqr_policy_jvp
 * writes the tangents (dK, dk, dV, dv) of the policy sipoc_lqr_factor_solve_policy returned.
 * It is the tangent of the Riccati recursion, one sweep from the leaves to the root, the
 * direction of the factorization: each edge needs only its child's dV, dv.  Per edge
 * e = (p -> c), with the primal recomputed as sipoc_lqr_policy_vjp does (D = diag delta_c):
 *   P = (I + D^1/2 V_c D^1/2)^-1   W = D^-1/2 (I - P) D^-1/2   S = (I + D V_c)^-1
 *   G = R + B'WB   Y = WA   H = M' + B'Y   K = -G^-1 H
 *   f = delta_c .* v_c - c_c   g = v_c - W f   h = r + B'g   k = -G^-1 h
 *   dW = S' dV_c S - W dD W   dG = sym(dR) + dB'WB + B'W dB + B' dW B
 *   dY = dW A + W dA   dH = dM' + dB'Y + B' dY   dK = -G^-1 (dH + dG K)
 *   df = ddelta_c .* v_c + delta_c .* dv_c - dc_c   dg = dv_c - dW f - W df
 *   dh = dr + dB'g + B' dg   dk = -G^-1 (dh + dG k)
 *   dV_p += dA'Y + Y'dA + A' dW A + dH'K + K'dH + K' dG K   (exactly symmetric)
 *   dv_p += dA'g + A' dg + dK'h + K' dh
 * where every node starts from dV_i = sym(dQ_i), dv_i = dq_i.  Each convention is the
 * transpose of one of sipoc_lqr_policy_vjp, so <cot, JVP(t)> = <t, VJP(cot)> for every tangent:
 * dQ and dR enter through their symmetric parts (the full matrices are read), and the root's
 * dc and ddelta are not read (K and V do not depend on them).  Tangents of q, r and c alone give
 * dK = 0 and dV = 0 exactly.
 *   in      : R, M, r, A, B, c, delta of the forward are read; Q and q are not and may be NULL.
 *   V, v    : the forward's policy arrays, required.  Only the lower triangle of V is read.
 *   status  : the forward's per-problem FactorStatus, required.
 *   tangent : required; any of its nine arrays may be NULL, which is not read and gives
 *             bitwise the same result as zeros.
 *   dpolicy : required; any of its four arrays may be NULL, and is then not written.
 * Every requested output array is written in full: zeros in problems whose status != 0 and in
 * the padding lanes batch <= b < batch_stride.  dV is exactly symmetric.  Any structure
 * sipoc_lqr_factor_solve_policy accepts.  FP64, engine layout, 16-byte aligned arrays.  Trees
 * and shapes without a specialised kernel use an engine-owned workspace sized on the first
 * call, so the call can be recorded in a graph once it has run eagerly. */
sipoc_error sipoc_lqr_policy_jvp(sipoc_engine *engine, const sipoc_lqr_input *in,
                                 const double *V, const double *v, const int *status,
                                 const sipoc_lqr_input *tangent,
                                 const sipoc_lqr_policy *dpolicy, void *stream);

/* ---- layout conversion (device <-> device) ------------------------------ */
/* src: problem-major [batch][size]; dst: engine layout [size][batch_stride]. */
sipoc_error sipoc_pack(sipoc_engine *engine, const double *src, double *dst,
                       int64_t size, void *stream);
sipoc_error sipoc_unpack(sipoc_engine *engine, const double *src, double *dst,
                         int64_t size, void *stream);

/* ---- LQR, host buffers, problem-major (the reference-facing call) ------- */
/* Copies inputs host->device, converts layout, runs the fused factor+solve,
 * converts back and copies x/u/y and status to the host.  Synchronous. */
sipoc_error sipoc_lqr_factor_solve_host(sipoc_engine *engine,
                                        const sipoc_lqr_input *host_in,
                                        const sipoc_lqr_output *host_out,
                                        int *host_status);
/* The same call for a caller who can hand over less: the host-buffer path is bound by the
 * bus (177 KB per quadrotor problem), and a third of those bytes are the upper triangles of
 * the symmetric Q / R blocks and a cross term M that the reference's own benchmark sets to
 * zero (lqr_benchmark.cpp:61-96).  Here in->Q and in->R hold the PACKED LOWER TRIANGLES of
 * their blocks (column-major: entry (i, j), i >= j, of an n x n block at j n - j (j - 1) / 2
 * + (i - j); n (n + 1) / 2 doubles per block), in->M may be NULL (= 0); everything else as in
 * sipoc_lqr_factor_solve_host.  Uniform dims, plans on the interleaved layout (state
 * dimension < 16).  Not a reference interface: LQR::Input carries dense blocks. */
sipoc_error sipoc_lqr_factor_solve_host_packed(sipoc_engine *engine, const sipoc_lqr_input *in,
                                               const sipoc_lqr_output *out, int *host_status);
/* factor-once / solve-many on host buffers (BM_LQRSolve semantics,
 * lqr_benchmark.cpp:611-638): factor keeps the inputs and the factorization
 * resident; solve re-reads only q, r, c from host_in. */
sipoc_error sipoc_lqr_factor_host(sipoc_engine *engine, const sipoc_lqr_input *host_in,
                                  int *host_status);
sipoc_error sipoc_lqr_solve_host(sipoc_engine *engine, const sipoc_lqr_input *host_in,
                                 const sipoc_lqr_output *host_out);

/* ---- Newton-KKT ---------------------------------------------------------- */
/* With theta_dim > 0 the factor adds the Schur complement on the global variables
 * (helpers.cpp:372-407: J_theta, K_s^-1 J_theta by theta_dim stagewise solves against the
 * kept factorization, Cholesky of S) and solve / apply carry the theta rows
 * (helpers.cpp:902-951, theta branches of :1019-1368).
 * Flat vectors use the reference wire format (types.cpp:24-64):
 *   x = [x_0,u_0,...,x_{E-1},u_{E-1},x_E,theta]
 *   y = [dyn_0,node_c_0,...,dyn_E,node_c_E, edge_c_0..edge_c_{E-1}]
 *   z = [node_g_0..node_g_E, edge_g_0..edge_g_{E-1}],  KKT vectors = [x|y|z]. */
typedef struct sipoc_kkt_sizes {
  int64_t x_dim, y_dim, z_dim, kkt_dim;
  /* elements per problem of every model block array */
  int64_t node_hxx, node_jc, node_jg;
  int64_t edge_hxx, edge_hxu, edge_huu, edge_A, edge_B;
  int64_t edge_jcx, edge_jcu, edge_jgx, edge_jgu;
  /* theta (all zero when theta_dim == 0): x_dim = stagewise_x_dim + theta_dim */
  int64_t theta_dim, stagewise_x_dim;
  int64_t node_hxt, node_jct, node_jgt, node_htt;
  int64_t edge_hxt, edge_hut, edge_dynt, edge_jct, edge_jgt, edge_htt;
} sipoc_kkt_sizes;
sipoc_error sipoc_kkt_get_sizes(const sipoc_engine *engine, sipoc_kkt_sizes *out);
/* Offsets of every node / edge block in x, y, z (arrays sized E+1 or E). */
sipoc_error sipoc_kkt_offsets(const sipoc_engine *engine, int *x_state, int *x_control,
                              int *y_dyn, int *y_node_c, int *y_edge_c, int *z_node,
                              int *z_edge);

/* The ModelCallbackOutput blocks the reduction reads (types.hpp:48-89):
 * node d2L_dx2, dc_dx, dg_dx; edge d2L_dx2, d2L_dxdu, d2L_du2, ddyn_dx,
 * ddyn_du, dc_dx, dc_du, dg_dx, dg_du — flat, column-major per block. */
/* theta blocks of ModelCallbackOutput, p = theta_dim columns each, column-major:
 * node d2L_dxdtheta [n x p], dc_dtheta [c x p], dg_dtheta [g x p], d2L_dtheta2 [p x p];
 * edge d2L_dxdtheta [n_parent x p], d2L_dudtheta [m x p], ddyn_dtheta [n_child x p],
 * dc_dtheta [c x p], dg_dtheta [g x p], d2L_dtheta2 [p x p]   (helpers.cpp:190-240). */
typedef struct sipoc_kkt_theta_model {
  const double *node_hxt, *node_jct, *node_jgt, *node_htt;
  const double *edge_hxt, *edge_hut, *edge_dynt, *edge_jct, *edge_jgt, *edge_htt;
} sipoc_kkt_theta_model;
typedef struct sipoc_kkt_model {
  const double *node_hxx, *node_jc, *node_jg;
  const double *edge_hxx, *edge_hxu, *edge_huu, *edge_A, *edge_B;
  const double *edge_jcx, *edge_jcu, *edge_jgx, *edge_jgu;
  const sipoc_kkt_theta_model *theta; /* NULL when theta_dim == 0 */
} sipoc_kkt_model;

/* ok: device int[batch_stride]; 1 where CallbackProvider::factor returns true. */
sipoc_error sipoc_kkt_factor(sipoc_engine *engine, const sipoc_kkt_model *model,
                             const double *w, const double *r1, const double *r2,
                             const double *r3, int *ok, void *stream);
sipoc_error sipoc_kkt_solve(sipoc_engine *engine, const sipoc_kkt_model *model,
                            const double *b, double *sol, void *stream);
/* y += K(w, r1, r2, r3) x over [x|y|z] vectors (add_Kx_to_y). */
sipoc_error sipoc_kkt_apply(sipoc_engine *engine, const sipoc_kkt_model *model,
                            const double *w, const double *r1, const double *r2,
                            const double *r3, const double *x, double *y,
                            void *stream);
/* One block of that operator on its own (add_Hx_to_y, add_Cx_to_y, add_CTx_to_y,
 * add_Gx_to_y, add_GTx_to_y; helpers.hpp:17-21, helpers.cpp:979-1368), without the
 * regularization terms:  y += B x  with
 *   H : x, y of length x_dim      C : x x_dim, y y_dim      CT: x y_dim, y x_dim
 *   G : x x_dim, y z_dim          GT: x z_dim, y x_dim
 * (C holds the dynamics rows, node and edge equalities; G the inequalities). */
typedef enum sipoc_kkt_block {
  SIPOC_KKT_BLOCK_H = 0,
  SIPOC_KKT_BLOCK_C = 1,
  SIPOC_KKT_BLOCK_CT = 2,
  SIPOC_KKT_BLOCK_G = 3,
  SIPOC_KKT_BLOCK_GT = 4
} sipoc_kkt_block;
sipoc_error sipoc_kkt_apply_block(sipoc_engine *engine, const sipoc_kkt_model *model,
                                  int block, const double *x, double *y, void *stream);
/* ||K sol - b||_2 per problem and the 4 all-reducible statistics (see
 * sipoc_lqr_residual); ok may be NULL. */
sipoc_error sipoc_kkt_residual(sipoc_engine *engine, const sipoc_kkt_model *model,
                               const double *w, const double *r1, const double *r2,
                               const double *r3, const double *sol, const double *b,
                               const int *ok, double *residual_norm, double *stats,
                               void *stream);

/* ---- reverse-mode derivative of the Newton-KKT solve -----------------------------------
 * sipoc_kkt_solve computes sol = K^-1 b with K(w, r1, r2, r3) the operator of
 * sipoc_kkt_apply:
 *   K = [ H + diag(r1)   C'           G'            ]
 *       [ C              -diag(r2)    0             ]
 *       [ G              0            -diag(w + r3) ]
 * K is symmetric.  For a cotangent g = dL/dsol, sipoc_kkt_vjp writes the adjoint
 * lam = K^-1 g (the same KKT solve with b := g) and, from dL = lam' db - lam' dK sol, the
 * gradient of L with respect to every model block, b and the regularization vectors, per
 * problem, in each array's own layout.  With s_R, lam_R the rows of sol, lam in a row range R
 * of [x | y | z], a block at K[R, C] (its transpose at K[C, R]) gets
 *   -(lam_R s_C' + s_R lam_C')            off-diagonal blocks
 *   -(lam_R s_R' + s_R lam_R') / 2        the symmetric Hessian blocks (R == C)
 * at (p / c: parent / child node of edge e; theta: the theta rows of x)
 *   node_hxx_i  x_state(i) x x_state(i)  sym     edge_hxx_e  x_state(p) x x_state(p)  sym
 *   edge_hxu_e  x_state(p) x x_control(e)        edge_huu_e  x_control(e) x x_control(e) sym
 *   edge_A_e, edge_B_e    y_dyn(c) x x_state(p), x_control(e)
 *   node_jc_i, node_jg_i  y_node_c(i), z_node(i) x x_state(i)
 *   edge_jcx_e, edge_jcu_e  y_edge_c(e) x x_state(p), x_control(e)
 *   edge_jgx_e, edge_jgu_e  z_edge(e) x x_state(p), x_control(e)
 *   node_hxt, node_jct, node_jgt  x_state(i), y_node_c(i), z_node(i) x theta
 *   edge_hxt, edge_hut, edge_dynt, edge_jct, edge_jgt
 *                         x_state(p), x_control(e), y_dyn(c), y_edge_c(e), z_edge(e) x theta
 *   node_htt_i, edge_htt_e  theta x theta  sym (every copy gets the same value)
 * and the vectors  db = lam,  dr1 = -lam_x .* s_x (theta rows included),
 * dr2 = lam_y .* s_y,  dw = dr3 = lam_z .* s_z.  The -I couplings of the dynamics rows are
 * constants.  Symmetric blocks get the gradient with respect to the SYMMETRIC matrix (the
 * same values in both triangles): what a caller who forms H = (P + P') / 2 receives as dL/dH.
 *   model, w, r1, r2, r3 : those of the forward (validated as by sipoc_kkt_factor).
 *   sol     : the forward's solution;  cot : dL/dsol, required.
 *   adjoint : caller-owned [x | y | z] vector, required, receives lam (unspecified where
 *             ok == 0).
 *   grad    : required; any of its arrays may be NULL, and is then neither computed nor
 *             written; theta may be NULL (no theta gradient).  w and r3 may be one array.
 *   ok      : device int[batch_stride] receiving the factorization's per-problem flags (as
 *             sipoc_kkt_factor), or NULL (an engine-owned buffer is used).
 * Every requested gradient array is written in full: zeros in problems whose ok == 0 and in
 * the padding lanes batch <= b < batch_stride.  All arrays in the engine layout.  FP64 only.
 * The factorization is recomputed on (model, w, r1, r2, r3) -- the call keeps no state from
 * the forward -- on the plan sipoc_kkt_factor uses, and it replaces the handle's kept KKT
 * factorization the way sipoc_kkt_factor does.  The call only enqueues work on `stream`, so
 * it can be recorded in a graph under the rules above. */
typedef struct sipoc_kkt_theta_grad {
  double *node_hxt, *node_jct, *node_jgt, *node_htt;
  double *edge_hxt, *edge_hut, *edge_dynt, *edge_jct, *edge_jgt, *edge_htt;
} sipoc_kkt_theta_grad;
typedef struct sipoc_kkt_grad {
  double *node_hxx, *node_jc, *node_jg;
  double *edge_hxx, *edge_hxu, *edge_huu, *edge_A, *edge_B;
  double *edge_jcx, *edge_jcu, *edge_jgx, *edge_jgu;
  const sipoc_kkt_theta_grad *theta; /* NULL: no theta gradient */
  double *b, *w, *r1, *r2, *r3;
} sipoc_kkt_grad;
sipoc_error sipoc_kkt_vjp(sipoc_engine *engine, const sipoc_kkt_model *model, const double *w,
                          const double *r1, const double *r2, const double *r3,
                          const double *sol, const double *cot, double *adjoint,
                          const sipoc_kkt_grad *grad, int *ok, void *stream);

/* ---- forward-mode derivative of the Newton-KKT solve -----------------------------------
 * From sol = K^-1 b, tangents of the inputs move the solution by d sol = K^-1 (db - dK sol):
 * the same KKT solve with b := t = db - dK sol.  dK holds the tangent model blocks where the
 * table of sipoc_kkt_vjp places them (every copy of node_htt / edge_htt adds to the theta x
 * theta block), diag(dr1) on the x rows (theta rows included), -diag(dr2) on the y rows and
 * -diag(dw + dr3) on the z rows; the -I couplings of the dynamics rows are constants.  The
 * symmetric Hessian blocks enter through their symmetric parts (dB + dB') / 2, read as full
 * matrices: the exact transpose of the symmetric gradient of sipoc_kkt_vjp.
 *   model, w, r1, r2, r3 : those of the forward (validated as by sipoc_kkt_factor).
 *   sol     : the forward's solution.
 *   tangent : required; every block pointer, model.theta, and b, w, r1, r2, r3 may be NULL
 *             (a zero tangent: not read).  w and r3 may be one array, here and in the forward.
 *   rhs     : caller-owned [x | y | z] vector, required, receiving t (zeros in the padding
 *             lanes).
 *   dsol    : caller-owned [x | y | z] vector, required, receives d sol.
 *   ok      : as for sipoc_kkt_vjp.
 * dsol is written in full: zeros in problems whose ok == 0 and in the padding lanes.
 * Everything else as for sipoc_kkt_vjp: engine layout, FP64, the factorization recomputed on
 * the forward's plan (replacing the handle's kept one), graph-capturable. */
typedef struct sipoc_kkt_tangent {
  sipoc_kkt_model model;
  const double *b, *w, *r1, *r2, *r3;
} sipoc_kkt_tangent;
sipoc_error sipoc_kkt_jvp(sipoc_engine *engine, const sipoc_kkt_model *model, const double *w,
                          const double *r1, const double *r2, const double *r3,
                          const double *sol, const sipoc_kkt_tangent *tangent, double *rhs,
                          double *dsol, int *ok, void *stream);

/* ---- optional FP32 mode ----------------------------------------------------------------
 * north_star: "an optional FP32 mode is reported separately with its own stated tolerance".
 * Factor + solve (LQR::factor + LQR::solve, lqr.hpp:192-194) entirely in single precision:
 * every array is float in the engine layout X[flat * batch_stride + problem].  Covered:
 * uniform chains with state dimension 4 and 1..4 controls (the cartpole row of the
 * reference benchmark grid, lqr_benchmark.cpp:537-545) -- sipoc_f32_supported tells.
 * Stated tolerance: 5e-4 relative on (x, u, y) against the FP64 oracle run on the same
 * (float-rounded) inputs, on the benchmark distribution (delta in [1e-3, 0.101]); the same
 * per-problem FactorStatus values as the FP64 path.  The kept factorization is private to the
 * call (no separate solve).  sipoc_lqr_factor_solve_thread_f64 runs the SAME kernels
 * instantiated on double: their numerical control, held to the FP64 tolerance by the tests. */
typedef struct sipoc_lqr_input_f32 {
  const float *Q, *M, *R, *q, *r, *A, *B, *c, *delta;
} sipoc_lqr_input_f32;
typedef struct sipoc_lqr_output_f32 {
  float *x, *u, *y;
} sipoc_lqr_output_f32;
int sipoc_f32_supported(const sipoc_engine *engine);
sipoc_error sipoc_lqr_factor_solve_f32(sipoc_engine *engine, const sipoc_lqr_input_f32 *in,
                                       const sipoc_lqr_output_f32 *out, int *status,
                                       void *stream);
sipoc_error sipoc_lqr_factor_solve_thread_f64(sipoc_engine *engine, const sipoc_lqr_input *in,
                                              const sipoc_lqr_output *out, int *status,
                                              void *stream);

/* ---- model-callback scatter ----------------------------------------------------------
 * The model_callback lambda of sip_optimal_control.cpp:13-127, after the user's callback has
 * produced the node / edge values of one evaluation: objective f = sum of the node and edge
 * f (:44-50); gradient_f = df_dx, df_du, df_dtheta scattered to the x layout (:54-85);
 * c = [initial_state - x_root | node c | edge dyn_res | edge c] in the y layout (:87-109);
 * g = node / edge g in the z layout (:111-122).  Value arrays concatenate the per-node
 * (per-edge) vectors in index order (NodeModelCallbackOutput / EdgeModelCallbackOutput,
 * types.hpp:48-89); sipoc_model_value_sizes gives the elements per problem of each.
 * new_x == 0 computes f only (the reference's `if (mci.new_x)`, :52).  Sums are formed in
 * the reference's order, so the result is bit-identical to it. */
typedef struct sipoc_model_value_sizes_t {
  int64_t node_f, node_df_dx, node_df_dtheta, node_c, node_g;
  int64_t edge_f, edge_df_dx, edge_df_du, edge_df_dtheta, edge_dyn_res, edge_c, edge_g;
} sipoc_model_value_sizes_t;
typedef struct sipoc_model_values {
  const double *node_f, *node_df_dx, *node_df_dtheta, *node_c, *node_g;
  const double *edge_f, *edge_df_dx, *edge_df_du, *edge_df_dtheta, *edge_dyn_res, *edge_c,
      *edge_g;
} sipoc_model_values;
sipoc_error sipoc_model_value_sizes(const sipoc_engine *engine, sipoc_model_value_sizes_t *out);
/* Device arrays, engine layout: x [x_dim], initial_state [n_root], f [1], gradient_f [x_dim],
 * c [y_dim], g [z_dim] elements per problem. */
sipoc_error sipoc_model_scatter(sipoc_engine *engine, const sipoc_model_values *values,
                                const double *x, const double *initial_state, int new_x,
                                double *f, double *gradient_f, double *c, double *g,
                                void *stream);
/* Host buffers, problem-major ([batch][elements per problem]), synchronous. */
sipoc_error sipoc_model_scatter_host(sipoc_engine *engine, const sipoc_model_values *values,
                                     const double *x, const double *initial_state, int new_x,
                                     double *f, double *gradient_f, double *c, double *g);

/* Host-buffer variants (problem-major), synchronous. */
sipoc_error sipoc_kkt_factor_host(sipoc_engine *engine, const sipoc_kkt_model *host_model,
                                  const double *w, const double *r1, const double *r2,
                                  const double *r3, int *host_ok);
sipoc_error sipoc_kkt_solve_host(sipoc_engine *engine, const double *b, double *sol);
/* Uploads the model alone: what sipoc_kkt_apply_host / sipoc_kkt_apply_block_host read.  The
 * reference's add_*x_to_y read the CURRENT model_callback_output (helpers.cpp:1161-1183), so
 * a shim calls this whenever the model callback has run since the last upload. */
sipoc_error sipoc_kkt_set_model_host(sipoc_engine *engine, const sipoc_kkt_model *host_model);
sipoc_error sipoc_kkt_apply_host(sipoc_engine *engine, const double *w, const double *r1,
                                 const double *r2, const double *r3, const double *x,
                                 double *y);

/* y += B x for one block, against the model uploaded by the last
 * sipoc_kkt_factor_host (vector lengths as for sipoc_kkt_apply_block). */
sipoc_error sipoc_kkt_apply_block_host(sipoc_engine *engine, int block, const double *x,
                                       double *y);

/* ---- several devices ------------------------------------------------------
 * The path shards trivially: problems are independent, so a batch is cut into contiguous
 * slices, one engine handle per device, with no data-path collective.  The only exchange
 * per Newton iteration is the all-reduce of the 4 statistics the residual / status entry
 * points write ({sum of squared norms, max norm, #failed, #problems}: slots 0, 2, 3 are
 * summed, slot 1 is max-reduced).  A communicator is one rank's endpoint of an NCCL
 * clique (NCCL is loaded with dlopen on first use; SIPOC_UNSUPPORTED if absent):
 *   one process per GPU : rank 0 calls sipoc_comm_unique_id and ships the 128 bytes to the
 *                         other ranks by whatever channel the host has (MPI, torch.distributed,
 *                         a file); every rank calls sipoc_comm_create.
 *   one process, n GPUs : sipoc_comm_create_all; collectives issued for several
 *                         communicators from one thread go between sipoc_comm_group_begin / _end.
 * sipoc_attach_comm makes the engine finish every `stats` it writes (sipoc_lqr_residual,
 * sipoc_kkt_residual, sipoc_status_stats) with that all-reduce, on the call's stream --
 * one all-gather of 4 doubles per rank plus a one-warp fold kernel, capturable in a graph. */
#define SIPOC_COMM_ID_BYTES 128
typedef struct sipoc_comm sipoc_comm;
sipoc_error sipoc_shard_range(int64_t total, int rank, int world, int64_t *begin, int64_t *end);
sipoc_error sipoc_comm_unique_id(void *id_out /* SIPOC_COMM_ID_BYTES */);
sipoc_error sipoc_comm_create(const void *id, int rank, int world, int device /* -1 = current */,
                              sipoc_comm **out);
sipoc_error sipoc_comm_create_all(const int *device_ids, int n_dev, sipoc_comm **out /* [n_dev] */);
void sipoc_comm_destroy(sipoc_comm *comm);
int sipoc_comm_rank(const sipoc_comm *comm);
int sipoc_comm_size(const sipoc_comm *comm);
sipoc_error sipoc_comm_group_begin(void);
sipoc_error sipoc_comm_group_end(void);
/* stats: device double[4] on the communicator's device, reduced in place. */
sipoc_error sipoc_comm_allreduce_stats(sipoc_comm *comm, double *stats, void *stream);
/* The two halves, for several communicators driven by one thread: all gathers inside one
 * group, then the folds. */
sipoc_error sipoc_comm_allgather_stats(sipoc_comm *comm, const double *stats, void *stream);
sipoc_error sipoc_comm_fold_stats(sipoc_comm *comm, double *stats, void *stream);
/* comm may be NULL (detach).  The communicator must outlive the engine's calls. */
sipoc_error sipoc_attach_comm(sipoc_engine *engine, sipoc_comm *comm);

/* ---- synthetic workloads (bench / test tooling) -------------------------- */
/* Fills engine-layout device buffers with the distribution of the reference's
 * LQRProblem generator (benchmarks/lqr_benchmark.cpp:61-96): A = I + 0.05 N,
 * B = 0.1 N, M = 0, R = Z'Z + 1.01 I, Q = Z'Z + 1e-3 I, q, r, c ~ N(0,1),
 * delta = 1e-3 + 0.1 U(0,1), from a counter-based generator keyed by
 * (seed, problem_offset + b, array, element).  Uniform chains only. */
sipoc_error sipoc_generate_lqr_benchmark(sipoc_engine *engine, uint64_t seed,
                                         int64_t problem_offset, double *Q, double *M,
                                         double *R, double *q, double *r, double *A,
                                         double *B, double *c, double *delta,
                                         void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SIPOC_H_ */
