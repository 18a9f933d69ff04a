// C ABI of the engine (include/sipoc.h): handle management, dispatch between
// the generic and the shape-specialised kernels, and the host-buffer entry
// points that wrap copies + layout conversion around the device path.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <iterator>
#include <new>
#include <string>
#include <vector>

#include "../../include/sipoc.h"
#include "generic_kernels.cuh"
#include "kkt_fast.cuh"
#include "kkt_theta.cuh"
#include "jvp.cuh"
#include "kkt_vjp.cuh"
#include "lqr_vjp.cuh"
#include "policy.cuh"
#include "policy_jvp.cuh"
#include "policy_vjp.cuh"
#include "scan.cuh"
#include "model_scatter.cuh"
#include "riccati_f32.cuh"
#include "profile.hpp"
#include "riccati_fast.cuh"
#include "structure.hpp"
#include "workload.cuh"

using namespace sipoc;

struct sipoc_engine {
  HostStructure hs;
  DevTables dt{};
  int *d_tab = nullptr;
  int device = 0;
  int flags = 0;
  int64_t batch = 0, ld = 0;
  const FastPlan *fast = nullptr;
  KktReduceFn kkt_reduce_fast = nullptr;
  KktApplyFn kkt_apply_fast = nullptr;
  int kkt_max_rows = 0;
  std::string variant;
  std::string last_error;
  int64_t launches = 0;
  bool capturing = false;          // between sipoc_graph_begin and sipoc_graph_end
  int64_t capture_launches0 = 0;
  // What a capture must not change: nothing runs while recording, so the "a factorization
  // exists" flags are put back at sipoc_graph_end.
  struct CaptureSaved {
    int factored = 0;
    bool kkt_factored = false, host_lqr_factored = false;
  } capture_saved;
  std::vector<struct sipoc_graph *> graphs;  // live graphs recorded on this handle
  Profiler prof;
  cudaStream_t host_stream = nullptr;

  // Every device allocation the handle owns.
  std::vector<void *> allocations;

  // Generic factorization workspace (lazy).
  LqrWs gws{};
  bool gws_ready = false;
  // Fast-path storage (lazy).
  double *fast_store = nullptr, *fast_scratch = nullptr;
  double *pm_in[9] = {nullptr};  // problem-major input copies (plans that ask for them)
  double *il_in[9] = {nullptr};  // interleaved copies of problem-major caller arrays (*_pm calls)
  // Chains whose dims vary from stage to stage run on the plan of the smallest uniform
  // shape that holds every stage, through decoupled padding (generic_kernels.cu, pad_chain_kernel).
  bool padded = false;
  double *pad_in[9] = {nullptr};
  double *pad_out[3] = {nullptr};
  enum class Factored { NONE, GENERIC, FAST } factored = Factored::NONE;

  // Newton-KKT reduction outputs (lazy).
  KktWs kws{};
  bool kws_ready = false;
  int *kkt_lqr_status = nullptr;
  bool kkt_factored = false;
  // The padded / problem-major copies of A, B, delta were made by kkt_factor from the model
  // it was given (so kkt_solve may skip refreshing them); any other solve overwrites them.
  bool kept_copies_are_kkt = false;
  double *kkt_product = nullptr;  // K * sol scratch of sipoc_kkt_residual
  // theta (Schur) layer (lazy): J and K_s^-1 J [kkt_dim x p], the factor of S [p x p], p scratch
  double *theta_J = nullptr, *theta_KinvJ = nullptr, *theta_S = nullptr, *theta_t = nullptr;

  // Host-API resident buffers (lazy).
  double *h_in[9] = {nullptr};
  double *h_out[3] = {nullptr};
  double *h_stage = nullptr;
  int64_t h_stage_elems = 0;
  int *h_status = nullptr;
  bool host_lqr_ready = false;
  bool host_lqr_factored = false;
  double *hk_model[12] = {nullptr};
  double *hk_theta[10] = {nullptr};
  double *hk_reg[4] = {nullptr};  // w, r1, r2, r3
  double *hk_vec[2] = {nullptr};  // b / x, sol / y
  bool host_kkt_ready = false;
  bool host_model_resident = false;  // hk_model / hk_theta hold a caller's model
  sipoc_comm *comm = nullptr;        // attached communicator: stats outputs are all-reduced
  // model-callback scatter, host-buffer variant: values, x, x0 | f, gradient_f, c, g
  double *hm_vals[12] = {}, *hm_x = nullptr, *hm_x0 = nullptr, *hm_out[4] = {};
  bool host_scatter_ready = false;
  // Optional FP32 mode (riccati_f32.cu): kept factorization + spill in single precision, and
  // the double instantiation of the same kernels (numerical control)
  float *f32_store = nullptr;
  double *f64t_store = nullptr;
  double *h_packed = nullptr;  // packed-symmetric host entry: Q / R triangles before expansion
  int *vjp_status = nullptr;   // status / ok of sipoc_*_vjp / _jvp when the caller passes none (lazy)
  double *policy_V = nullptr;  // V rebuilt in a padded plan's shape, before extraction (lazy)
  double *policy_vjp_ws = nullptr;  // edge scratch and per-node Vb, vb of the generic policy VJP (lazy)
  double *policy_jvp_ws = nullptr;  // edge scratch and per-node dV, dv of the generic policy JVP (lazy)

  // Parallel-in-time factor + solve (scan.cu): long uniform chains, small batches.
  struct Scan {
    bool enabled = false;
    int L = 0, S = 0, Sg = 0;  // edges per segment, segments, segments per group
    double *elems = nullptr, *gelems = nullptr, *maps = nullptr, *Vb = nullptr, *vb = nullptr, *xb = nullptr;
    double *store = nullptr, *scratch = nullptr;
    int *seg_status = nullptr, *sweep_status = nullptr;
  } scan;
};

namespace {

sipoc_error fail(sipoc_engine *e, sipoc_error code, const std::string &msg) {
  if (e != nullptr) e->last_error = msg;
  return code;
}

#define SIPOC_CUDA(e, call)                                                      \
  do {                                                                           \
    cudaError_t err__ = (call);                                                  \
    if (err__ != cudaSuccess) {                                                  \
      return fail((e),                                                           \
                  err__ == cudaErrorMemoryAllocation ? SIPOC_OUT_OF_MEMORY       \
                                                     : SIPOC_CUDA_ERROR,         \
                  std::string(#call) + ": " + cudaGetErrorString(err__));        \
    }                                                                            \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

sipoc_error dev_alloc(sipoc_engine *e, void **out, size_t bytes) {
  *out = nullptr;
  if (bytes == 0) bytes = 16;
  if (e->capturing)  // cudaMalloc would invalidate the capture (thread-local mode)
    return fail(e, SIPOC_INVALID_ARGUMENT,
                "a workspace would be allocated while a graph is being recorded: run the same "
                "sequence of calls eagerly once before sipoc_graph_begin");
  SIPOC_CUDA(e, cudaMalloc(out, bytes));
  e->allocations.push_back(*out);
  return SIPOC_OK;
}

sipoc_error alloc_doubles(sipoc_engine *e, double **out, int64_t elems_per_problem) {
  return dev_alloc(e, reinterpret_cast<void **>(out),
                   static_cast<size_t>(std::max<int64_t>(elems_per_problem, 1)) *
                       static_cast<size_t>(e->ld) * sizeof(double));
}

sipoc_error check_launch(sipoc_engine *e, const char *what) {
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess)
    return fail(e, SIPOC_CUDA_ERROR, std::string(what) + ": " + cudaGetErrorString(err));
  return SIPOC_OK;
}

void rebase(DevTables &t, const int *base) {
  const int **fields[] = {
      &t.parents,      &t.children,    &t.n,          &t.m,           &t.child_offsets,
      &t.child_edges,  &t.preorder,    &t.postorder,  &t.in_edge,     &t.nn_off,
      &t.n_off,        &t.nm_off,      &t.mm_off,     &t.m_off,       &t.a_off,
      &t.b_off,        &t.w_off,       &t.k_off,      &t.hxx_edge_off, &t.node_c,
      &t.node_g,       &t.edge_c,      &t.edge_g,     &t.x_state,     &t.y_dyn,
      &t.y_node_c,     &t.z_node,      &t.x_control,  &t.y_edge_c,    &t.z_edge,
      &t.jc_node_off,  &t.jg_node_off, &t.jcx_off,    &t.jcu_off,     &t.jgx_off,
      &t.jgu_off,      &t.node_c_off,  &t.node_g_off, &t.edge_c_off,  &t.edge_g_off,
      &t.pn_off,       &t.cn_off};
  for (const int **f : fields) {
    const size_t byte_off = reinterpret_cast<size_t>(*f);
    *f = reinterpret_cast<const int *>(reinterpret_cast<const char *>(base) + byte_off);
  }
}

sipoc_error ensure_generic_ws(sipoc_engine *e) {
  if (e->gws_ready) return SIPOC_OK;
  const HostStructure &h = e->hs;
  sipoc_error rc;
  const int64_t mn = std::max(1, h.max_n), mm = std::max(1, h.max_m);
#define A_(field, elems) \
  if ((rc = alloc_doubles(e, &e->gws.field, (elems))) != SIPOC_OK) return rc;
  A_(W, h.w_off[h.E]);
  A_(K, h.k_off[h.E]);
  A_(V, h.nn_off[h.N]);
  A_(Gf, h.mm_off[h.E]);
  A_(Ff, h.nn_off[h.N]);
  A_(sd, h.n_off[h.N]);
  A_(sdi, h.n_off[h.N]);
  A_(k, h.m_off[h.E]);
  A_(v, h.n_off[h.N]);
  A_(H, mm * mn);
  A_(F, mn * mn);
  A_(f, mn);
  A_(g, mn);
  A_(h, mm);
#undef A_
  e->gws_ready = true;
  return SIPOC_OK;
}

sipoc_error ensure_fast_store(sipoc_engine *e) {
  if (e->fast == nullptr || e->fast_store != nullptr) return SIPOC_OK;
  sipoc_error rc = alloc_doubles(e, &e->fast_store, e->fast->store_elems(e->hs.E));
  return rc;
}

sipoc_error ensure_fast_scratch(sipoc_engine *e) {
  if (e->fast == nullptr || e->fast_scratch != nullptr) return SIPOC_OK;
  return alloc_doubles(e, &e->fast_scratch, e->fast->scratch_elems(e->hs.E));
}

sipoc_error ensure_kkt_ws(sipoc_engine *e) {
  if (e->kws_ready) return SIPOC_OK;
  const HostStructure &h = e->hs;
  sipoc_error rc;
#define A_(field, elems) \
  if ((rc = alloc_doubles(e, &e->kws.field, (elems))) != SIPOC_OK) return rc;
  A_(Q_mod, h.nn_off[h.N]);
  A_(M_mod, h.nm_off[h.E]);
  A_(R_mod, h.mm_off[h.E]);
  A_(q_mod, h.n_off[h.N]);
  A_(r_mod, h.m_off[h.E]);
  A_(c_mod, h.n_off[h.N]);
  A_(dyn_r2, h.n_off[h.N]);
  A_(node_c_r2_inv, h.node_c_off[h.N]);
  A_(edge_c_r2_inv, h.edge_c_off[h.E]);
  A_(node_mod_w_inv, h.node_g_off[h.N]);
  A_(edge_mod_w_inv, h.edge_g_off[h.E]);
  A_(x, h.n_off[h.N]);
  A_(u, h.m_off[h.E]);
  A_(y, h.n_off[h.N]);
#undef A_
  rc = dev_alloc(e, reinterpret_cast<void **>(&e->kkt_lqr_status),
                 static_cast<size_t>(e->ld) * sizeof(int));
  if (rc != SIPOC_OK) return rc;
  e->kws_ready = true;
  return SIPOC_OK;
}

LqrIn to_in(const sipoc_lqr_input *in) {
  return LqrIn{in->Q, in->M, in->R, in->q, in->r, in->A, in->B, in->c, in->delta};
}

// The fused Newton-KKT solve kernels (rhs build inside the affine sweep, dual recovery
// inside the rollout) run one thread per problem; the unfused generic rhs / recovery
// kernels spread a problem over its nodes.  Measured on B200 at quadrotor dims, c = 6,
// g = 8: batch 8 192 -> fused 2.58 ms, unfused 1.76 ms; batch 65 536 -> fused 6.75 ms,
// unfused 7.41 ms.  Fusion pays once a thread per problem fills the machine.
constexpr int64_t kFusedKktMinBatch = 32768;

// The sub-warp kernels stage operands with 16-byte cp.async: every engine-layout
// array must be 16-byte aligned (any cudaMalloc / torch allocation is).  A
// misaligned call is served by the generic kernels instead.
bool aligned16(const LqrIn &in) {
  const double *p[9] = {in.Q, in.M, in.R, in.q, in.r, in.A, in.B, in.c, in.delta};
  for (const double *q : p)
    if ((reinterpret_cast<uintptr_t>(q) & 15u) != 0) return false;
  return true;
}
bool use_fast(const sipoc_engine *e, const LqrIn &in) {
  return e->fast != nullptr && aligned16(in);
}

int64_t lqr_in_size(const HostStructure &h, int i);
// Elements per problem of input array i as the plan's kernels see it: the uniform padded
// shape on padded plans, the structure's own sizes otherwise.
int64_t plan_in_size(const sipoc_engine *e, int i) {
  if (!e->padded) return lqr_in_size(e->hs, i);
  const int64_t np = e->fast->n, mp = e->fast->m, N = e->hs.N, E = e->hs.E;
  const int64_t sizes[9] = {N * np * np, E * np * mp, E * mp * mp, N * np, E * mp,
                            E * np * np, E * np * mp, N * np,      N * np};
  return sizes[i];
}

// Plans whose kernels run one problem per CTA read the inputs from problem-major copies
// [problem][flat]; this transposes the arrays the call touches (coalesced passes, a few
// percent of the work they feed).  `mask` bit i selects array i of
// {Q, M, R, q, r, A, B, c, delta}.
constexpr unsigned kPmMatrices = 0b101100111;  // Q M R A B delta
constexpr unsigned kPmAll = 0b111111111;
constexpr unsigned kPmSolve = 0b111111000;     // q r A B c delta
sipoc_error refresh_problem_major(sipoc_engine *e, const LqrIn &in, unsigned mask, LqrIn *pm,
                                  cudaStream_t s) {
  *pm = LqrIn{};
  if (e->fast == nullptr || !e->fast->problem_major_inputs) return SIPOC_OK;
  const double *src[9] = {in.Q, in.M, in.R, in.q, in.r, in.A, in.B, in.c, in.delta};
  for (int i = 0; i < 9; ++i) {
    if ((mask >> i & 1u) == 0) continue;
    const int64_t size = plan_in_size(e, i);
    if (e->pm_in[i] == nullptr) {
      sipoc_error rc = dev_alloc(e, reinterpret_cast<void **>(&e->pm_in[i]),
                                 static_cast<size_t>(std::max<int64_t>(size, 1)) *
                                     static_cast<size_t>(e->batch) * sizeof(double));
      if (rc != SIPOC_OK) return rc;
    }
    ProfScope ps(&e->prof, "unpack_kernel", s);
    launch_unpack(src[i], e->pm_in[i], size, e->batch, e->ld, s);
    e->launches += 1;
  }
  *pm = LqrIn{e->pm_in[0], e->pm_in[1], e->pm_in[2], e->pm_in[3], e->pm_in[4],
              e->pm_in[5], e->pm_in[6], e->pm_in[7], e->pm_in[8]};
  return SIPOC_OK;
}

// The *_pm entry points take the input arrays problem-major.  Plans that want that
// layout use the caller's arrays in place; for every other path the arrays `mask`
// selects are packed into interleaved copies first.
//   layout_pm == false: *il = in, *pm = the engine's problem-major copies (if the plan wants them)
//   layout_pm == true : *il = {} and *pm = in (native), or *il = packed copies and *pm = {}
sipoc_error resolve_inputs(sipoc_engine *e, const LqrIn &in, bool layout_pm, unsigned mask,
                           LqrIn *il, LqrIn *pm, cudaStream_t s) {
  *pm = LqrIn{};
  if (!layout_pm) {
    *il = in;
    // (padded plans transpose after the padding: pad_inputs)
    return use_fast(e, in) && !e->padded ? refresh_problem_major(e, in, mask, pm, s) : SIPOC_OK;
  }
  if (e->fast != nullptr && e->fast->problem_major_inputs && !e->padded && aligned16(in)) {
    *il = LqrIn{};
    *pm = in;
    return SIPOC_OK;
  }
  const double *src[9] = {in.Q, in.M, in.R, in.q, in.r, in.A, in.B, in.c, in.delta};
  for (int i = 0; i < 9; ++i) {
    if ((mask >> i & 1u) == 0) continue;
    const int64_t size = lqr_in_size(e->hs, i);
    if (e->il_in[i] == nullptr) {
      sipoc_error rc = alloc_doubles(e, &e->il_in[i], size);
      if (rc != SIPOC_OK) return rc;
    }
    ProfScope ps(&e->prof, "pack_kernel", s);
    launch_pack(src[i], e->il_in[i], size, e->batch, e->ld, s);
    e->launches += 1;
  }
  *il = LqrIn{e->il_in[0], e->il_in[1], e->il_in[2], e->il_in[3], e->il_in[4],
              e->il_in[5], e->il_in[6], e->il_in[7], e->il_in[8]};
  *pm = LqrIn{};
  return SIPOC_OK;
}

// --- device-path cores (shared by the device and host entry points) --------
// Padded plans: `in` (interleaved, the structure's own variable-dim layout) -> the engine's
// uniform padded arrays; the plan then runs on those and writes padded outputs.
sipoc_error pad_inputs(sipoc_engine *e, LqrIn *in, unsigned mask, cudaStream_t s,
                       LqrIn *pm = nullptr) {
  const int np = e->fast->n, mp = e->fast->m, N = e->hs.N, E = e->hs.E;
  const int64_t sizes[9] = {int64_t(N) * np * np, int64_t(E) * np * mp, int64_t(E) * mp * mp,
                            int64_t(N) * np,      int64_t(E) * mp,      int64_t(E) * np * np,
                            int64_t(E) * np * mp, int64_t(N) * np,      int64_t(N) * np};
  for (int i = 0; i < 9; ++i) {
    if (e->pad_in[i] != nullptr) continue;
    sipoc_error rc = alloc_doubles(e, &e->pad_in[i], sizes[i]);
    if (rc != SIPOC_OK) return rc;
  }
  const LqrIn dst{e->pad_in[0], e->pad_in[1], e->pad_in[2], e->pad_in[3], e->pad_in[4],
                  e->pad_in[5], e->pad_in[6], e->pad_in[7], e->pad_in[8]};
  {
    ProfScope ps(&e->prof, "pad_chain_kernel", s);
    launch_pad_chain(e->dt, *in, dst, np, mp, mask, e->batch, e->ld, s);
  }
  e->launches += 1;
  *in = dst;
  // CTA-per-problem plans read problem-major copies: transposed from the padded arrays
  if (pm != nullptr && e->fast->problem_major_inputs)
    return refresh_problem_major(e, dst, mask, pm, s);
  return SIPOC_OK;
}

sipoc_error padded_outputs(sipoc_engine *e, LqrOut *out) {
  const int np = e->fast->n, mp = e->fast->m, N = e->hs.N, E = e->hs.E;
  const int64_t sizes[3] = {int64_t(N) * np, int64_t(E) * mp, int64_t(N) * np};
  for (int i = 0; i < 3; ++i) {
    if (e->pad_out[i] != nullptr) continue;
    sipoc_error rc = alloc_doubles(e, &e->pad_out[i], sizes[i]);
    if (rc != SIPOC_OK) return rc;
  }
  *out = LqrOut{e->pad_out[0], e->pad_out[1], e->pad_out[2]};
  return SIPOC_OK;
}

void unpad_outputs(sipoc_engine *e, const LqrOut &padded, const LqrOut &out, cudaStream_t s) {
  ProfScope ps(&e->prof, "unpad_chain_kernel", s);
  launch_unpad_chain(e->dt, padded, out, e->fast->n, e->fast->m, e->batch, e->ld, s);
  e->launches += 1;
}

bool native_pm(const sipoc_engine *e, const LqrIn &in, bool layout_pm) {
  return layout_pm && e->fast != nullptr && e->fast->problem_major_inputs && !e->padded &&
         aligned16(in);
}

sipoc_error lqr_factor_core(sipoc_engine *e, const LqrIn &caller_in, int *status, cudaStream_t s,
                            bool layout_pm = false) {
  sipoc_error rc;
  e->kkt_factored = false;  // a new LQR factorization replaces the one a KKT solve would use
  LqrIn in, pm;
  if ((rc = resolve_inputs(e, caller_in, layout_pm, kPmMatrices, &in, &pm, s)) != SIPOC_OK)
    return rc;
  if (native_pm(e, caller_in, layout_pm) || use_fast(e, in)) {
    if ((rc = ensure_fast_store(e)) != SIPOC_OK) return rc;
    if (e->padded && (rc = pad_inputs(e, &in, kPmMatrices, s, &pm)) != SIPOC_OK) return rc;
    FastArgs a{in, pm, LqrOut{}, status, e->fast_store, nullptr, e->batch, e->ld, e->hs.E,
               &e->prof};
    a.tables = &e->dt;
    e->launches += e->fast->factor(a, s);
    e->factored = sipoc_engine::Factored::FAST;
  } else {
    if ((rc = ensure_generic_ws(e)) != SIPOC_OK) return rc;
    {
      ProfScope ps(&e->prof, "generic_lqr_factor_kernel", s);
      launch_generic_lqr_factor(e->dt, in, e->gws, status, e->batch, e->ld, s);
    }
    e->launches += 1;
    e->factored = sipoc_engine::Factored::GENERIC;
  }
  return check_launch(e, "lqr_factor");
}

// matrices_kept: A, B, delta are the arrays the factorization was given (the Newton-KKT
// solve right after its own factor): their problem-major / padded copies are still valid
// and only q, r, c are refreshed.
constexpr unsigned kPmVectors = 0b010011000;  // q r c
sipoc_error lqr_solve_core(sipoc_engine *e, const LqrIn &caller_in, const LqrOut &out,
                           cudaStream_t s, bool layout_pm = false, bool matrices_kept = false) {
  sipoc_error rc;
  if (e->factored == sipoc_engine::Factored::NONE)
    return fail(e, SIPOC_NOT_FACTORED, "solve called before a factor on this handle");
  if (e->factored == sipoc_engine::Factored::FAST && !aligned16(caller_in))
    return fail(e, SIPOC_INVALID_ARGUMENT,
                "solve against a fast-path factorization needs 16-byte aligned arrays");
  if (matrices_kept && !e->kept_copies_are_kkt) matrices_kept = false;  // refresh them
  const unsigned mask = matrices_kept ? kPmVectors : kPmSolve;
  if (!matrices_kept) e->kept_copies_are_kkt = false;
  LqrIn in, pm;
  if ((rc = resolve_inputs(e, caller_in, layout_pm, mask, &in, &pm, s)) != SIPOC_OK) return rc;
  if (e->factored == sipoc_engine::Factored::FAST) {
    if ((rc = ensure_fast_scratch(e)) != SIPOC_OK) return rc;
    LqrOut plan_out = out;
    if (e->padded) {
      if ((rc = pad_inputs(e, &in, mask, s, &pm)) != SIPOC_OK) return rc;
      if ((rc = padded_outputs(e, &plan_out)) != SIPOC_OK) return rc;
    }
    FastArgs a{in, pm, plan_out, nullptr, e->fast_store, e->fast_scratch, e->batch, e->ld,
               e->hs.E, &e->prof};
    a.tables = &e->dt;
    e->launches += e->fast->solve(a, s);
    if (e->padded) unpad_outputs(e, plan_out, out, s);
  } else {
    {
      ProfScope ps(&e->prof, "generic_lqr_solve_kernel", s);
      launch_generic_lqr_solve(e->dt, in, e->gws, out, e->batch, e->ld, s);
    }
    e->launches += 1;
  }
  return check_launch(e, "lqr_solve");
}

sipoc_error ensure_scan_ws(sipoc_engine *e) {
  sipoc_engine::Scan &sc = e->scan;
  if (sc.elems != nullptr) return SIPOC_OK;
  const int n = e->fast->n;
  const int64_t S = sc.S;
  sipoc_error rc;
  auto plain = [&](double **p, int64_t doubles) {
    return dev_alloc(e, reinterpret_cast<void **>(p), static_cast<size_t>(doubles) * sizeof(double));
  };
  if ((rc = plain(&sc.elems, e->batch * S * scan_elem_doubles(n))) != SIPOC_OK) return rc;
  const int64_t G = S / sc.Sg;
  if ((rc = plain(&sc.gelems, e->batch * G * scan_elem_doubles(n))) != SIPOC_OK) return rc;
  if ((rc = plain(&sc.maps, e->batch * (S + G) * scan_map_doubles(n))) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &sc.Vb, (S + 1) * n * n)) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &sc.vb, (S + 1) * n)) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &sc.xb, (S + 1) * n)) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &sc.store, S * e->fast->store_elems(sc.L))) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &sc.scratch, S * e->fast->scratch_elems(sc.L))) != SIPOC_OK) return rc;
  const size_t ints = static_cast<size_t>(S) * e->ld * sizeof(int);
  if ((rc = dev_alloc(e, reinterpret_cast<void **>(&sc.seg_status), ints)) != SIPOC_OK) return rc;
  return dev_alloc(e, reinterpret_cast<void **>(&sc.sweep_status), ints);
}

// Parallel in time: segment elements and boundary data (scan.cu), then the fused sweep +
// rollout of every (problem, segment) tile at once.
sipoc_error lqr_factor_solve_scan(sipoc_engine *e, const LqrIn &in, const LqrOut &out,
                                  int *status, cudaStream_t s) {
  sipoc_error rc;
  if ((rc = ensure_scan_ws(e)) != SIPOC_OK) return rc;
  sipoc_engine::Scan &sc = e->scan;
  const ScanArgs sa{in,       e->fast->n, e->fast->m, sc.L,    sc.S,  sc.Sg, e->batch,      e->ld,
                    sc.elems, sc.gelems,  sc.maps,    sc.Vb,   sc.vb, sc.xb, sc.seg_status, &e->prof};
  const int front = launch_scan_front(sa, s);
  if (front < 0) return fail(e, SIPOC_UNSUPPORTED, "no scan kernels for this shape");
  e->launches += front;
  if ((rc = check_launch(e, "scan front")) != SIPOC_OK) return rc;
  FastArgs a{in, LqrIn{}, out, sc.sweep_status, sc.store, sc.scratch, e->batch, e->ld, sc.L,
             &e->prof};
  e->launches += e->fast->factor_solve_segments(a, sc.Vb, sc.vb, sc.xb, sc.S, s);
  if (status != nullptr) {
    launch_scan_status(sc.sweep_status, sc.seg_status, sc.S, e->batch, e->ld, status, s);
    e->launches += 1;
  }
  // The factorization is kept per segment, not in the layout sipoc_lqr_solve reads.
  e->factored = sipoc_engine::Factored::NONE;
  return check_launch(e, "lqr_factor_solve (parallel in time)");
}

sipoc_error lqr_factor_solve_core(sipoc_engine *e, const LqrIn &caller_in, const LqrOut &out,
                                  int *status, cudaStream_t s, bool layout_pm = false) {
  sipoc_error rc;
  e->kkt_factored = false;
  LqrIn in, pm;
  if (e->scan.enabled && !layout_pm && use_fast(e, caller_in))
    return lqr_factor_solve_scan(e, caller_in, out, status, s);
  if ((rc = resolve_inputs(e, caller_in, layout_pm, kPmAll, &in, &pm, s)) != SIPOC_OK) return rc;
  if (native_pm(e, caller_in, layout_pm) || use_fast(e, in)) {
    if ((rc = ensure_fast_store(e)) != SIPOC_OK) return rc;
    if ((rc = ensure_fast_scratch(e)) != SIPOC_OK) return rc;
    LqrOut plan_out = out;
    if (e->padded) {
      if ((rc = pad_inputs(e, &in, kPmAll, s, &pm)) != SIPOC_OK) return rc;
      if ((rc = padded_outputs(e, &plan_out)) != SIPOC_OK) return rc;
    }
    FastArgs a{in, pm, plan_out, status, e->fast_store, e->fast_scratch, e->batch, e->ld, e->hs.E,
               &e->prof};
    a.tables = &e->dt;
    e->launches += e->fast->factor_solve(a, s);
    if (e->padded) unpad_outputs(e, plan_out, out, s);
    // The backward kernel keeps W, K and G^-1, so later solves may reuse them.
    e->factored = sipoc_engine::Factored::FAST;
    return check_launch(e, "lqr_factor_solve");
  }
  // `in` is interleaved here (the caller's own arrays or their packed copies).
  if ((rc = lqr_factor_core(e, in, status, s)) != SIPOC_OK) return rc;
  return lqr_solve_core(e, in, out, s);
}

bool null_in(const sipoc_lqr_input *in, bool need_matrices, bool need_vectors) {
  if (in == nullptr) return true;
  if (need_matrices && (!in->Q || !in->M || !in->R || !in->A || !in->B || !in->delta))
    return true;
  if (need_vectors && (!in->q || !in->r || !in->c || !in->A || !in->B || !in->delta))
    return true;
  return false;
}

int64_t lqr_in_size(const HostStructure &h, int i) {
  switch (i) {
    case 0: return h.nn_off[h.N];  // Q
    case 1: return h.nm_off[h.E];  // M
    case 2: return h.mm_off[h.E];  // R
    case 3: return h.n_off[h.N];   // q
    case 4: return h.m_off[h.E];   // r
    case 5: return h.a_off[h.E];   // A
    case 6: return h.b_off[h.E];   // B
    case 7: return h.n_off[h.N];   // c
    default: return h.n_off[h.N];  // delta
  }
}

int64_t kkt_model_size(const HostStructure &h, int i) {
  switch (i) {
    case 0: return h.nn_off[h.N];
    case 1: return h.jc_node_off[h.N];
    case 2: return h.jg_node_off[h.N];
    case 3: return h.hxx_edge_off[h.E];
    case 4: return h.nm_off[h.E];
    case 5: return h.mm_off[h.E];
    case 6: return h.a_off[h.E];
    case 7: return h.b_off[h.E];
    case 8: return h.jcx_off[h.E];
    case 9: return h.jcu_off[h.E];
    case 10: return h.jgx_off[h.E];
    default: return h.jgu_off[h.E];
  }
}

// theta blocks (KktThetaModel order): node hxt, jct, jgt, htt; edge hxt, hut, dynt, jct, jgt, htt
int64_t kkt_theta_size(const HostStructure &h, int i) {
  const int64_t p = h.theta_dim;
  switch (i) {
    case 0: return h.n_off[h.N] * p;
    case 1: return h.node_c_off[h.N] * p;
    case 2: return h.node_g_off[h.N] * p;
    case 3: return h.N * p * p;
    case 4: return h.pn_off[h.E] * p;
    case 5: return h.m_off[h.E] * p;
    case 6: return h.cn_off[h.E] * p;
    case 7: return h.edge_c_off[h.E] * p;
    case 8: return h.edge_g_off[h.E] * p;
    default: return h.E * p * p;
  }
}

sipoc_error ensure_stage(sipoc_engine *e, int64_t elems_per_problem) {
  if (e->h_stage_elems >= elems_per_problem) return SIPOC_OK;
  // Never shrinks; the old buffer stays owned by the handle until destroy.
  sipoc_error rc = dev_alloc(e, reinterpret_cast<void **>(&e->h_stage),
                             static_cast<size_t>(std::max<int64_t>(elems_per_problem, 1)) *
                                 static_cast<size_t>(e->ld) * sizeof(double));
  if (rc == SIPOC_OK) e->h_stage_elems = elems_per_problem;
  return rc;
}

// host (problem-major) -> device engine layout
sipoc_error upload(sipoc_engine *e, const double *host, double *dev, int64_t size) {
  if (size == 0) return SIPOC_OK;
  if (host == nullptr) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL host input array");
  SIPOC_CUDA(e, cudaMemcpyAsync(e->h_stage, host,
                                static_cast<size_t>(size) * e->batch * sizeof(double),
                                cudaMemcpyHostToDevice, e->host_stream));
  {
    ProfScope ps(&e->prof, "pack_kernel", e->host_stream);
    launch_pack(e->h_stage, dev, size, e->batch, e->ld, e->host_stream);
  }
  e->launches += 1;
  return check_launch(e, "pack");
}

sipoc_error download(sipoc_engine *e, const double *dev, double *host, int64_t size) {
  if (size == 0) return SIPOC_OK;
  if (host == nullptr) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL host output array");
  {
    ProfScope ps(&e->prof, "unpack_kernel", e->host_stream);
    launch_unpack(dev, e->h_stage, size, e->batch, e->ld, e->host_stream);
  }
  e->launches += 1;
  sipoc_error rc = check_launch(e, "unpack");
  if (rc != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaMemcpyAsync(host, e->h_stage,
                                static_cast<size_t>(size) * e->batch * sizeof(double),
                                cudaMemcpyDeviceToHost, e->host_stream));
  return SIPOC_OK;
}

sipoc_error ensure_host_lqr(sipoc_engine *e) {
  if (e->host_lqr_ready) return SIPOC_OK;
  const HostStructure &h = e->hs;
  sipoc_error rc;
  int64_t biggest = 1;
  // (problem-major plans upload straight into their own input buffers: no interleaved copies)
  const bool pm_path = e->fast != nullptr && e->fast->problem_major_inputs;
  for (int i = 0; i < 9 && !pm_path; ++i) {
    if ((rc = alloc_doubles(e, &e->h_in[i], lqr_in_size(h, i))) != SIPOC_OK) return rc;
    biggest = std::max(biggest, lqr_in_size(h, i));
  }
  const int64_t out_sizes[3] = {h.n_off[h.N], h.m_off[h.E], h.n_off[h.N]};
  for (int i = 0; i < 3; ++i) {
    if ((rc = alloc_doubles(e, &e->h_out[i], out_sizes[i])) != SIPOC_OK) return rc;
    biggest = std::max(biggest, out_sizes[i]);
  }
  if ((rc = ensure_stage(e, biggest)) != SIPOC_OK) return rc;
  if (e->h_status == nullptr) {
    rc = dev_alloc(e, reinterpret_cast<void **>(&e->h_status),
                   static_cast<size_t>(e->ld) * sizeof(int));
    if (rc != SIPOC_OK) return rc;
  }
  e->host_lqr_ready = true;
  return SIPOC_OK;
}

sipoc_error ensure_host_kkt(sipoc_engine *e) {
  if (e->host_kkt_ready) return SIPOC_OK;
  const HostStructure &h = e->hs;
  sipoc_error rc;
  int64_t biggest = std::max<int64_t>(1, h.kkt_dim);
  for (int i = 0; i < 12; ++i) {
    if ((rc = alloc_doubles(e, &e->hk_model[i], kkt_model_size(h, i))) != SIPOC_OK) return rc;
    biggest = std::max(biggest, kkt_model_size(h, i));
  }
  const int64_t reg_sizes[4] = {h.z_dim, h.x_dim, h.y_dim, h.z_dim};
  for (int i = 0; i < 4; ++i)
    if ((rc = alloc_doubles(e, &e->hk_reg[i], reg_sizes[i])) != SIPOC_OK) return rc;
  for (int i = 0; i < 2; ++i)
    if ((rc = alloc_doubles(e, &e->hk_vec[i], h.kkt_dim)) != SIPOC_OK) return rc;
  for (int i = 0; i < 10 && h.theta_dim > 0; ++i) {
    if ((rc = alloc_doubles(e, &e->hk_theta[i], kkt_theta_size(h, i))) != SIPOC_OK) return rc;
    biggest = std::max(biggest, kkt_theta_size(h, i));
  }
  if ((rc = ensure_stage(e, biggest)) != SIPOC_OK) return rc;
  if (e->h_status == nullptr) {
    rc = dev_alloc(e, reinterpret_cast<void **>(&e->h_status),
                   static_cast<size_t>(e->ld) * sizeof(int));
    if (rc != SIPOC_OK) return rc;
  }
  e->host_kkt_ready = true;
  return SIPOC_OK;
}

KktModel to_model(const sipoc_kkt_model *m) {
  return KktModel{m->node_hxx, m->node_jc,  m->node_jg, m->edge_hxx, m->edge_hxu, m->edge_huu,
                  m->edge_A,   m->edge_B,   m->edge_jcx, m->edge_jcu, m->edge_jgx, m->edge_jgu};
}

// Zero-sized blocks may be NULL; the kernels never dereference them.
KktThetaModel to_theta(const sipoc_kkt_model *m) {
  const sipoc_kkt_theta_model *t = m->theta;
  if (t == nullptr) return KktThetaModel{};
  return KktThetaModel{t->node_hxt, t->node_jct, t->node_jgt, t->node_htt, t->edge_hxt,
                       t->edge_hut, t->edge_dynt, t->edge_jct, t->edge_jgt, t->edge_htt};
}

bool theta_has_null(const sipoc_engine *e, const sipoc_kkt_model *m) {
  if (e->hs.theta_dim == 0) return false;
  if (m == nullptr || m->theta == nullptr) return true;
  const sipoc_kkt_theta_model *t = m->theta;
  const double *ptr[10] = {t->node_hxt, t->node_jct, t->node_jgt, t->node_htt, t->edge_hxt,
                           t->edge_hut, t->edge_dynt, t->edge_jct, t->edge_jgt, t->edge_htt};
  for (int i = 0; i < 10; ++i)
    if (ptr[i] == nullptr && kkt_theta_size(e->hs, i) > 0) return true;
  return false;
}

sipoc_error ensure_theta_ws(sipoc_engine *e) {
  if (e->theta_J != nullptr || e->hs.theta_dim == 0) return SIPOC_OK;
  const int64_t p = e->hs.theta_dim, kd = e->hs.kkt_dim;
  sipoc_error rc;
  if ((rc = alloc_doubles(e, &e->theta_KinvJ, kd * p)) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &e->theta_S, p * p)) != SIPOC_OK) return rc;
  if ((rc = alloc_doubles(e, &e->theta_t, p)) != SIPOC_OK) return rc;
  return alloc_doubles(e, &e->theta_J, kd * p);
}

bool model_has_null(const sipoc_kkt_model *m) {
  return m == nullptr || !m->node_hxx || !m->node_jc || !m->node_jg || !m->edge_hxx ||
         !m->edge_hxu || !m->edge_huu || !m->edge_A || !m->edge_B || !m->edge_jcx ||
         !m->edge_jcu || !m->edge_jgx || !m->edge_jgu;
}

sipoc_error kkt_solve_stagewise(sipoc_engine *e, const KktModel &mdl, const double *b,
                                double *sol, cudaStream_t s);

sipoc_error kkt_factor_core(sipoc_engine *e, const KktModel &mdl, const KktThetaModel &tm,
                            const double *w, const double *r1, const double *r2,
                            const double *r3, int *ok, cudaStream_t s) {
  sipoc_error rc;
  if ((rc = ensure_kkt_ws(e)) != SIPOC_OK) return rc;
  if (e->kkt_reduce_fast != nullptr) {
    ProfScope ps(&e->prof, "kkt_reduce_chain", s);
    e->kkt_reduce_fast(e->dt, mdl, w, r1, r2, r3, e->kws, ok, e->batch, e->ld, e->kkt_max_rows,
                       s);
  } else {
    ProfScope ps(&e->prof, "kkt_reduce_kernel", s);
    launch_kkt_reduce(e->dt, mdl, w, r1, r2, r3, e->kws, ok, e->batch, e->ld, s);
  }
  e->launches += 2;
  if ((rc = check_launch(e, "kkt_reduce")) != SIPOC_OK) return rc;
  // helpers.cpp:362-368: LQR on (Q_mod, M_mod, R_mod, ddyn_dx, ddyn_du, dyn_r2).
  LqrIn in{e->kws.Q_mod, e->kws.M_mod, e->kws.R_mod, nullptr, nullptr,
           mdl.edge_A,   mdl.edge_B,   nullptr,      e->kws.dyn_r2};
  if ((rc = lqr_factor_core(e, in, e->kkt_lqr_status, s)) != SIPOC_OK) return rc;
  launch_kkt_finish_factor(e->kkt_lqr_status, ok, e->batch, s);
  e->launches += 1;
  e->kkt_factored = true;
  e->kept_copies_are_kkt = true;
  e->host_lqr_factored = false;  // the factorization sipoc_lqr_solve_host would read is gone
  if ((rc = check_launch(e, "kkt_finish_factor")) != SIPOC_OK) return rc;
  const int p = e->hs.theta_dim;
  if (p == 0) return SIPOC_OK;
  // helpers.cpp:372-407: J, K_s^-1 J column by column against the factorization just kept
  // (the reference's multi-RHS stagewise solve, :422-747), S and its Cholesky factor.
  if ((rc = ensure_theta_ws(e)) != SIPOC_OK) return rc;
  {
    ProfScope ps(&e->prof, "theta_jacobian_kernel", s);
    launch_theta_jacobian(e->dt, tm, e->theta_J, e->batch, e->ld, s);
  }
  e->launches += 1;
  if ((rc = check_launch(e, "theta_jacobian")) != SIPOC_OK) return rc;
  const size_t col = static_cast<size_t>(e->hs.kkt_dim) * e->ld;
  for (int j = 0; j < p; ++j)
    if ((rc = kkt_solve_stagewise(e, mdl, e->theta_J + j * col, e->theta_KinvJ + j * col, s)) !=
        SIPOC_OK)
      return rc;
  {
    ProfScope ps(&e->prof, "theta_schur_kernel", s);
    launch_theta_schur(e->dt, tm, r1, e->theta_J, e->theta_KinvJ, e->theta_S, ok, e->batch, e->ld,
                       s);
  }
  e->launches += 2;
  return check_launch(e, "theta_schur");
}

// CallbackProvider::solve_stagewise_kkt (helpers.cpp:411-413, 749-894): K_s^-1 on the
// stagewise rows of full-layout vectors; theta rows are neither read nor written.
sipoc_error kkt_solve_stagewise(sipoc_engine *e, const KktModel &mdl, const double *b,
                                double *sol, cudaStream_t s) {
  if (!e->kkt_factored)
    return fail(e, SIPOC_NOT_FACTORED, "kkt_solve called before kkt_factor");
  if (e->factored == sipoc_engine::Factored::FAST && !e->padded &&
      e->fast->kkt_solve != nullptr && e->batch >= kFusedKktMinBatch) {
    // Uniform chain: rhs build fused into the affine sweep, dual recovery into the rollout.
    sipoc_error rc = ensure_fast_scratch(e);
    if (rc != SIPOC_OK) return rc;
    FastKktArgs k{&e->dt, &mdl, &e->kws, b, sol, e->fast_store, e->fast_scratch,
                  e->batch, e->ld, e->hs.E, &e->prof};
    e->launches += e->fast->kkt_solve(k, s);
    return check_launch(e, "kkt_solve");
  }
  {
    ProfScope ps(&e->prof, "kkt_build_rhs_kernel", s);
    launch_kkt_build_rhs(e->dt, mdl, e->kws, b, e->batch, e->ld, s);
  }
  e->launches += 1;
  sipoc_error rc = check_launch(e, "kkt_build_rhs");
  if (rc != SIPOC_OK) return rc;
  LqrIn in{e->kws.Q_mod, e->kws.M_mod, e->kws.R_mod, e->kws.q_mod, e->kws.r_mod,
           mdl.edge_A,   mdl.edge_B,   e->kws.c_mod, e->kws.dyn_r2};
  LqrOut out{e->kws.x, e->kws.u, e->kws.y};
  if ((rc = lqr_solve_core(e, in, out, s, false, /*matrices_kept=*/true)) != SIPOC_OK) return rc;
  {
    ProfScope ps(&e->prof, "kkt_recover_kernel", s);
    launch_kkt_recover(e->dt, mdl, e->kws, b, sol, e->batch, e->ld, s);
  }
  e->launches += 1;
  return check_launch(e, "kkt_recover");
}

// CallbackProvider::solve (helpers.cpp:896-951).
sipoc_error kkt_solve_core(sipoc_engine *e, const KktModel &mdl, const double *b, double *sol,
                           cudaStream_t s) {
  sipoc_error rc = kkt_solve_stagewise(e, mdl, b, sol, s);
  if (rc != SIPOC_OK || e->hs.theta_dim == 0) return rc;
  {
    ProfScope ps(&e->prof, "theta_solve_kernels", s);
    launch_theta_solve(e->dt, b, e->theta_J, e->theta_KinvJ, e->theta_S, e->theta_t, sol,
                       e->batch, e->ld, s);
  }
  e->launches += 3;
  return check_launch(e, "theta_solve");
}

// y += K x on full [x | y | z] vectors: the stagewise operator, then the theta terms.
sipoc_error kkt_apply_core(sipoc_engine *e, const KktModel &mdl, const KktThetaModel &tm,
                           const double *w, const double *r1, const double *r2,
                           const double *r3, const double *x, double *y, cudaStream_t s) {
  {
    ProfScope ps(&e->prof, e->kkt_apply_fast != nullptr ? "kkt_apply_chain" : "kkt_apply_kernel", s);
    (e->kkt_apply_fast != nullptr ? e->kkt_apply_fast : &launch_kkt_apply)(
        e->dt, mdl, w, r1, r2, r3, x, y, e->batch, e->ld, s);
  }
  e->launches += 1;
  if (e->hs.theta_dim > 0) {
    const size_t oy = static_cast<size_t>(e->hs.x_dim) * e->ld,
                 oz = oy + static_cast<size_t>(e->hs.y_dim) * e->ld;
    ProfScope ps(&e->prof, "theta_apply_kernel", s);
    launch_theta_apply(e->dt, tm, kKktAll, r1, x, x + oy, x + oz, y, y + oy, y + oz, e->batch,
                       e->ld, s);
    e->launches += 1;
  }
  return check_launch(e, "kkt_apply");
}

}  // namespace

// ===========================================================================
extern "C" {

int sipoc_version(void) { return SIPOC_VERSION; }

sipoc_error sipoc_attach_comm(sipoc_engine *e, sipoc_comm *comm) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  e->comm = comm;
  return SIPOC_OK;
}

// The per-iteration exchange (SURVEY.md 8e): with a communicator attached, every `stats`
// the engine writes is all-reduced over the ranks on the same stream.
static sipoc_error reduce_stats(sipoc_engine *e, double *stats, void *stream) {
  if (e->comm == nullptr || stats == nullptr) return SIPOC_OK;
  const sipoc_error rc = sipoc_comm_allreduce_stats(e->comm, stats, stream);
  if (rc != SIPOC_OK) return fail(e, rc, "all-reduce of the statistics failed");
  e->launches += 1;  // the fold kernel (the all-gather is NCCL's)
  return SIPOC_OK;
}

sipoc_error sipoc_validate(const sipoc_structure *s) {
  if (s == nullptr) return SIPOC_INVALID_ARGUMENT;
  HostStructure hs;
  std::string err;
  return hs.build(*s, err);
}

sipoc_error sipoc_create(const sipoc_structure *s, sipoc_engine **out) {
  if (out == nullptr) return SIPOC_INVALID_ARGUMENT;
  *out = nullptr;
  if (s == nullptr || s->batch <= 0) return SIPOC_INVALID_ARGUMENT;
  sipoc_engine *e = new (std::nothrow) sipoc_engine();
  if (e == nullptr) return SIPOC_OUT_OF_MEMORY;
  std::string err;
  sipoc_error rc = e->hs.build(*s, err);
  if (rc != SIPOC_OK) {
    delete e;
    return rc;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    // No CPU fallback by design.
    delete e;
    return SIPOC_CUDA_ERROR;
  }
  int dev = s->device;
  if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess) {
    delete e;
    return SIPOC_CUDA_ERROR;
  }
  if (dev >= ndev) {
    delete e;
    return SIPOC_INVALID_ARGUMENT;
  }
  e->device = dev;
  e->flags = s->flags;
  e->batch = s->batch;
  e->ld = (s->batch + 31) / 32 * 32;
  DeviceGuard guard(dev);

  DevTables t{};
  std::vector<int> buf = e->hs.serialise(t);
  void *d = nullptr;
  if (cudaMalloc(&d, buf.size() * sizeof(int)) != cudaSuccess ||
      cudaMemcpy(d, buf.data(), buf.size() * sizeof(int), cudaMemcpyHostToDevice) !=
          cudaSuccess ||
      cudaStreamCreateWithFlags(&e->host_stream, cudaStreamNonBlocking) != cudaSuccess) {
    if (d != nullptr) cudaFree(d);
    delete e;
    return SIPOC_CUDA_ERROR;
  }
  e->d_tab = static_cast<int *>(d);
  e->allocations.push_back(d);
  rebase(t, e->d_tab);
  e->dt = t;

  const HostStructure &h = e->hs;
  if (!(e->flags & SIPOC_FLAG_FORCE_GENERIC) && h.is_chain && h.is_uniform && h.E >= 1)
    e->fast = select_fast_plan(h.n[0], h.m[0]);
  if (e->fast == nullptr && !(e->flags & SIPOC_FLAG_FORCE_GENERIC) && h.is_chain &&
      h.is_uniform && h.E >= 1)
    e->fast = select_cta_plan(h.n[0], h.m[0]);
  if (e->fast == nullptr && !(e->flags & SIPOC_FLAG_FORCE_GENERIC) &&
      !(e->flags & SIPOC_FLAG_PAD_VARIABLE_DIMS) && h.is_chain && h.E >= 1 &&
      (e->fast = select_strict_plan(h.max_n, h.max_m)) != nullptr) {
    // Small chains without a plan of their own (dims that change from stage to stage, or a
    // uniform shape that is not instantiated): the reference-order register kernels on the
    // chain padded to the smallest shape that holds every stage -- the generic kernels'
    // operations in the same order on the real entries (riccati_strict.cu).
    e->padded = true;
  }
  if (e->fast == nullptr && !(e->flags & SIPOC_FLAG_FORCE_GENERIC) && !h.is_chain && h.E >= 1 &&
      (e->fast = select_strict_tree_plan(h.max_n, h.max_m)) != nullptr) {
    // Small trees: the same reference-order register kernels, walking the tree.
    e->padded = true;
  }
  if (e->fast == nullptr && !(e->flags & SIPOC_FLAG_FORCE_GENERIC) &&
      (e->flags & SIPOC_FLAG_PAD_VARIABLE_DIMS) && h.is_chain && !h.is_uniform && h.E >= 1) {
    // smallest instantiated register / sub-warp shape that holds every stage
    const int shapes[][2] = {{4, 1}, {6, 2}, {8, 3}, {12, 4}};
    for (const auto &sh : shapes) {
      if (sh[0] >= h.max_n && sh[1] >= h.max_m && (e->fast = select_fast_plan(sh[0], sh[1]))) {
        e->padded = true;
        break;
      }
    }
  }
  if (e->fast == nullptr && !(e->flags & SIPOC_FLAG_FORCE_GENERIC) && h.is_chain &&
      h.is_uniform && h.E >= 1) {
    // A uniform shape that is not instantiated (e.g. n = 16 with m < 4 of the reference
    // grid, lqr_benchmark.cpp:537-545): padded up to the next shape that is, sub-warp shapes
    // first, then the CTA-per-problem ones.
    const int shapes[][2] = {{6, 1}, {6, 2}, {6, 3}, {6, 4}, {8, 1}, {8, 2}, {8, 3}, {8, 4}, {12, 4}};
    for (const auto &sh : shapes)
      if (sh[0] >= h.max_n && sh[1] >= h.max_m && (e->fast = select_fast_plan(sh[0], sh[1])))
        break;
    const int cta_shapes[][2] = {{16, 4}, {32, 8}, {64, 24}};
    for (const auto &sh : cta_shapes)
      if (e->fast == nullptr && sh[0] >= h.max_n && sh[1] >= h.max_m)
        e->fast = select_cta_plan(sh[0], sh[1]);
    e->padded = e->fast != nullptr;
  }
  if (!(e->flags & SIPOC_FLAG_FORCE_GENERIC) && h.is_chain && h.is_uniform && h.E >= 1) {
    e->kkt_reduce_fast = select_kkt_reduce(h.n[0], h.m[0]);
    e->kkt_apply_fast = select_kkt_apply(h.n[0], h.m[0]);
    for (int i = 0; i < h.N; ++i) {
      int rows = h.node_c[i] + h.node_g[i];
      if (i < h.E) rows += h.edge_c[i] + h.edge_g[i];
      e->kkt_max_rows = std::max(e->kkt_max_rows, rows);
    }
    if (kkt_reduce_smem_bytes(h.n[0], h.m[0], std::max(1, e->kkt_max_rows)) > 200 * 1024)
      e->kkt_reduce_fast = nullptr;
  }
  if (e->fast != nullptr && !e->padded && e->fast->factor_solve_segments != nullptr &&
      !(e->flags & SIPOC_FLAG_SERIAL_IN_TIME) && scan_supports(e->fast->n, e->fast->m)) {
    // Parallel in time pays when the serial sweep cannot fill the GPU: a long horizon and a
    // batch far below one wave of tiles.  The segment length is the divisor of the horizon
    // nearest 32 (measured best at N = 4 096: 16 -> 2.29, 32 -> 1.96, 64 -> 2.14 ms); SIPOC_SCAN_SEGMENT overrides it.
    const bool wanted = (e->flags & SIPOC_FLAG_PARALLEL_IN_TIME) != 0 ||
                        (h.E >= 512 && e->batch <= 512);
    int target = 32;
    if (const char *env = getenv("SIPOC_SCAN_SEGMENT")) target = std::max(1, atoi(env));
    int best = 0;
    for (int L = 2; L <= h.E / 2; ++L)
      if (h.E % L == 0 && (best == 0 || std::abs(L - target) < std::abs(best - target))) best = L;
    if (wanted && best >= 2) {
      e->scan.enabled = true;
      e->scan.L = best;
      e->scan.S = h.E / best;
      e->scan.Sg = scan_group_size(e->scan.S);
      if (const char *env = getenv("SIPOC_SCAN_GROUP"))
        if (atoi(env) >= 1 && e->scan.S % atoi(env) == 0) e->scan.Sg = atoi(env);
    }
  }
  e->variant = e->fast != nullptr ? e->fast->name : "generic_thread_per_problem";
  if (e->scan.enabled) e->variant = "scan_" + e->variant;
  if (e->padded) e->variant = "padded_to_" + e->variant;
  *out = e;
  return SIPOC_OK;
}

void invalidate_graph(struct sipoc_graph *g);  // below, with the graph type

void sipoc_destroy(sipoc_engine *e) {
  if (e == nullptr) return;
  {
    DeviceGuard guard(e->device);
    cudaDeviceSynchronize();
    for (sipoc_graph *g : e->graphs) invalidate_graph(g);
    for (void *p : e->allocations) cudaFree(p);
    if (e->host_stream != nullptr) cudaStreamDestroy(e->host_stream);
  }
  delete e;
}

const char *sipoc_last_error(const sipoc_engine *e) {
  return e == nullptr ? "" : e->last_error.c_str();
}

const char *sipoc_kernel_variant(const sipoc_engine *e) {
  return e == nullptr ? "" : e->variant.c_str();
}

int64_t sipoc_launch_count(const sipoc_engine *e) { return e == nullptr ? 0 : e->launches; }

// ---- CUDA graphs ------------------------------------------------------------
// The device entry points only enqueue work on the caller's stream (workspaces are
// sized on first use, so one eager pass precedes a capture); any sequence of them can
// therefore be recorded once and relaunched with a single driver call.
struct sipoc_graph {
  cudaGraphExec_t exec = nullptr;
  int device = 0;
  int64_t launches = 0;  // engine kernels inside one launch of the graph
  // The kernels of the graph point into this handle's workspaces: sipoc_destroy(owner)
  // invalidates the graph (exec destroyed, owner cleared) instead of leaving it dangling.
  sipoc_engine *owner = nullptr;
};

void invalidate_graph(sipoc_graph *g) {  // its engine is going away
  if (g->exec != nullptr) cudaGraphExecDestroy(g->exec);
  g->exec = nullptr;
  g->owner = nullptr;
}

sipoc_error sipoc_graph_begin(sipoc_engine *e, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (e->capturing) return fail(e, SIPOC_INVALID_ARGUMENT, "sipoc_graph_begin: already capturing");
  if (e->prof.enabled())
    return fail(e, SIPOC_INVALID_ARGUMENT,
                "sipoc_graph_begin: per-kernel profiling records events; disable it first");
  DeviceGuard guard(e->device);
  SIPOC_CUDA(e, cudaStreamBeginCapture(static_cast<cudaStream_t>(stream),
                                       cudaStreamCaptureModeThreadLocal));
  e->capturing = true;
  e->capture_launches0 = e->launches;
  e->capture_saved = {static_cast<int>(e->factored), e->kkt_factored, e->host_lqr_factored};
  return SIPOC_OK;
}

sipoc_error sipoc_graph_end(sipoc_engine *e, void *stream, sipoc_graph **out) {
  if (e == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  *out = nullptr;
  if (!e->capturing) return fail(e, SIPOC_INVALID_ARGUMENT, "sipoc_graph_end: not capturing");
  DeviceGuard guard(e->device);
  e->capturing = false;
  e->factored = static_cast<sipoc_engine::Factored>(e->capture_saved.factored);
  e->kkt_factored = e->capture_saved.kkt_factored;
  e->host_lqr_factored = e->capture_saved.host_lqr_factored;
  cudaGraph_t graph = nullptr;
  SIPOC_CUDA(e, cudaStreamEndCapture(static_cast<cudaStream_t>(stream), &graph));
  cudaGraphExec_t exec = nullptr;
  cudaError_t err = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (err != cudaSuccess)
    return fail(e, SIPOC_CUDA_ERROR,
                std::string("cudaGraphInstantiate: ") + cudaGetErrorString(err));
  sipoc_graph *g = new sipoc_graph;
  g->exec = exec;
  g->device = e->device;
  g->launches = e->launches - e->capture_launches0;
  g->owner = e;
  e->graphs.push_back(g);
  *out = g;
  return SIPOC_OK;
}

sipoc_error sipoc_graph_launch(sipoc_engine *e, sipoc_graph *g, void *stream) {
  if (e == nullptr || g == nullptr || g->exec == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (g->owner != e)
    return fail(e, SIPOC_INVALID_ARGUMENT, "sipoc_graph_launch: graph recorded on another handle");
  DeviceGuard guard(e->device);
  SIPOC_CUDA(e, cudaGraphLaunch(g->exec, static_cast<cudaStream_t>(stream)));
  e->launches += g->launches;
  return SIPOC_OK;
}

int64_t sipoc_graph_kernel_count(const sipoc_graph *g) { return g == nullptr ? 0 : g->launches; }

void sipoc_graph_destroy(sipoc_graph *g) {
  if (g == nullptr) return;
  if (g->owner != nullptr) {
    auto &live = g->owner->graphs;
    live.erase(std::remove(live.begin(), live.end(), g), live.end());
  }
  if (g->exec != nullptr) {
    DeviceGuard guard(g->device);
    cudaGraphExecDestroy(g->exec);
  }
  delete g;
}

sipoc_error sipoc_profile_enable(sipoc_engine *e, int on) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  e->prof.reset();
  e->prof.enable(on != 0);
  return SIPOC_OK;
}

int sipoc_profile_collect(sipoc_engine *e) {
  if (e == nullptr) return 0;
  DeviceGuard guard(e->device);
  return static_cast<int>(e->prof.summarise().size());
}

sipoc_error sipoc_profile_get(const sipoc_engine *e, int index, const char **name,
                              double *total_ms, int64_t *launches) {
  if (e == nullptr || index < 0 || index >= static_cast<int>(e->prof.summary().size()))
    return SIPOC_INVALID_ARGUMENT;
  const Profiler::Summary &s = e->prof.summary()[index];
  if (name) *name = s.name.c_str();
  if (total_ms) *total_ms = s.total_ms;
  if (launches) *launches = s.launches;
  return SIPOC_OK;
}
int64_t sipoc_batch(const sipoc_engine *e) { return e == nullptr ? 0 : e->batch; }
int64_t sipoc_batch_stride(const sipoc_engine *e) { return e == nullptr ? 0 : e->ld; }

sipoc_error sipoc_get_topology(const sipoc_engine *e, int *child_offsets, int *child_edges,
                               int *preorder, int *postorder) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  const HostStructure &h = e->hs;
  if (child_offsets) {
    std::copy(h.child_offsets.begin(), h.child_offsets.end(), child_offsets);
  }
  if (child_edges) std::copy(h.child_edges.begin(), h.child_edges.end(), child_edges);
  if (preorder) std::copy(h.preorder.begin(), h.preorder.end(), preorder);
  if (postorder) std::copy(h.postorder.begin(), h.postorder.end(), postorder);
  return SIPOC_OK;
}

sipoc_error sipoc_lqr_get_sizes(const sipoc_engine *e, sipoc_lqr_sizes *o) {
  if (e == nullptr || o == nullptr) return SIPOC_INVALID_ARGUMENT;
  const HostStructure &h = e->hs;
  o->Q = h.nn_off[h.N];
  o->M = h.nm_off[h.E];
  o->R = h.mm_off[h.E];
  o->q = o->c = o->delta = o->x = o->y = h.n_off[h.N];
  o->r = o->u = h.m_off[h.E];
  o->A = h.a_off[h.E];
  o->B = h.b_off[h.E];
  return SIPOC_OK;
}

sipoc_error sipoc_lqr_factor(sipoc_engine *e, const sipoc_lqr_input *in, int *status,
                             void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, false)) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input");
  DeviceGuard guard(e->device);
  return lqr_factor_core(e, to_in(in), status, static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_lqr_solve(sipoc_engine *e, const sipoc_lqr_input *in,
                            const sipoc_lqr_output *out, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, false, true) || out == nullptr || !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output");
  DeviceGuard guard(e->device);
  return lqr_solve_core(e, to_in(in), LqrOut{out->x, out->u, out->y},
                        static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_lqr_factor_solve(sipoc_engine *e, const sipoc_lqr_input *in,
                                   const sipoc_lqr_output *out, int *status, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, true) || out == nullptr || !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output");
  DeviceGuard guard(e->device);
  return lqr_factor_solve_core(e, to_in(in), LqrOut{out->x, out->u, out->y}, status,
                               static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_lqr_factor_pm(sipoc_engine *e, const sipoc_lqr_input *in, int *status,
                                void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, false)) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input");
  DeviceGuard guard(e->device);
  return lqr_factor_core(e, to_in(in), status, static_cast<cudaStream_t>(stream), true);
}

sipoc_error sipoc_lqr_solve_pm(sipoc_engine *e, const sipoc_lqr_input *in,
                               const sipoc_lqr_output *out, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, false, true) || out == nullptr || !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output");
  DeviceGuard guard(e->device);
  return lqr_solve_core(e, to_in(in), LqrOut{out->x, out->u, out->y},
                        static_cast<cudaStream_t>(stream), true);
}

sipoc_error sipoc_lqr_factor_solve_pm(sipoc_engine *e, const sipoc_lqr_input *in,
                                      const sipoc_lqr_output *out, int *status, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, true) || out == nullptr || !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output");
  DeviceGuard guard(e->device);
  return lqr_factor_solve_core(e, to_in(in), LqrOut{out->x, out->u, out->y}, status,
                               static_cast<cudaStream_t>(stream), true);
}

sipoc_error sipoc_lqr_residual(sipoc_engine *e, const sipoc_lqr_input *in,
                               const sipoc_lqr_output *out, const int *status,
                               double *residual_norm, double *stats, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, true) || out == nullptr || !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output");
  DeviceGuard guard(e->device);
  {
    ProfScope ps(&e->prof, "lqr_residual_kernel", static_cast<cudaStream_t>(stream));
    launch_lqr_residual(e->dt, to_in(in), LqrOut{out->x, out->u, out->y}, status,
                        residual_norm, stats, e->batch, e->ld,
                        static_cast<cudaStream_t>(stream));
  }
  e->launches += stats != nullptr ? 2 : 1;
  sipoc_error rc = check_launch(e, "lqr_residual");
  return rc != SIPOC_OK ? rc : reduce_stats(e, stats, stream);
}

// The per-problem flags of a VJP / JVP call whose caller passes none: an engine-owned buffer.
static sipoc_error default_vjp_status(sipoc_engine *e, int **status) {
  if (*status != nullptr) return SIPOC_OK;
  if (e->vjp_status == nullptr) {
    const sipoc_error rc = dev_alloc(e, reinterpret_cast<void **>(&e->vjp_status),
                                     static_cast<size_t>(e->ld) * sizeof(int));
    if (rc != SIPOC_OK) return rc;
  }
  *status = e->vjp_status;
  return SIPOC_OK;
}

sipoc_error sipoc_lqr_vjp(sipoc_engine *e, const sipoc_lqr_input *in,
                          const sipoc_lqr_output *sol, const sipoc_lqr_cotangent *cot,
                          const sipoc_lqr_output *adjoint, const sipoc_lqr_grad *grad,
                          int *status, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, false) || sol == nullptr || !sol->x || !sol->u || !sol->y ||
      cot == nullptr || !cot->x || !cot->u || !cot->y || adjoint == nullptr || !adjoint->x ||
      !adjoint->u || !adjoint->y || grad == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / solution / cotangent / adjoint / grad");
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if ((rc = default_vjp_status(e, &status)) != SIPOC_OK) return rc;
  // K is symmetric: the adjoint is the same LQR with the cotangent as (q, r, c).
  const LqrIn adj_in{in->Q, in->M, in->R, cot->x, cot->u, in->A, in->B, cot->y, in->delta};
  const LqrOut adj{adjoint->x, adjoint->u, adjoint->y};
  if ((rc = lqr_factor_solve_core(e, adj_in, adj, status, s)) != SIPOC_OK) return rc;
  const LqrGrad g{grad->Q, grad->M, grad->R, grad->q, grad->r, grad->A, grad->B, grad->c,
                  grad->delta};
  if (!g.Q && !g.M && !g.R && !g.q && !g.r && !g.A && !g.B && !g.c && !g.delta) return SIPOC_OK;
  {
    ProfScope ps(&e->prof, "lqr_vjp_kernel", s);
    launch_lqr_vjp(e->dt, LqrOut{sol->x, sol->u, sol->y}, adj, status, g, e->batch, e->ld, s);
  }
  e->launches += 1;
  return check_launch(e, "lqr_vjp");
}

sipoc_error sipoc_lqr_jvp(sipoc_engine *e, const sipoc_lqr_input *in,
                          const sipoc_lqr_output *sol, const sipoc_lqr_input *tangent,
                          const sipoc_lqr_output *rhs, const sipoc_lqr_output *dsol,
                          int *status, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, false) || sol == nullptr || !sol->x || !sol->u || !sol->y ||
      tangent == nullptr || rhs == nullptr || !rhs->x || !rhs->u || !rhs->y || dsol == nullptr ||
      !dsol->x || !dsol->u || !dsol->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / solution / tangent / rhs / dsol");
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if ((rc = default_vjp_status(e, &status)) != SIPOC_OK) return rc;
  const LqrOut t{rhs->x, rhs->u, rhs->y}, d{dsol->x, dsol->u, dsol->y};
  {
    ProfScope ps(&e->prof, "lqr_jvp_kernel", s);
    launch_lqr_jvp(e->dt, LqrOut{sol->x, sol->u, sol->y},
                   LqrTangent{tangent->Q, tangent->M, tangent->R, tangent->q, tangent->r,
                              tangent->A, tangent->B, tangent->c, tangent->delta},
                   t, e->batch, e->ld, s);
  }
  e->launches += 1;
  if ((rc = check_launch(e, "lqr_jvp")) != SIPOC_OK) return rc;
  // The tangent is the same LQR with t as (q, r, c).
  const LqrIn tan_in{in->Q, in->M, in->R, t.x, t.u, in->A, in->B, t.y, in->delta};
  if ((rc = lqr_factor_solve_core(e, tan_in, d, status, s)) != SIPOC_OK) return rc;
  {
    ProfScope ps(&e->prof, "jvp_zero_dead_lanes", s);
    const HostStructure &h = e->hs;
    launch_zero_dead_lanes(d.x, h.n_off[h.N], status, false, e->batch, e->ld, s);
    launch_zero_dead_lanes(d.u, h.m_off[h.E], status, false, e->batch, e->ld, s);
    launch_zero_dead_lanes(d.y, h.n_off[h.N], status, false, e->batch, e->ld, s);
  }
  e->launches += 3;
  return check_launch(e, "lqr_jvp zero pass");
}

// The policy of the factor + solve that has just run (policy.cuh).  `scan`: it ran parallel
// in time, on the per-segment stores.  Generic and strict plans keep V; the others keep
// F^-1, from which V is rebuilt; padded plans are exported in their own shape and the
// leading blocks extracted.
static sipoc_error lqr_policy_export(sipoc_engine *e, const LqrIn &caller_in, const LqrPolicy &pol,
                                     const int *status, bool scan, cudaStream_t s) {
  const HostStructure &h = e->hs;
  auto gather = [&](PolicyArray which, const PolicySrc &src, double *dst) {
    if (dst == nullptr) return;
    ProfScope ps(&e->prof, "policy_gather_kernel", s);
    launch_policy_gather(e->dt, which, src, dst, status, e->batch, e->ld, s);
    e->launches += 1;
  };
  if (!scan && e->factored == sipoc_engine::Factored::GENERIC) {
    PolicySrc src;
    src.same_as_out = true;
    src.p = e->gws.K;
    gather(PolicyArray::K, src, pol.K);
    src.p = e->gws.k;
    gather(PolicyArray::k, src, pol.k);
    src.p = e->gws.V;
    gather(PolicyArray::V, src, pol.V);
    src.p = e->gws.v;
    gather(PolicyArray::v, src, pol.v);
    return check_launch(e, "lqr policy export");
  }
  const FastPlan *plan = e->fast;
  const int n = plan->n, m = plan->m;
  const bool strict = plan == select_strict_plan(n, m) || plan == select_strict_tree_plan(n, m);
  const PolicyStore kind = plan->problem_major_inputs ? PolicyStore::CTA
                           : strict                   ? PolicyStore::STRICT
                                                      : PolicyStore::FAST;
  const int T = scan ? e->scan.L : h.E;
  PolicySources src = policy_sources(kind, n, m, T, scan ? e->scan.store : e->fast_store,
                                     scan ? e->scan.scratch : e->fast_scratch);
  if (scan) {
    for (PolicySrc *p : {&src.K, &src.k, &src.v, &src.V_or_P}) {
      p->seg_len = e->scan.L;
      p->segs = e->scan.S;
    }
    src.K.seg_stride = src.V_or_P.seg_stride = plan->store_elems(T);
    src.k.seg_stride = src.v.seg_stride = plan->scratch_elems(T);
  }
  gather(PolicyArray::K, src.K, pol.K);
  gather(PolicyArray::k, src.k, pol.k);
  gather(PolicyArray::v, src.v, pol.v);
  if (pol.V != nullptr && kind == PolicyStore::STRICT) {
    gather(PolicyArray::V, src.V_or_P, pol.V);
  } else if (pol.V != nullptr) {
    // the arrays the plan ran on: its padded copies on padded plans
    const LqrIn in = e->padded ? LqrIn{e->pad_in[0], e->pad_in[1], e->pad_in[2],
                                       e->pad_in[3], e->pad_in[4], e->pad_in[5],
                                       e->pad_in[6], e->pad_in[7], e->pad_in[8]}
                               : caller_in;
    double *V = pol.V;
    if (e->padded) {
      if (e->policy_V == nullptr) {
        const sipoc_error rc = alloc_doubles(e, &e->policy_V, int64_t(h.E + 1) * n * n);
        if (rc != SIPOC_OK) return rc;
      }
      V = e->policy_V;
    }
    bool ok;
    {
      ProfScope ps(&e->prof, "policy_rebuild_v_kernel", s);
      ok = launch_policy_rebuild_v(n, m, in, src.V_or_P, src.K, V, status, h.E, e->batch, e->ld, s);
    }
    if (!ok) return fail(e, SIPOC_UNSUPPORTED, "no V rebuild kernel for the plan's shape");
    e->launches += 1;
    if (e->padded) {
      PolicySrc pad;
      pad.p = e->policy_V;
      pad.rows = n;
      pad.block = int64_t(n) * n;
      gather(PolicyArray::V, pad, pol.V);
    }
  }
  return check_launch(e, "lqr policy export");
}

sipoc_error sipoc_lqr_factor_solve_policy(sipoc_engine *e, const sipoc_lqr_input *in,
                                          const sipoc_lqr_output *out,
                                          const sipoc_lqr_policy *policy, int *status,
                                          void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (null_in(in, true, true) || out == nullptr || !out->x || !out->u || !out->y ||
      policy == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL LQR input / output / policy");
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if ((rc = default_vjp_status(e, &status)) != SIPOC_OK) return rc;
  const LqrIn cin = to_in(in);
  const bool scan = e->scan.enabled && use_fast(e, cin);  // the branch lqr_factor_solve_core takes
  if ((rc = lqr_factor_solve_core(e, cin, LqrOut{out->x, out->u, out->y}, status, s)) != SIPOC_OK)
    return rc;
  const LqrPolicy pol{policy->K, policy->k, policy->V, policy->v};
  if (!pol.K && !pol.k && !pol.V && !pol.v) return SIPOC_OK;
  return lqr_policy_export(e, cin, pol, status, scan, s);
}

// Reverse mode of the policy (policy_vjp.cuh): the adjoint Riccati sweep, root to leaves.
// Uniform chains at the shapes of the thread and four-lane plans run the shape-specialised
// kernel, every other structure the generic one; the choice depends on the structure only.
sipoc_error sipoc_lqr_policy_vjp(sipoc_engine *e, const sipoc_lqr_input *in, const double *V,
                                 const double *v, const int *status,
                                 const sipoc_lqr_policy_cotangent *cot,
                                 const sipoc_lqr_grad *grad, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (in == nullptr || !in->M || !in->R || !in->r || !in->A || !in->B || !in->c || !in->delta ||
      V == nullptr || v == nullptr || status == nullptr || cot == nullptr || grad == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT,
                "NULL LQR input / policy V, v / status / cotangent / grad");
  const LqrGrad g{grad->Q, grad->M, grad->R, grad->q, grad->r, grad->A, grad->B, grad->c,
                  grad->delta};
  if (!g.Q && !g.M && !g.R && !g.q && !g.r && !g.A && !g.B && !g.c && !g.delta) return SIPOC_OK;
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const HostStructure &h = e->hs;
  const PolicyVjpIn pin{to_in(in), V, v};
  const LqrPolicyCot pc{cot->K, cot->k, cot->V, cot->v};
  if (h.is_chain && h.is_uniform && h.E >= 1 && policy_vjp_chain_shape(h.n[0], h.m[0])) {
    ProfScope ps(&e->prof, "policy_vjp_kernel", s);
    launch_policy_vjp_chain(h.n[0], h.m[0], h.E, pin, pc, g, status, e->batch, e->ld, s);
  } else {
    if (e->policy_vjp_ws == nullptr) {
      const sipoc_error rc =
          alloc_doubles(e, &e->policy_vjp_ws,
                        policy_vjp_scratch_elems(h.max_n, h.max_m) + h.nn_off[h.N] + h.n_off[h.N]);
      if (rc != SIPOC_OK) return rc;
    }
    ProfScope ps(&e->prof, "policy_vjp_generic_kernel", s);
    launch_policy_vjp_generic(e->dt, h, pin, pc, g, e->policy_vjp_ws, status, e->batch, e->ld, s);
  }
  e->launches += 1;
  return check_launch(e, "lqr policy vjp");
}

// Forward mode of the policy (policy_jvp.cuh): the tangent Riccati sweep, leaves to root.
// Uniform chains at the shapes of the thread and four-lane plans run the sub-warp kernel,
// every other structure the generic one; the choice depends on the structure only.
sipoc_error sipoc_lqr_policy_jvp(sipoc_engine *e, const sipoc_lqr_input *in, const double *V,
                                 const double *v, const int *status,
                                 const sipoc_lqr_input *tangent, const sipoc_lqr_policy *dpolicy,
                                 void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (in == nullptr || !in->M || !in->R || !in->r || !in->A || !in->B || !in->c || !in->delta ||
      V == nullptr || v == nullptr || status == nullptr || tangent == nullptr ||
      dpolicy == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT,
                "NULL LQR input / policy V, v / status / tangent / dpolicy");
  const LqrPolicy out{dpolicy->K, dpolicy->k, dpolicy->V, dpolicy->v};
  if (!out.K && !out.k && !out.V && !out.v) return SIPOC_OK;
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const HostStructure &h = e->hs;
  const PolicyVjpIn pin{to_in(in), V, v};
  const LqrIn tan = to_in(tangent);
  if (h.is_chain && h.is_uniform && h.E >= 1 && policy_jvp_subwarp_shape(h.n[0], h.m[0])) {
    bool ok;
    {
      ProfScope ps(&e->prof, "policy_jvp_subwarp", s);
      ok = launch_policy_jvp_subwarp(h.n[0], h.m[0], h.E, pin, tan, out, status, e->batch, e->ld,
                                     s);
    }
    if (!ok) return fail(e, SIPOC_CUDA_ERROR, "policy JVP: sub-warp kernel not configured");
  } else {
    if (e->policy_jvp_ws == nullptr) {
      const sipoc_error rc = alloc_doubles(e, &e->policy_jvp_ws, policy_jvp_generic_ws_elems(h));
      if (rc != SIPOC_OK) return rc;
    }
    ProfScope ps(&e->prof, "policy_jvp_generic_kernel", s);
    launch_policy_jvp_generic(e->dt, h, pin, tan, out, e->policy_jvp_ws, status, e->batch, e->ld,
                              s);
  }
  e->launches += 1;
  return check_launch(e, "lqr policy jvp");
}

sipoc_error sipoc_status_stats(sipoc_engine *e, const int *status, double *stats,
                               void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (status == nullptr || stats == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL status / stats");
  DeviceGuard guard(e->device);
  {
    ProfScope ps(&e->prof, "status_stats_kernel", static_cast<cudaStream_t>(stream));
    launch_status_stats(status, stats, e->batch, static_cast<cudaStream_t>(stream));
  }
  e->launches += 2;
  sipoc_error rc = check_launch(e, "status_stats");
  return rc != SIPOC_OK ? rc : reduce_stats(e, stats, stream);
}

sipoc_error sipoc_pack(sipoc_engine *e, const double *src, double *dst, int64_t size,
                       void *stream) {
  if (e == nullptr || src == nullptr || dst == nullptr || size < 0)
    return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  launch_pack(src, dst, size, e->batch, e->ld, static_cast<cudaStream_t>(stream));
  e->launches += 1;
  return check_launch(e, "pack");
}

sipoc_error sipoc_unpack(sipoc_engine *e, const double *src, double *dst, int64_t size,
                         void *stream) {
  if (e == nullptr || src == nullptr || dst == nullptr || size < 0)
    return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  launch_unpack(src, dst, size, e->batch, e->ld, static_cast<cudaStream_t>(stream));
  e->launches += 1;
  return check_launch(e, "unpack");
}

// ---- host-buffer LQR --------------------------------------------------------
// Plans that read problem-major inputs take the host arrays as they are: one H2D copy
// per array straight into the engine's problem-major buffers, no pack, no unpack.
static bool host_path_is_pm(const sipoc_engine *e) {
  return e->fast != nullptr && e->fast->problem_major_inputs;
}

static sipoc_error host_upload_lqr(sipoc_engine *e, const sipoc_lqr_input *in,
                                   bool matrices, bool vectors) {
  const double *src[9] = {in->Q, in->M, in->R, in->q, in->r, in->A, in->B, in->c, in->delta};
  const bool is_vec[9] = {false, false, false, true, true, false, false, true, false};
  for (int i = 0; i < 9; ++i) {
    if ((is_vec[i] && !vectors) || (!is_vec[i] && !matrices)) continue;
    const int64_t size = lqr_in_size(e->hs, i);
    if (host_path_is_pm(e)) {
      if (size == 0) continue;
      if (src[i] == nullptr) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL host input array");
      if (e->pm_in[i] == nullptr) {
        sipoc_error rc = dev_alloc(e, reinterpret_cast<void **>(&e->pm_in[i]),
                                   static_cast<size_t>(size) * static_cast<size_t>(e->batch) *
                                       sizeof(double));
        if (rc != SIPOC_OK) return rc;
      }
      SIPOC_CUDA(e, cudaMemcpyAsync(e->pm_in[i], src[i],
                                    static_cast<size_t>(size) * e->batch * sizeof(double),
                                    cudaMemcpyHostToDevice, e->host_stream));
      continue;
    }
    sipoc_error rc = upload(e, src[i], e->h_in[i], size);
    if (rc != SIPOC_OK) return rc;
  }
  return SIPOC_OK;
}

static LqrIn host_resident_in(const sipoc_engine *e) {
  double *const *a = host_path_is_pm(e) ? e->pm_in : e->h_in;
  return LqrIn{a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8]};
}

static sipoc_error host_download_out(sipoc_engine *e, const sipoc_lqr_output *out) {
  const HostStructure &h = e->hs;
  sipoc_error rc;
  if ((rc = download(e, e->h_out[0], out->x, h.n_off[h.N])) != SIPOC_OK) return rc;
  // The staging buffer is reused: order copies on the stream (same stream, so
  // the unpack of the next array waits for the previous D2H).
  if ((rc = download(e, e->h_out[1], out->u, h.m_off[h.E])) != SIPOC_OK) return rc;
  return download(e, e->h_out[2], out->y, h.n_off[h.N]);
}

sipoc_error sipoc_lqr_factor_solve_host(sipoc_engine *e, const sipoc_lqr_input *in,
                                        const sipoc_lqr_output *out, int *host_status) {
  if (e == nullptr || in == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = ensure_host_lqr(e)) != SIPOC_OK) return rc;
  if ((rc = host_upload_lqr(e, in, true, true)) != SIPOC_OK) return rc;
  rc = lqr_factor_solve_core(e, host_resident_in(e),
                             LqrOut{e->h_out[0], e->h_out[1], e->h_out[2]}, e->h_status,
                             e->host_stream, host_path_is_pm(e));
  if (rc != SIPOC_OK) return rc;
  e->host_lqr_factored = false;
  if ((rc = host_download_out(e, out)) != SIPOC_OK) return rc;
  if (host_status != nullptr)
    SIPOC_CUDA(e, cudaMemcpyAsync(host_status, e->h_status, e->batch * sizeof(int),
                                  cudaMemcpyDeviceToHost, e->host_stream));
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_lqr_factor_host(sipoc_engine *e, const sipoc_lqr_input *in,
                                  int *host_status) {
  if (e == nullptr || in == nullptr) return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = ensure_host_lqr(e)) != SIPOC_OK) return rc;
  if ((rc = host_upload_lqr(e, in, true, false)) != SIPOC_OK) return rc;
  if ((rc = lqr_factor_core(e, host_resident_in(e), e->h_status, e->host_stream,
                            host_path_is_pm(e))) != SIPOC_OK)
    return rc;
  e->host_lqr_factored = true;
  if (host_status != nullptr)
    SIPOC_CUDA(e, cudaMemcpyAsync(host_status, e->h_status, e->batch * sizeof(int),
                                  cudaMemcpyDeviceToHost, e->host_stream));
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_lqr_solve_host(sipoc_engine *e, const sipoc_lqr_input *in,
                                 const sipoc_lqr_output *out) {
  if (e == nullptr || in == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (!e->host_lqr_factored)
    return fail(e, SIPOC_NOT_FACTORED, "sipoc_lqr_solve_host before sipoc_lqr_factor_host");
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = host_upload_lqr(e, in, false, true)) != SIPOC_OK) return rc;
  rc = lqr_solve_core(e, host_resident_in(e), LqrOut{e->h_out[0], e->h_out[1], e->h_out[2]},
                      e->host_stream, host_path_is_pm(e));
  if (rc != SIPOC_OK) return rc;
  if ((rc = host_download_out(e, out)) != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

// ---- Newton-KKT -------------------------------------------------------------
sipoc_error sipoc_kkt_get_sizes(const sipoc_engine *e, sipoc_kkt_sizes *o) {
  if (e == nullptr || o == nullptr) return SIPOC_INVALID_ARGUMENT;
  const HostStructure &h = e->hs;
  o->x_dim = h.x_dim;
  o->y_dim = h.y_dim;
  o->z_dim = h.z_dim;
  o->kkt_dim = h.kkt_dim;
  o->node_hxx = kkt_model_size(h, 0);
  o->node_jc = kkt_model_size(h, 1);
  o->node_jg = kkt_model_size(h, 2);
  o->edge_hxx = kkt_model_size(h, 3);
  o->edge_hxu = kkt_model_size(h, 4);
  o->edge_huu = kkt_model_size(h, 5);
  o->edge_A = kkt_model_size(h, 6);
  o->edge_B = kkt_model_size(h, 7);
  o->edge_jcx = kkt_model_size(h, 8);
  o->edge_jcu = kkt_model_size(h, 9);
  o->edge_jgx = kkt_model_size(h, 10);
  o->edge_jgu = kkt_model_size(h, 11);
  o->theta_dim = h.theta_dim;
  o->stagewise_x_dim = h.sx_dim;
  int64_t *ts[10] = {&o->node_hxt, &o->node_jct, &o->node_jgt, &o->node_htt, &o->edge_hxt,
                     &o->edge_hut, &o->edge_dynt, &o->edge_jct, &o->edge_jgt, &o->edge_htt};
  for (int i = 0; i < 10; ++i) *ts[i] = kkt_theta_size(h, i);
  return SIPOC_OK;
}

sipoc_error sipoc_kkt_offsets(const sipoc_engine *e, int *x_state, int *x_control, int *y_dyn,
                              int *y_node_c, int *y_edge_c, int *z_node, int *z_edge) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  const HostStructure &h = e->hs;
  auto cp = [](const std::vector<int> &v, int *dst) {
    if (dst != nullptr) std::copy(v.begin(), v.end(), dst);
  };
  cp(h.x_state, x_state);
  cp(h.x_control, x_control);
  cp(h.y_dyn, y_dyn);
  cp(h.y_node_c, y_node_c);
  cp(h.y_edge_c, y_edge_c);
  cp(h.z_node, z_node);
  cp(h.z_edge, z_edge);
  return SIPOC_OK;
}

sipoc_error sipoc_kkt_factor(sipoc_engine *e, const sipoc_kkt_model *model, const double *w,
                             const double *r1, const double *r2, const double *r3, int *ok,
                             void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || theta_has_null(e, model) || !w || !r1 || !r2 || !r3 || !ok)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT factor argument");
  DeviceGuard guard(e->device);
  return kkt_factor_core(e, to_model(model), to_theta(model), w, r1, r2, r3, ok,
                         static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_kkt_solve(sipoc_engine *e, const sipoc_kkt_model *model, const double *b,
                            double *sol, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || !b || !sol)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT solve argument");
  DeviceGuard guard(e->device);
  return kkt_solve_core(e, to_model(model), b, sol, static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_kkt_apply(sipoc_engine *e, const sipoc_kkt_model *model, const double *w,
                            const double *r1, const double *r2, const double *r3,
                            const double *x, double *y, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || theta_has_null(e, model) || !w || !r1 || !r2 || !r3 || !x || !y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT apply argument");
  DeviceGuard guard(e->device);
  return kkt_apply_core(e, to_model(model), to_theta(model), w, r1, r2, r3, x, y,
                        static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_kkt_vjp(sipoc_engine *e, const sipoc_kkt_model *model, const double *w,
                          const double *r1, const double *r2, const double *r3,
                          const double *sol, const double *cot, double *adjoint,
                          const sipoc_kkt_grad *grad, int *ok, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || theta_has_null(e, model) || !w || !r1 || !r2 || !r3 || !sol ||
      !cot || !adjoint || grad == nullptr)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT VJP argument");
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if ((rc = default_vjp_status(e, &ok)) != SIPOC_OK) return rc;
  // K is symmetric: the adjoint is the same KKT solve with b := cot.
  const KktModel mdl = to_model(model);
  if ((rc = kkt_factor_core(e, mdl, to_theta(model), w, r1, r2, r3, ok, s)) != SIPOC_OK) return rc;
  if ((rc = kkt_solve_core(e, mdl, cot, adjoint, s)) != SIPOC_OK) return rc;
  const sipoc_kkt_theta_grad no_theta{};
  const sipoc_kkt_theta_grad &tg = grad->theta != nullptr ? *grad->theta : no_theta;
  const KktGrad g{grad->node_hxx, grad->node_jc,  grad->node_jg,  grad->edge_hxx, grad->edge_hxu,
                  grad->edge_huu, grad->edge_A,   grad->edge_B,   grad->edge_jcx, grad->edge_jcu,
                  grad->edge_jgx, grad->edge_jgu, tg.node_hxt,    tg.node_jct,    tg.node_jgt,
                  tg.node_htt,    tg.edge_hxt,    tg.edge_hut,    tg.edge_dynt,   tg.edge_jct,
                  tg.edge_jgt,    tg.edge_htt,    grad->b,        grad->w,        grad->r1,
                  grad->r2,       grad->r3};
  const double *const arrays[] = {
      g.node_hxx, g.node_jc,  g.node_jg,  g.edge_hxx,  g.edge_hxu, g.edge_huu, g.edge_A,
      g.edge_B,   g.edge_jcx, g.edge_jcu, g.edge_jgx,  g.edge_jgu, g.node_hxt, g.node_jct,
      g.node_jgt, g.node_htt, g.edge_hxt, g.edge_hut,  g.edge_dynt, g.edge_jct, g.edge_jgt,
      g.edge_htt, g.b,        g.w,        g.r1,        g.r2,       g.r3};
  if (std::all_of(std::begin(arrays), std::end(arrays), [](const double *a) { return !a; }))
    return SIPOC_OK;
  {
    ProfScope ps(&e->prof, "kkt_vjp_kernel", s);
    launch_kkt_vjp(e->dt, sol, adjoint, ok, g, e->batch, e->ld, s);
  }
  e->launches += 1;
  return check_launch(e, "kkt_vjp");
}

sipoc_error sipoc_kkt_jvp(sipoc_engine *e, const sipoc_kkt_model *model, const double *w,
                          const double *r1, const double *r2, const double *r3,
                          const double *sol, const sipoc_kkt_tangent *tangent, double *rhs,
                          double *dsol, int *ok, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || theta_has_null(e, model) || !w || !r1 || !r2 || !r3 || !sol ||
      tangent == nullptr || !rhs || !dsol)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT JVP argument");
  DeviceGuard guard(e->device);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if ((rc = default_vjp_status(e, &ok)) != SIPOC_OK) return rc;
  const sipoc_kkt_model &tm = tangent->model;
  const KktThetaModel tt = to_theta(&tm);
  const KktTangent d{tm.node_hxx, tm.node_jc,  tm.node_jg,  tm.edge_hxx,  tm.edge_hxu, tm.edge_huu,
                     tm.edge_A,   tm.edge_B,   tm.edge_jcx, tm.edge_jcu,  tm.edge_jgx, tm.edge_jgu,
                     tt.node_hxt, tt.node_jct, tt.node_jgt, tt.node_htt,  tt.edge_hxt, tt.edge_hut,
                     tt.edge_dynt, tt.edge_jct, tt.edge_jgt, tt.edge_htt, tangent->b,  tangent->w,
                     tangent->r1, tangent->r2, tangent->r3};
  {
    ProfScope ps(&e->prof, "kkt_jvp_kernel", s);
    launch_kkt_jvp(e->dt, sol, d, rhs, e->batch, e->ld, s);
  }
  e->launches += 1;
  if ((rc = check_launch(e, "kkt_jvp")) != SIPOC_OK) return rc;
  // The tangent is the same KKT solve with b := t.
  const KktModel mdl = to_model(model);
  if ((rc = kkt_factor_core(e, mdl, to_theta(model), w, r1, r2, r3, ok, s)) != SIPOC_OK) return rc;
  if ((rc = kkt_solve_core(e, mdl, rhs, dsol, s)) != SIPOC_OK) return rc;
  {
    ProfScope ps(&e->prof, "jvp_zero_dead_lanes", s);
    launch_zero_dead_lanes(dsol, e->hs.kkt_dim, ok, true, e->batch, e->ld, s);
  }
  e->launches += 1;
  return check_launch(e, "kkt_jvp zero pass");
}

namespace {
// block -> (mask, length of x, length of y) and the launch on the right vector slots
sipoc_error kkt_apply_block_core(sipoc_engine *e, const KktModel &mdl, const KktThetaModel &tm,
                                 int block, const double *x, double *y, cudaStream_t s) {
  const double *ix = nullptr, *iy = nullptr, *iz = nullptr;
  double *ox = nullptr, *oy = nullptr, *oz = nullptr;
  unsigned parts = 0;
  switch (block) {
    case SIPOC_KKT_BLOCK_H: parts = kKktH; ix = x; ox = y; break;
    case SIPOC_KKT_BLOCK_C: parts = kKktC; ix = x; oy = y; break;
    case SIPOC_KKT_BLOCK_CT: parts = kKktCT; iy = x; ox = y; break;
    case SIPOC_KKT_BLOCK_G: parts = kKktG; ix = x; oz = y; break;
    case SIPOC_KKT_BLOCK_GT: parts = kKktGT; iz = x; ox = y; break;
    default: return fail(e, SIPOC_INVALID_ARGUMENT, "unknown KKT block");
  }
  {
    ProfScope ps(&e->prof, "kkt_apply_kernel", s);
    launch_kkt_apply_parts(e->dt, mdl, parts, ix, iy, iz, ox, oy, oz, e->batch, e->ld, s);
  }
  e->launches += 1;
  if (e->hs.theta_dim > 0) {  // theta branches of helpers.cpp:1019-1368
    ProfScope ps(&e->prof, "theta_apply_kernel", s);
    launch_theta_apply(e->dt, tm, parts, nullptr, ix, iy, iz, ox, oy, oz, e->batch, e->ld, s);
    e->launches += 1;
  }
  return check_launch(e, "kkt_apply_block");
}

void kkt_block_dims(const sipoc_engine *e, int block, int64_t *nx, int64_t *ny) {
  const HostStructure &h = e->hs;
  const int64_t in[5] = {h.x_dim, h.x_dim, h.y_dim, h.x_dim, h.z_dim};
  const int64_t out[5] = {h.x_dim, h.y_dim, h.x_dim, h.z_dim, h.x_dim};
  *nx = in[block];
  *ny = out[block];
}
}  // namespace

sipoc_error sipoc_kkt_apply_block(sipoc_engine *e, const sipoc_kkt_model *model, int block,
                                  const double *x, double *y, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (block < SIPOC_KKT_BLOCK_H || block > SIPOC_KKT_BLOCK_GT)
    return fail(e, SIPOC_INVALID_ARGUMENT, "unknown KKT block");
  int64_t nx = 0, ny = 0;
  kkt_block_dims(e, block, &nx, &ny);
  if (nx == 0 || ny == 0) return SIPOC_OK;  // an empty block (e.g. no inequalities)
  if (model_has_null(model) || theta_has_null(e, model) || !x || !y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT apply argument");
  DeviceGuard guard(e->device);
  return kkt_apply_block_core(e, to_model(model), to_theta(model), block, x, y,
                              static_cast<cudaStream_t>(stream));
}

sipoc_error sipoc_kkt_residual(sipoc_engine *e, const sipoc_kkt_model *model, const double *w,
                               const double *r1, const double *r2, const double *r3,
                               const double *sol, const double *b, const int *ok,
                               double *residual_norm, double *stats, void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (model_has_null(model) || theta_has_null(e, model) || !w || !r1 || !r2 || !r3 || !sol || !b)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL KKT residual argument");
  DeviceGuard guard(e->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  sipoc_error rc;
  if (e->kkt_product == nullptr &&
      (rc = alloc_doubles(e, &e->kkt_product, e->hs.kkt_dim)) != SIPOC_OK)
    return rc;
  SIPOC_CUDA(e, cudaMemsetAsync(e->kkt_product, 0,
                                static_cast<size_t>(std::max(1, e->hs.kkt_dim)) * e->ld *
                                    sizeof(double),
                                s));
  if ((rc = kkt_apply_core(e, to_model(model), to_theta(model), w, r1, r2, r3, sol,
                           e->kkt_product, s)) != SIPOC_OK)
    return rc;
  {
    ProfScope ps(&e->prof, "kkt_residual_kernel", s);
    launch_kkt_residual(e->dt, e->kkt_product, b, ok, residual_norm, stats, e->batch, e->ld,
                        s);
  }
  e->launches += stats != nullptr ? 2 : 1;
  if ((rc = check_launch(e, "kkt_residual")) != SIPOC_OK) return rc;
  return reduce_stats(e, stats, stream);
}

static KktThetaModel host_resident_theta(const sipoc_engine *e) {
  const double *const *t = e->hk_theta;
  return KktThetaModel{t[0], t[1], t[2], t[3], t[4], t[5], t[6], t[7], t[8], t[9]};
}

static KktModel host_resident_model(const sipoc_engine *e) {
  return KktModel{e->hk_model[0], e->hk_model[1], e->hk_model[2],  e->hk_model[3],
                  e->hk_model[4], e->hk_model[5], e->hk_model[6],  e->hk_model[7],
                  e->hk_model[8], e->hk_model[9], e->hk_model[10], e->hk_model[11]};
}

sipoc_error sipoc_kkt_factor_host(sipoc_engine *e, const sipoc_kkt_model *m, const double *w,
                                  const double *r1, const double *r2, const double *r3,
                                  int *host_ok) {
  if (e == nullptr || m == nullptr) return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = ensure_host_kkt(e)) != SIPOC_OK) return rc;
  const double *src[12] = {m->node_hxx, m->node_jc,  m->node_jg,  m->edge_hxx,
                           m->edge_hxu, m->edge_huu, m->edge_A,   m->edge_B,
                           m->edge_jcx, m->edge_jcu, m->edge_jgx, m->edge_jgu};
  for (int i = 0; i < 12; ++i)
    if ((rc = upload(e, src[i], e->hk_model[i], kkt_model_size(e->hs, i))) != SIPOC_OK)
      return rc;
  if (e->hs.theta_dim > 0) {
    if (theta_has_null(e, m)) return fail(e, SIPOC_INVALID_ARGUMENT, "NULL theta model block");
    const sipoc_kkt_theta_model *t = m->theta;
    const double *tsrc[10] = {t->node_hxt, t->node_jct, t->node_jgt, t->node_htt, t->edge_hxt,
                              t->edge_hut, t->edge_dynt, t->edge_jct, t->edge_jgt, t->edge_htt};
    for (int i = 0; i < 10; ++i)
      if ((rc = upload(e, tsrc[i], e->hk_theta[i], kkt_theta_size(e->hs, i))) != SIPOC_OK)
        return rc;
  }
  e->host_model_resident = true;
  if (w == nullptr && r1 == nullptr && r2 == nullptr && r3 == nullptr && host_ok == nullptr) {
    // sipoc_kkt_set_model_host: the model only (the operator entry points read it)
    SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
    return SIPOC_OK;
  }
  const double *reg[4] = {w, r1, r2, r3};
  const int64_t reg_sizes[4] = {e->hs.z_dim, e->hs.x_dim, e->hs.y_dim, e->hs.z_dim};
  for (int i = 0; i < 4; ++i)
    if ((rc = upload(e, reg[i], e->hk_reg[i], reg_sizes[i])) != SIPOC_OK) return rc;
  rc = kkt_factor_core(e, host_resident_model(e), host_resident_theta(e), e->hk_reg[0],
                       e->hk_reg[1], e->hk_reg[2], e->hk_reg[3], e->h_status, e->host_stream);
  if (rc != SIPOC_OK) return rc;
  if (host_ok != nullptr)
    SIPOC_CUDA(e, cudaMemcpyAsync(host_ok, e->h_status, e->batch * sizeof(int),
                                  cudaMemcpyDeviceToHost, e->host_stream));
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_kkt_set_model_host(sipoc_engine *e, const sipoc_kkt_model *m) {
  return sipoc_kkt_factor_host(e, m, nullptr, nullptr, nullptr, nullptr, nullptr);
}

sipoc_error sipoc_kkt_solve_host(sipoc_engine *e, const double *b, double *sol) {
  if (e == nullptr || b == nullptr || sol == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (!e->host_kkt_ready || !e->kkt_factored)
    return fail(e, SIPOC_NOT_FACTORED, "sipoc_kkt_solve_host before sipoc_kkt_factor_host");
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = upload(e, b, e->hk_vec[0], e->hs.kkt_dim)) != SIPOC_OK) return rc;
  rc = kkt_solve_core(e, host_resident_model(e), e->hk_vec[0], e->hk_vec[1], e->host_stream);
  if (rc != SIPOC_OK) return rc;
  if ((rc = download(e, e->hk_vec[1], sol, e->hs.kkt_dim)) != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_kkt_apply_host(sipoc_engine *e, const double *w, const double *r1,
                                 const double *r2, const double *r3, const double *x,
                                 double *y) {
  if (e == nullptr || !w || !r1 || !r2 || !r3 || !x || !y) return SIPOC_INVALID_ARGUMENT;
  if (!e->host_kkt_ready || !e->host_model_resident)
    return fail(e, SIPOC_NOT_FACTORED,
                "sipoc_kkt_apply_host needs the model uploaded by sipoc_kkt_factor_host / "
                "sipoc_kkt_set_model_host");
  DeviceGuard guard(e->device);
  sipoc_error rc;
  const double *reg[4] = {w, r1, r2, r3};
  const int64_t reg_sizes[4] = {e->hs.z_dim, e->hs.x_dim, e->hs.y_dim, e->hs.z_dim};
  for (int i = 0; i < 4; ++i)
    if ((rc = upload(e, reg[i], e->hk_reg[i], reg_sizes[i])) != SIPOC_OK) return rc;
  if ((rc = upload(e, x, e->hk_vec[0], e->hs.kkt_dim)) != SIPOC_OK) return rc;
  if ((rc = upload(e, y, e->hk_vec[1], e->hs.kkt_dim)) != SIPOC_OK) return rc;
  if ((rc = kkt_apply_core(e, host_resident_model(e), host_resident_theta(e), e->hk_reg[0],
                           e->hk_reg[1], e->hk_reg[2], e->hk_reg[3], e->hk_vec[0], e->hk_vec[1],
                           e->host_stream)) != SIPOC_OK)
    return rc;
  if ((rc = download(e, e->hk_vec[1], y, e->hs.kkt_dim)) != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_kkt_apply_block_host(sipoc_engine *e, int block, const double *x, double *y) {
  if (e == nullptr || !x || !y) return SIPOC_INVALID_ARGUMENT;
  if (block < SIPOC_KKT_BLOCK_H || block > SIPOC_KKT_BLOCK_GT)
    return fail(e, SIPOC_INVALID_ARGUMENT, "unknown KKT block");
  if (!e->host_kkt_ready || !e->host_model_resident)
    return fail(e, SIPOC_NOT_FACTORED,
                "sipoc_kkt_apply_block_host needs the model uploaded by sipoc_kkt_factor_host / "
                "sipoc_kkt_set_model_host");
  DeviceGuard guard(e->device);
  sipoc_error rc;
  int64_t nx = 0, ny = 0;
  kkt_block_dims(e, block, &nx, &ny);
  if (nx == 0 || ny == 0) return SIPOC_OK;
  if ((rc = upload(e, x, e->hk_vec[0], nx)) != SIPOC_OK) return rc;
  if ((rc = upload(e, y, e->hk_vec[1], ny)) != SIPOC_OK) return rc;
  if ((rc = kkt_apply_block_core(e, host_resident_model(e), host_resident_theta(e), block,
                                 e->hk_vec[0], e->hk_vec[1], e->host_stream)) != SIPOC_OK)
    return rc;
  if ((rc = download(e, e->hk_vec[1], y, ny)) != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

sipoc_error sipoc_generate_lqr_benchmark(sipoc_engine *e, uint64_t seed, int64_t problem_offset,
                                         double *Q, double *M, double *R, double *q, double *r,
                                         double *A, double *B, double *c, double *delta,
                                         void *stream) {
  if (e == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (!Q || !M || !R || !q || !r || !A || !B || !c || !delta)
    return fail(e, SIPOC_INVALID_ARGUMENT, "NULL generator output");
  const HostStructure &h = e->hs;
  if (!(h.is_chain && h.is_uniform))
    return fail(e, SIPOC_UNSUPPORTED, "the benchmark generator covers uniform chains only");
  DeviceGuard guard(e->device);
  e->launches += launch_generate_lqr_benchmark(seed, problem_offset, h.E, h.n[0],
                                               h.E > 0 ? h.m[0] : 0, e->batch, e->ld, Q, M, R,
                                               q, r, A, B, c, delta,
                                               static_cast<cudaStream_t>(stream));
  return check_launch(e, "generate_lqr_benchmark");
}

}  // extern "C"

// ---- model-callback scatter (sip_optimal_control.cpp:13-127) --------------------------
namespace {
int64_t model_value_size(const HostStructure &h, int i) {
  const int64_t p = h.theta_dim;
  switch (i) {
    case 0: return h.N;
    case 1: return h.n_off[h.N];
    case 2: return h.N * p;
    case 3: return h.node_c_off[h.N];
    case 4: return h.node_g_off[h.N];
    case 5: return h.E;
    case 6: return h.pn_off[h.E];
    case 7: return h.m_off[h.E];
    case 8: return h.E * p;
    case 9: return h.cn_off[h.E];
    case 10: return h.edge_c_off[h.E];
    default: return h.edge_g_off[h.E];
  }
}
}  // namespace

extern "C" {

sipoc_error sipoc_model_value_sizes(const sipoc_engine *e, sipoc_model_value_sizes_t *o) {
  if (e == nullptr || o == nullptr) return SIPOC_INVALID_ARGUMENT;
  int64_t *fields[12] = {&o->node_f,      &o->node_df_dx, &o->node_df_dtheta, &o->node_c,
                         &o->node_g,      &o->edge_f,     &o->edge_df_dx,     &o->edge_df_du,
                         &o->edge_df_dtheta, &o->edge_dyn_res, &o->edge_c,    &o->edge_g};
  for (int i = 0; i < 12; ++i) *fields[i] = model_value_size(e->hs, i);
  return SIPOC_OK;
}

sipoc_error sipoc_model_scatter(sipoc_engine *e, const sipoc_model_values *v, const double *x,
                                const double *initial_state, int new_x, double *f,
                                double *gradient_f, double *c, double *g, void *stream) {
  if (e == nullptr || v == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (f == nullptr || (new_x && (!x || !initial_state || !gradient_f || !c || !g)))
    return fail(e, SIPOC_INVALID_ARGUMENT, "sipoc_model_scatter: NULL vector");
  if (e->hs.N + e->hs.E + 1 > 65535)
    return fail(e, SIPOC_UNSUPPORTED, "sipoc_model_scatter: more than 32 767 edges");
  DeviceGuard guard(e->device);
  const ModelValues mv{v->node_f, v->node_df_dx, v->node_df_dtheta, v->node_c, v->node_g,
                       v->edge_f, v->edge_df_dx, v->edge_df_du, v->edge_df_dtheta,
                       v->edge_dyn_res, v->edge_c, v->edge_g};
  e->launches += launch_model_scatter(e->dt, mv, x, initial_state, new_x != 0, f, gradient_f, c, g,
                                      e->batch, e->ld, static_cast<cudaStream_t>(stream));
  return check_launch(e, "model_scatter");
}

sipoc_error sipoc_model_scatter_host(sipoc_engine *e, const sipoc_model_values *v,
                                     const double *x, const double *initial_state, int new_x,
                                     double *f, double *gradient_f, double *c, double *g) {
  if (e == nullptr || v == nullptr || f == nullptr) return SIPOC_INVALID_ARGUMENT;
  DeviceGuard guard(e->device);
  const HostStructure &h = e->hs;
  sipoc_error rc;
  const int64_t out_sizes[4] = {1, h.x_dim, h.y_dim, h.z_dim};
  if (!e->host_scatter_ready) {
    int64_t biggest = std::max<int64_t>(h.x_dim, std::max(h.y_dim, h.z_dim));
    for (int i = 0; i < 12; ++i) {
      if ((rc = alloc_doubles(e, &e->hm_vals[i], model_value_size(h, i))) != SIPOC_OK) return rc;
      biggest = std::max(biggest, model_value_size(h, i));
    }
    if ((rc = alloc_doubles(e, &e->hm_x, h.x_dim)) != SIPOC_OK) return rc;
    if ((rc = alloc_doubles(e, &e->hm_x0, h.n[h.root])) != SIPOC_OK) return rc;
    for (int i = 0; i < 4; ++i)
      if ((rc = alloc_doubles(e, &e->hm_out[i], out_sizes[i])) != SIPOC_OK) return rc;
    if ((rc = ensure_stage(e, biggest)) != SIPOC_OK) return rc;
    e->host_scatter_ready = true;
  }
  const double *src[12] = {v->node_f, v->node_df_dx, v->node_df_dtheta, v->node_c, v->node_g,
                           v->edge_f, v->edge_df_dx, v->edge_df_du, v->edge_df_dtheta,
                           v->edge_dyn_res, v->edge_c, v->edge_g};
  for (int i = 0; i < 12; ++i) {
    const bool needed = new_x || i == 0 || i == 5;  // f alone reads the two f arrays
    if (needed && (rc = upload(e, src[i], e->hm_vals[i], model_value_size(h, i))) != SIPOC_OK)
      return rc;
  }
  if (new_x) {
    if ((rc = upload(e, x, e->hm_x, h.x_dim)) != SIPOC_OK) return rc;
    if ((rc = upload(e, initial_state, e->hm_x0, h.n[h.root])) != SIPOC_OK) return rc;
  }
  const sipoc_model_values dv{e->hm_vals[0], e->hm_vals[1], e->hm_vals[2],  e->hm_vals[3],
                              e->hm_vals[4], e->hm_vals[5], e->hm_vals[6],  e->hm_vals[7],
                              e->hm_vals[8], e->hm_vals[9], e->hm_vals[10], e->hm_vals[11]};
  if ((rc = sipoc_model_scatter(e, &dv, e->hm_x, e->hm_x0, new_x, e->hm_out[0], e->hm_out[1],
                                e->hm_out[2], e->hm_out[3], e->host_stream)) != SIPOC_OK)
    return rc;
  double *dst[4] = {f, gradient_f, c, g};
  for (int i = 0; i < (new_x ? 4 : 1); ++i)
    if ((rc = download(e, e->hm_out[i], dst[i], out_sizes[i])) != SIPOC_OK) return rc;
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}

}  // extern "C"

// ---- optional FP32 mode (riccati_f32.cu) ---------------------------------------------
extern "C" {

int sipoc_f32_supported(const sipoc_engine *e) {
  if (e == nullptr) return 0;
  const HostStructure &h = e->hs;
  return h.is_chain && h.is_uniform && h.E > 0 && f32_supports(h.n[0], h.m[0]) &&
                 f32_fits_index(h.n[0], h.m[0], h.E, e->ld)
             ? 1
             : 0;
}

sipoc_error sipoc_lqr_factor_solve_f32(sipoc_engine *e, const sipoc_lqr_input_f32 *in,
                                       const sipoc_lqr_output_f32 *out, int *status,
                                       void *stream) {
  if (e == nullptr || in == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (!sipoc_f32_supported(e))
    return fail(e, SIPOC_UNSUPPORTED,
                "the FP32 mode covers uniform chains with state dimension 4 and 1..4 controls");
  if (!in->Q || !in->M || !in->R || !in->q || !in->r || !in->A || !in->B || !in->c || !in->delta ||
      !out->x || !out->u || !out->y)
    return fail(e, SIPOC_INVALID_ARGUMENT, "sipoc_lqr_factor_solve_f32: NULL array");
  DeviceGuard guard(e->device);
  const HostStructure &h = e->hs;
  sipoc_error rc;
  if (e->f32_store == nullptr &&
      (rc = dev_alloc(e, reinterpret_cast<void **>(&e->f32_store),
                      static_cast<size_t>(f32_store_elems(h.n[0], h.m[0], h.E)) * e->ld *
                          sizeof(float))) != SIPOC_OK)
    return rc;
  const LqrInT<float> i{in->Q, in->M, in->R, in->q, in->r, in->A, in->B, in->c, in->delta};
  const LqrOutT<float> o{out->x, out->u, out->y};
  e->launches += launch_lqr_factor_solve_f32(h.n[0], h.m[0], i, o, status, e->f32_store, e->batch,
                                             e->ld, h.E, &e->prof,
                                             static_cast<cudaStream_t>(stream));
  return check_launch(e, "lqr_factor_solve_f32");
}

sipoc_error sipoc_lqr_factor_solve_thread_f64(sipoc_engine *e, const sipoc_lqr_input *in,
                                              const sipoc_lqr_output *out, int *status,
                                              void *stream) {
  if (e == nullptr || in == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  if (!sipoc_f32_supported(e))
    return fail(e, SIPOC_UNSUPPORTED,
                "the FP32 mode covers uniform chains with state dimension 4 and 1..4 controls");
  DeviceGuard guard(e->device);
  const HostStructure &h = e->hs;
  sipoc_error rc;
  if (e->f64t_store == nullptr &&
      (rc = alloc_doubles(e, &e->f64t_store, f32_store_elems(h.n[0], h.m[0], h.E))) != SIPOC_OK)
    return rc;
  const LqrInT<double> i{in->Q, in->M, in->R, in->q, in->r, in->A, in->B, in->c, in->delta};
  const LqrOutT<double> o{out->x, out->u, out->y};
  e->launches += launch_lqr_factor_solve_thread_f64(h.n[0], h.m[0], i, o, status, e->f64t_store,
                                                    e->batch, e->ld, h.E, &e->prof,
                                                    static_cast<cudaStream_t>(stream));
  return check_launch(e, "lqr_factor_solve_thread_f64");
}

}  // extern "C"

// ---- packed-symmetric host entry ---------------------------------------------------------
namespace {

// Symmetric n x n blocks from their packed lower triangles, both in the engine layout:
// dense[(blk n n + j n + i) ld + b] = packed[(blk tri + pk(max(i, j), min(i, j))) ld + b].
__global__ void __launch_bounds__(128)
expand_symmetric_kernel(const double *__restrict__ packed, double *__restrict__ dense, int n,
                        int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * 128 + threadIdx.x;
  if (b >= batch) return;
  const int nn = n * n, tri = n * (n + 1) / 2;
  const int f = blockIdx.y, blk = f / nn, rem = f % nn, i = rem % n, j = rem / n;
  const int r = i > j ? i : j, c = i > j ? j : i;
  const size_t src = static_cast<size_t>(blk) * tri + c * n - c * (c - 1) / 2 + (r - c);
  dense[static_cast<size_t>(f) * ld + b] = __ldcs(packed + src * ld + b);
}

sipoc_error upload_packed_symmetric(sipoc_engine *e, const double *host, double *dense, int n,
                                    int blocks) {
  if (blocks == 0 || n == 0) return SIPOC_OK;
  const int64_t tri = static_cast<int64_t>(n) * (n + 1) / 2;
  sipoc_error rc = upload(e, host, e->h_packed, blocks * tri);
  if (rc != SIPOC_OK) return rc;
  const dim3 grid(static_cast<unsigned>((e->batch + 127) / 128),
                  static_cast<unsigned>(blocks * n * n));
  {
    ProfScope ps(&e->prof, "expand_symmetric_kernel", e->host_stream);
    expand_symmetric_kernel<<<grid, 128, 0, e->host_stream>>>(e->h_packed, dense, n, e->batch,
                                                              e->ld);
  }
  e->launches += 1;
  return check_launch(e, "expand_symmetric");
}

}  // namespace

extern "C" sipoc_error sipoc_lqr_factor_solve_host_packed(sipoc_engine *e,
                                                          const sipoc_lqr_input *in,
                                                          const sipoc_lqr_output *out,
                                                          int *host_status) {
  if (e == nullptr || in == nullptr || out == nullptr) return SIPOC_INVALID_ARGUMENT;
  const HostStructure &h = e->hs;
  if (!h.is_uniform)
    return fail(e, SIPOC_UNSUPPORTED, "the packed host entry needs uniform state / control dims");
  if (host_path_is_pm(e))
    return fail(e, SIPOC_UNSUPPORTED,
                "the packed host entry serves the plans on the interleaved layout (state dim < 16)");
  const int n = h.n[0], m = h.E > 0 ? h.m[0] : 0;
  if (static_cast<int64_t>(h.N) * n * n > 65535)
    return fail(e, SIPOC_UNSUPPORTED, "the packed host entry: more than 65 535 dense Q entries");
  DeviceGuard guard(e->device);
  sipoc_error rc;
  if ((rc = ensure_host_lqr(e)) != SIPOC_OK) return rc;
  const int64_t tq = static_cast<int64_t>(h.N) * n * (n + 1) / 2,
                tr = static_cast<int64_t>(h.E) * m * (m + 1) / 2;
  if (e->h_packed == nullptr) {
    if ((rc = alloc_doubles(e, &e->h_packed, std::max(tq, tr))) != SIPOC_OK) return rc;
    if ((rc = ensure_stage(e, std::max(tq, tr))) != SIPOC_OK) return rc;
  }
  // Q, R: lower triangles over the bus, expanded on the device; M: NULL means zero
  if ((rc = upload_packed_symmetric(e, in->Q, e->h_in[0], n, h.N)) != SIPOC_OK) return rc;
  if ((rc = upload_packed_symmetric(e, in->R, e->h_in[2], m, h.E)) != SIPOC_OK) return rc;
  if (in->M != nullptr) {
    if ((rc = upload(e, in->M, e->h_in[1], lqr_in_size(h, 1))) != SIPOC_OK) return rc;
  } else if (lqr_in_size(h, 1) > 0) {
    SIPOC_CUDA(e, cudaMemsetAsync(e->h_in[1], 0,
                                  static_cast<size_t>(lqr_in_size(h, 1)) * e->ld * sizeof(double),
                                  e->host_stream));
  }
  const double *rest[9] = {nullptr, nullptr, nullptr, in->q, in->r, in->A, in->B, in->c, in->delta};
  for (int i = 3; i < 9; ++i)
    if ((rc = upload(e, rest[i], e->h_in[i], lqr_in_size(h, i))) != SIPOC_OK) return rc;
  rc = lqr_factor_solve_core(e, host_resident_in(e),
                             LqrOut{e->h_out[0], e->h_out[1], e->h_out[2]}, e->h_status,
                             e->host_stream, false);
  if (rc != SIPOC_OK) return rc;
  e->host_lqr_factored = false;
  if ((rc = host_download_out(e, out)) != SIPOC_OK) return rc;
  if (host_status != nullptr)
    SIPOC_CUDA(e, cudaMemcpyAsync(host_status, e->h_status, e->batch * sizeof(int),
                                  cudaMemcpyDeviceToHost, e->host_stream));
  SIPOC_CUDA(e, cudaStreamSynchronize(e->host_stream));
  return SIPOC_OK;
}
