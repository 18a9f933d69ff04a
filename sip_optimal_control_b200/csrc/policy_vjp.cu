// Adjoint Riccati sweep of the policy VJP (see policy_vjp.cuh for the formulas).
//
// One device routine, edge_adjoint, does the per-edge algebra on any scratch view: the
// shape-specialised chain kernel instantiates it with compile-time dims and a thread-local
// scratch (the loops fold to constants), the generic kernel with runtime dims and an
// engine-layout workspace (coalesced across the 32 problems of a warp).  Statement order is
// the same in both.  The primal recompute of an edge and the small helpers are shared with the
// policy JVP (policy_common.cuh).
#include "policy_vjp.cuh"

#include <algorithm>

#include "policy_common.cuh"

namespace sipoc {

namespace {

using namespace policy_detail;

constexpr int kThreads = 128;

// Offsets of the per-edge scratch arrays, for state dims <= nx and controls <= mx.
struct Slots {
  int sd, sdi, Lf, P, W, Y, Yb, Wb, WB, BG, Lg, Gb, K, Kb, KV, f, g, h, k, kb, hb, gb, fb, total;
};

__host__ __device__ constexpr Slots make_slots(int nx, int mx) {
  const int nn = nx * nx, nm = nx * mx, mm = mx * mx;
  Slots s{};
  int o = 0;
  s.sd = o; o += nx;
  s.sdi = o; o += nx;
  s.Lf = o; o += nn;  // Cholesky factor of F, later T = D^-1/2 Wb D^-1/2 P
  s.P = o; o += nn;
  s.W = o; o += nn;
  s.Y = o; o += nn;
  s.Yb = o; o += nn;  // Yb, later A Vb_p + Yb
  s.Wb = o; o += nn;
  s.WB = o; o += nm;  // W B
  s.BG = o; o += nm;  // B Gb
  s.Lg = o; o += mm;
  s.Gb = o; o += mm;
  s.K = o; o += nm;
  s.Kb = o; o += nm;  // Kb, then G^-1 Kb
  s.KV = o; o += nm;  // K Vb_p, then Hb
  s.f = o; o += nx;
  s.g = o; o += nx;
  s.gb = o; o += nx;
  s.fb = o; o += nx;
  s.h = o; o += mx;
  s.k = o; o += mx;
  s.kb = o; o += mx;  // kb, then G^-1 kb
  s.hb = o; o += mx;
  s.total = o;
  return s;
}

// A thread's local array (chain kernel).
struct Loc {
  double *p;
  __device__ __forceinline__ double &operator()(int i) const { return p[i]; }
};

struct Lanes {
  GCVec A, B, M, R, r, c, delta, V, v;
  OptIn cK, ck, cV, cv;
  OptOut Q, Mg, Rg, q, rg, Ag, Bg, cg, dg;
};

__device__ __forceinline__ Lanes make_lanes(const PolicyVjpIn &in, const LqrPolicyCot &cot,
                                            const LqrGrad &g, int64_t b, size_t L) {
  return Lanes{GCVec{in.in.A + b, L},     GCVec{in.in.B + b, L},  GCVec{in.in.M + b, L},
               GCVec{in.in.R + b, L},     GCVec{in.in.r + b, L},  GCVec{in.in.c + b, L},
               GCVec{in.in.delta + b, L}, GCVec{in.V + b, L},     GCVec{in.v + b, L},
               OptIn{cot.K ? cot.K + b : nullptr, L}, OptIn{cot.k ? cot.k + b : nullptr, L},
               OptIn{cot.V ? cot.V + b : nullptr, L}, OptIn{cot.v ? cot.v + b : nullptr, L},
               OptOut{g.Q ? g.Q + b : nullptr, L},     OptOut{g.M ? g.M + b : nullptr, L},
               OptOut{g.R ? g.R + b : nullptr, L},     OptOut{g.q ? g.q + b : nullptr, L},
               OptOut{g.r ? g.r + b : nullptr, L},     OptOut{g.A ? g.A + b : nullptr, L},
               OptOut{g.B ? g.B + b : nullptr, L},     OptOut{g.c ? g.c + b : nullptr, L},
               OptOut{g.delta ? g.delta + b : nullptr, L}};
}

// Element counts of the nine input arrays of one problem (the gradient arrays' sizes).
struct GradSizes {
  int Q, M, R, q, r, A, B, c, delta;
};

__device__ void zero_grads(const Lanes &l, const GradSizes &z) {
  for (int i = 0; i < z.Q; ++i) l.Q.set(i, 0.0);
  for (int i = 0; i < z.M; ++i) l.Mg.set(i, 0.0);
  for (int i = 0; i < z.R; ++i) l.Rg.set(i, 0.0);
  for (int i = 0; i < z.q; ++i) l.q.set(i, 0.0);
  for (int i = 0; i < z.r; ++i) l.rg.set(i, 0.0);
  for (int i = 0; i < z.A; ++i) l.Ag.set(i, 0.0);
  for (int i = 0; i < z.B; ++i) l.Bg.set(i, 0.0);
  for (int i = 0; i < z.c; ++i) l.cg.set(i, 0.0);
  for (int i = 0; i < z.delta; ++i) l.dg.set(i, 0.0);
}

// The adjoint of edge e (policy_vjp.cuh).  Vp / vp hold Vb_p (np x np) and vb_p at vpo / vpv;
// Vb_c and vb_c of the child, its own cotangent included, go to Vc / vc at vco / vcv.
template <class S, class VP, class VC>
__device__ __forceinline__ void edge_adjoint(const Edge &e, const Slots &s, const S &w,
                                             const Lanes &l, const VP &Vp, int vpo, int vpv,
                                             const VC &Vc, int vco, int vcv) {
  const int np = e.np, nc = e.nc, m = e.m;
  auto A = [&](int i, int j) { return l.A(e.a + i + j * nc); };
  auto B = [&](int i, int a) { return l.B(e.b + i + a * nc); };
  auto Vb = [&](int i, int j) -> double & { return Vp(vpo + i + j * np); };
  auto vb = [&](int i) -> double & { return Vp(vpv + i); };
  auto X = [&](int slot, int i, int j, int rows) -> double & { return w(slot + i + j * rows); };

  edge_primal(e, s, w, l);

  // ---- adjoint.  Kb = cot K + h vb_p', kb = cot k, then G^-1 Kb, G^-1 kb in place
  for (int j = 0; j < np; ++j)
    for (int a = 0; a < m; ++a) X(s.Kb, a, j, m) = l.cK(e.mo + a + j * m) + w(s.h + a) * vb(j);
  for (int a = 0; a < m; ++a) w(s.kb + a) = l.ck(e.ru + a);
  chol_solve(w, s.Lg, m, s.Kb, np);
  chol_solve(w, s.Lg, m, s.kb, 1);
  // KV = K Vb_p;  hb = K vb_p - G^-1 kb
  for (int j = 0; j < np; ++j)
    for (int a = 0; a < m; ++a) {
      double t = 0.0;
      for (int k = 0; k < np; ++k) t += X(s.K, a, k, m) * Vb(k, j);
      X(s.KV, a, j, m) = t;
    }
  for (int a = 0; a < m; ++a) {
    double t = -w(s.kb + a);
    for (int j = 0; j < np; ++j) t += X(s.K, a, j, m) * vb(j);
    w(s.hb + a) = t;
  }
  // Gb = sym((K Vb_p - G^-1 Kb) K' - G^-1 kb k')
  for (int bb = 0; bb < m; ++bb)
    for (int a = bb; a < m; ++a) {
      double x = -w(s.kb + a) * w(s.k + bb), y = -w(s.kb + bb) * w(s.k + a);
      for (int j = 0; j < np; ++j) {
        x += (X(s.KV, a, j, m) - X(s.Kb, a, j, m)) * X(s.K, bb, j, m);
        y += (X(s.KV, bb, j, m) - X(s.Kb, bb, j, m)) * X(s.K, a, j, m);
      }
      X(s.Gb, a, bb, m) = X(s.Gb, bb, a, m) = 0.5 * (x + y);
    }
  // Hb = 2 K Vb_p - G^-1 Kb (over KV)
  for (int i = 0; i < m * np; ++i) w(s.KV + i) = 2.0 * w(s.KV + i) - w(s.Kb + i);
  // gb = A vb_p + B hb;  fb = -W_c gb
  for (int i = 0; i < nc; ++i) {
    double t = 0.0;
    for (int j = 0; j < np; ++j) t += A(i, j) * vb(j);
    for (int a = 0; a < m; ++a) t += B(i, a) * w(s.hb + a);
    w(s.gb + i) = t;
  }
  for (int i = 0; i < nc; ++i) {
    double t = 0.0;
    for (int k = 0; k < nc; ++k) t -= X(s.W, i, k, nc) * w(s.gb + k);
    w(s.fb + i) = t;
  }
  // rb = hb, Mb = Hb', Rb = Gb
  if (l.rg)
    for (int a = 0; a < m; ++a) l.rg.set(e.ru + a, w(s.hb + a));
  if (l.Mg)
    for (int a = 0; a < m; ++a)
      for (int j = 0; j < np; ++j) l.Mg.set(e.mo + j + a * np, X(s.KV, a, j, m));
  if (l.Rg)
    for (int i = 0; i < m * m; ++i) l.Rg.set(e.ro + i, w(s.Gb + i));
  // Yb = B Hb
  for (int j = 0; j < np; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int a = 0; a < m; ++a) t += B(i, a) * X(s.KV, a, j, m);
      X(s.Yb, i, j, nc) = t;
    }
  // Ab = g vb_p' + 2 Y Vb_p + W_c Yb
  if (l.Ag)
    for (int j = 0; j < np; ++j)
      for (int i = 0; i < nc; ++i) {
        double y = 0.0, t = 0.0;
        for (int k = 0; k < np; ++k) y += X(s.Y, i, k, nc) * Vb(k, j);
        for (int k = 0; k < nc; ++k) t += X(s.W, i, k, nc) * X(s.Yb, k, j, nc);
        l.Ag.set(e.a + i + j * nc, w(s.g + i) * vb(j) + 2.0 * y + t);
      }
  // Bb = g hb' + Y Hb' + 2 W_c B Gb
  if (l.Bg)
    for (int a = 0; a < m; ++a)
      for (int i = 0; i < nc; ++i) {
        double y = 0.0, t = 0.0;
        for (int j = 0; j < np; ++j) y += X(s.Y, i, j, nc) * X(s.KV, a, j, m);
        for (int bb = 0; bb < m; ++bb) t += X(s.WB, i, bb, nc) * X(s.Gb, bb, a, m);
        l.Bg.set(e.b + i + a * nc, w(s.g + i) * w(s.hb + a) + y + 2.0 * t);
      }
  // Wb = sym((A Vb_p + Yb) A' + (B Gb) B' - gb f')
  for (int j = 0; j < np; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = X(s.Yb, i, j, nc);
      for (int k = 0; k < np; ++k) t += A(i, k) * Vb(k, j);
      X(s.Yb, i, j, nc) = t;
    }
  for (int a = 0; a < m; ++a)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int bb = 0; bb < m; ++bb) t += B(i, bb) * X(s.Gb, bb, a, m);
      X(s.BG, i, a, nc) = t;
    }
  for (int j = 0; j < nc; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = -w(s.gb + i) * w(s.f + j);
      for (int k = 0; k < np; ++k) t += X(s.Yb, i, k, nc) * A(j, k);
      for (int a = 0; a < m; ++a) t += X(s.BG, i, a, nc) * B(j, a);
      X(s.Wb, i, j, nc) = t;
    }
  for (int j = 0; j < nc; ++j)
    for (int i = j + 1; i < nc; ++i)
      X(s.Wb, i, j, nc) = X(s.Wb, j, i, nc) = 0.5 * (X(s.Wb, i, j, nc) + X(s.Wb, j, i, nc));
  // cb_c = -fb;  deltab_c = fb .* v_c - diag(W_c Wb W_c)
  if (l.cg)
    for (int i = 0; i < nc; ++i) l.cg.set(e.cv + i, -w(s.fb + i));
  if (l.dg)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int j = 0; j < nc; ++j) {
        double u = 0.0;
        for (int k = 0; k < nc; ++k) u += X(s.Wb, j, k, nc) * X(s.W, k, i, nc);
        t += X(s.W, i, j, nc) * u;
      }
      l.dg.set(e.cv + i, w(s.fb + i) * l.v(e.cv + i) - t);
    }
  // Vb_c = sym(cot V_c) + D^1/2 P_c (D^-1/2 Wb D^-1/2) P_c D^1/2;  vb_c = cot v_c + gb + delta .* fb
  for (int j = 0; j < nc; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.Wb, i, k, nc) * w(s.sdi + k) * X(s.P, k, j, nc);
      X(s.Lf, i, j, nc) = w(s.sdi + i) * t;
    }
  for (int j = 0; j < nc; ++j)
    for (int i = j; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.P, i, k, nc) * X(s.Lf, k, j, nc);
      const double v = w(s.sd + i) * t * w(s.sd + j) +
                       0.5 * (l.cV(e.cnn + i + j * nc) + l.cV(e.cnn + j + i * nc));
      Vc(vco + i + j * nc) = v;
      Vc(vco + j + i * nc) = v;
    }
  for (int i = 0; i < nc; ++i)
    Vc(vcv + i) = l.cv(e.cv + i) + w(s.gb + i) + l.delta(e.cv + i) * w(s.fb + i);
}

// Vb_r = sym(cot V_r), vb_r = cot v_r of the root, into V at vo / vv; its c and delta get 0.
template <class VS>
__device__ __forceinline__ void root_adjoint(const Lanes &l, int n, int nn, int nv, const VS &V,
                                             int vo, int vv) {
  for (int j = 0; j < n; ++j)
    for (int i = j; i < n; ++i) {
      const double v = 0.5 * (l.cV(nn + i + j * n) + l.cV(nn + j + i * n));
      V(vo + i + j * n) = v;
      V(vo + j + i * n) = v;
    }
  for (int i = 0; i < n; ++i) {
    V(vv + i) = l.cv(nv + i);
    l.cg.set(nv + i, 0.0);
    l.dg.set(nv + i, 0.0);
  }
}

// Qb_i = Vb_i, qb_i = vb_i.
template <class VS>
__device__ __forceinline__ void node_grads(const Lanes &l, int n, int nn, int nv, const VS &V,
                                           int vo, int vv) {
  if (l.Q)
    for (int i = 0; i < n * n; ++i) l.Q.set(nn + i, V(vo + i));
  if (l.q)
    for (int i = 0; i < n; ++i) l.q.set(nv + i, V(vv + i));
}

template <int N, int M>
__global__ void __launch_bounds__(kThreads)
policy_vjp_kernel(PolicyVjpIn in, LqrPolicyCot cot, LqrGrad g, const int *status, int E,
                  int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const Lanes l = make_lanes(in, cot, g, b, L);
  if (!(b < batch && status[b] == SIPOC_FACTOR_SUCCESS)) {
    const int T1 = E + 1;
    zero_grads(l, GradSizes{T1 * N * N, E * N * M, E * M * M, T1 * N, E * M, E * N * N,
                            E * N * M, T1 * N, T1 * N});
    return;
  }
  constexpr Slots s = make_slots(N, M);
  double scratch[s.total];
  double vbuf[2][N * N + N];  // Vb, vb of the current parent and of its child
  const Loc w{scratch};
  root_adjoint(l, N, 0, 0, Loc{vbuf[0]}, 0, N * N);
  node_grads(l, N, 0, 0, Loc{vbuf[0]}, 0, N * N);
#pragma unroll 1
  for (int e = 0; e < E; ++e) {
    const Loc cur{vbuf[e & 1]}, nxt{vbuf[(e & 1) ^ 1]};
    const Edge ed{N,         N,         M,           e * N * N,       e * N * M,
                  e * N * M, e * M * M, e * M,       e * N,           e * N * N,
                  (e + 1) * N, (e + 1) * N * N};
    edge_adjoint(ed, s, w, l, cur, 0, N * N, nxt, 0, N * N);
    node_grads(l, N, (e + 1) * N * N, (e + 1) * N, nxt, 0, N * N);
  }
}

__global__ void __launch_bounds__(kThreads)
policy_vjp_generic_kernel(DevTables t, GradSizes z, Slots s, PolicyVjpIn in, LqrPolicyCot cot,
                          LqrGrad g, double *ws, const int *status, int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const Lanes l = make_lanes(in, cot, g, b, L);
  if (!(b < batch && status[b] == SIPOC_FACTOR_SUCCESS)) {
    zero_grads(l, z);
    return;
  }
  const GVec w{ws + b, L};
  // Vb of node i at s.total + nn_off[i], vb at s.total + nn_off[N] + n_off[i]
  const int vvo = s.total + t.nn_off[t.N];
  const int r = t.root;
  root_adjoint(l, t.n[r], t.nn_off[r], t.n_off[r], w, s.total + t.nn_off[r], vvo + t.n_off[r]);
  for (int order = 0; order < t.N; ++order) {
    const int p = t.preorder[order];
    const int np = t.n[p], pnn = t.nn_off[p], pv = t.n_off[p];
    node_grads(l, np, pnn, pv, w, s.total + pnn, vvo + pv);
    for (int ci = t.child_offsets[p]; ci < t.child_offsets[p + 1]; ++ci) {
      const int e = t.child_edges[ci], c = t.children[e];
      const Edge ed{np,          t.n[c],        t.m[e],      t.a_off[e], t.b_off[e],
                    t.nm_off[e], t.mm_off[e],   t.m_off[e],  pv,         pnn,
                    t.n_off[c],  t.nn_off[c]};
      edge_adjoint(ed, s, w, l, w, s.total + pnn, vvo + pv, w, s.total + ed.cnn, vvo + ed.cv);
    }
  }
}

template <int N, int M>
void chain(int E, const PolicyVjpIn &in, const LqrPolicyCot &cot, const LqrGrad &g,
           const int *status, int64_t batch, int64_t ld, cudaStream_t s) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  policy_vjp_kernel<N, M><<<static_cast<unsigned>((ld + threads - 1) / threads), threads, 0, s>>>(
      in, cot, g, status, E, batch, ld);
}

}  // namespace

int64_t policy_vjp_scratch_elems(int nx, int mx) { return make_slots(nx, mx).total; }

bool policy_vjp_chain_shape(int n, int m) {
  return ((n == 4 || n == 6 || n == 8) && m >= 1 && m <= 4) || (n == 12 && m == 4);
}

bool launch_policy_vjp_chain(int n, int m, int E, const PolicyVjpIn &in, const LqrPolicyCot &cot,
                             const LqrGrad &grad, const int *status, int64_t batch, int64_t ld,
                             cudaStream_t s) {
#define SIPOC_PVJP(NN, MM)                                      \
  if (n == NN && m == MM) {                                     \
    chain<NN, MM>(E, in, cot, grad, status, batch, ld, s);      \
    return true;                                                \
  }
  SIPOC_PVJP(4, 1) SIPOC_PVJP(4, 2) SIPOC_PVJP(4, 3) SIPOC_PVJP(4, 4)
  SIPOC_PVJP(6, 1) SIPOC_PVJP(6, 2) SIPOC_PVJP(6, 3) SIPOC_PVJP(6, 4)
  SIPOC_PVJP(8, 1) SIPOC_PVJP(8, 2) SIPOC_PVJP(8, 3) SIPOC_PVJP(8, 4)
  SIPOC_PVJP(12, 4)
#undef SIPOC_PVJP
  return false;
}

void launch_policy_vjp_generic(const DevTables &t, const HostStructure &h, const PolicyVjpIn &in,
                               const LqrPolicyCot &cot, const LqrGrad &grad, double *ws,
                               const int *status, int64_t batch, int64_t ld, cudaStream_t s) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));
  const GradSizes z{h.nn_off[h.N], h.nm_off[h.E], h.mm_off[h.E], h.n_off[h.N], h.m_off[h.E],
                    h.a_off[h.E],  h.b_off[h.E],  h.n_off[h.N],  h.n_off[h.N]};
  policy_vjp_generic_kernel<<<static_cast<unsigned>((ld + threads - 1) / threads), threads, 0,
                              s>>>(t, z, make_slots(h.max_n, h.max_m), in, cot, grad, ws, status,
                                   batch, ld);
}

}  // namespace sipoc
