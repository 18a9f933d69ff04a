// Tangent Riccati sweep of the policy JVP (see policy_jvp.cuh for the formulas and the two
// kernels).  Both kernels run the statements in the same order as tests/policy_jvp_reference.py.
#include "policy_jvp.cuh"

#include <algorithm>

#include "policy_common.cuh"

namespace sipoc {

namespace {

using namespace policy_detail;

// ---------------------------------------------------------------------------------------------
// Generic kernel: one thread per problem, runtime dims, engine-layout workspace.

constexpr int kThreads = 128;

// Offsets of the per-edge scratch arrays, for state dims <= nx and controls <= mx.  The first
// thirteen are those edge_primal fills.
struct Slots {
  int sd, sdi, Lf, P, W, Y, WB, Lg, K, f, g, h, k;
  int dW, dWA, dY, dWB, dG, dH, dGK, dK, df, dg, dh, dk, total;
};

__host__ __device__ constexpr Slots make_slots(int nx, int mx) {
  const int nn = nx * nx, nm = nx * mx, mm = mx * mx;
  Slots s{};
  int o = 0;
  s.sd = o; o += nx;
  s.sdi = o; o += nx;
  s.Lf = o; o += nn;  // Cholesky factor of F, later T = dV_c S
  s.P = o; o += nn;
  s.W = o; o += nn;
  s.Y = o; o += nn;
  s.WB = o; o += nm;
  s.Lg = o; o += mm;
  s.K = o; o += nm;
  s.f = o; o += nx;
  s.g = o; o += nx;
  s.h = o; o += mx;
  s.k = o; o += mx;
  s.dW = o; o += nn;
  s.dWA = o; o += nn;
  s.dY = o; o += nn;
  s.dWB = o; o += nm;
  s.dG = o; o += mm;
  s.dH = o; o += nm;
  s.dGK = o; o += nm;
  s.dK = o; o += nm;  // dH + dG K, then dK
  s.df = o; o += nx;
  s.dg = o; o += nx;
  s.dh = o; o += mx;
  s.dk = o; o += mx;  // dh + dG k, then dk
  s.total = o;
  return s;
}

struct Lanes {
  GCVec A, B, M, R, r, c, delta, V, v;
  OptIn dQ, dM, dR, dq, dr, dA, dB, dc, dd;
  OptOut oK, ok, oV, ov;
};

__device__ __forceinline__ OptIn opt_in(const double *p, int64_t b, size_t L) {
  return OptIn{p ? p + b : nullptr, L};
}
__device__ __forceinline__ OptOut opt_out(double *p, int64_t b, size_t L) {
  return OptOut{p ? p + b : nullptr, L};
}

__device__ __forceinline__ Lanes make_lanes(const PolicyVjpIn &in, const LqrIn &t,
                                            const LqrPolicy &o, int64_t b, size_t L) {
  return Lanes{GCVec{in.in.A + b, L},     GCVec{in.in.B + b, L},  GCVec{in.in.M + b, L},
               GCVec{in.in.R + b, L},     GCVec{in.in.r + b, L},  GCVec{in.in.c + b, L},
               GCVec{in.in.delta + b, L}, GCVec{in.V + b, L},     GCVec{in.v + b, L},
               opt_in(t.Q, b, L),         opt_in(t.M, b, L),      opt_in(t.R, b, L),
               opt_in(t.q, b, L),         opt_in(t.r, b, L),      opt_in(t.A, b, L),
               opt_in(t.B, b, L),         opt_in(t.c, b, L),      opt_in(t.delta, b, L),
               opt_out(o.K, b, L),        opt_out(o.k, b, L),     opt_out(o.V, b, L),
               opt_out(o.v, b, L)};
}

// dV_i = sym(dQ_i), dv_i = dq_i into V at vo / vv.
template <class VS>
__device__ __forceinline__ void node_init(const Lanes &l, int n, int nn, int nv, const VS &V,
                                          int vo, int vv) {
  for (int j = 0; j < n; ++j)
    for (int i = j; i < n; ++i) {
      const double x = 0.5 * (l.dQ(nn + i + j * n) + l.dQ(nn + j + i * n));
      V(vo + i + j * n) = x;
      V(vo + j + i * n) = x;
    }
  for (int i = 0; i < n; ++i) V(vv + i) = l.dq(nv + i);
}

// The tangent of edge e (policy_jvp.cuh).  dV_c, dv_c are read at Vc (vco, vcv); the edge's
// terms are added to dV_p, dv_p at Vp (vpo, vpv); dK, dk are written when requested.
template <class S, class VC, class VP>
__device__ __forceinline__ void edge_tangent(const Edge &e, const Slots &s, const S &w,
                                             const Lanes &l, const VC &Vc, int vco, int vcv,
                                             const VP &Vp, int vpo, int vpv) {
  const int np = e.np, nc = e.nc, m = e.m;
  auto A = [&](int i, int j) { return l.A(e.a + i + j * nc); };
  auto B = [&](int i, int a) { return l.B(e.b + i + a * nc); };
  auto dA = [&](int i, int j) { return l.dA(e.a + i + j * nc); };
  auto dB = [&](int i, int a) { return l.dB(e.b + i + a * nc); };
  auto X = [&](int slot, int i, int j, int rows) -> double & { return w(slot + i + j * rows); };

  edge_primal(e, s, w, l);

  // T = dV_c S over Lf;  dW = S' T - W dD W   (S = D^1/2 P D^-1/2)
  for (int j = 0; j < nc; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += Vc(vco + i + k * nc) * (w(s.sd + k) * X(s.P, k, j, nc));
      X(s.Lf, i, j, nc) = t * w(s.sdi + j);
    }
  for (int j = 0; j < nc; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0, u = 0.0;
      for (int k = 0; k < nc; ++k) {
        t += (w(s.sd + k) * X(s.P, k, i, nc)) * X(s.Lf, k, j, nc);
        u += X(s.W, i, k, nc) * l.dd(e.cv + k) * X(s.W, k, j, nc);
      }
      X(s.dW, i, j, nc) = w(s.sdi + i) * t - u;
    }
  // dWB = dW B;  dWA = dW A
  for (int a = 0; a < m; ++a)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.dW, i, k, nc) * B(k, a);
      X(s.dWB, i, a, nc) = t;
    }
  for (int j = 0; j < np; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.dW, i, k, nc) * A(k, j);
      X(s.dWA, i, j, nc) = t;
    }
  // dG = sym(dR) + dB' W B + (W B)' dB + B' dW B;  df
  for (int bb = 0; bb < m; ++bb)
    for (int a = 0; a < m; ++a) {
      double t = 0.5 * (l.dR(e.ro + a + bb * m) + l.dR(e.ro + bb + a * m));
      for (int i = 0; i < nc; ++i)
        t += dB(i, a) * X(s.WB, i, bb, nc) + X(s.WB, i, a, nc) * dB(i, bb) +
             B(i, a) * X(s.dWB, i, bb, nc);
      X(s.dG, a, bb, m) = t;
    }
  for (int i = 0; i < nc; ++i)
    w(s.df + i) = l.dd(e.cv + i) * l.v(e.cv + i) + l.delta(e.cv + i) * Vc(vcv + i) -
                  l.dc(e.cv + i);
  // dY = dWA + W dA;  dg = dv_c - dW f - W df
  for (int j = 0; j < np; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = X(s.dWA, i, j, nc);
      for (int k = 0; k < nc; ++k) t += X(s.W, i, k, nc) * dA(k, j);
      X(s.dY, i, j, nc) = t;
    }
  for (int i = 0; i < nc; ++i) {
    double t = Vc(vcv + i);
    for (int k = 0; k < nc; ++k) t -= X(s.dW, i, k, nc) * w(s.f + k) + X(s.W, i, k, nc) * w(s.df + k);
    w(s.dg + i) = t;
  }
  // dH = dM' + dB' Y + B' dY;  dh = dr + dB' g + B' dg
  for (int j = 0; j < np; ++j)
    for (int a = 0; a < m; ++a) {
      double t = l.dM(e.mo + j + a * np);
      for (int i = 0; i < nc; ++i) t += dB(i, a) * X(s.Y, i, j, nc) + B(i, a) * X(s.dY, i, j, nc);
      X(s.dH, a, j, m) = t;
    }
  for (int a = 0; a < m; ++a) {
    double t = l.dr(e.ru + a);
    for (int i = 0; i < nc; ++i) t += dB(i, a) * w(s.g + i) + B(i, a) * w(s.dg + i);
    w(s.dh + a) = t;
  }
  // dGK = dG K;  dK = -G^-1 (dH + dGK);  dk = -G^-1 (dh + dG k)
  for (int j = 0; j < np; ++j)
    for (int a = 0; a < m; ++a) {
      double t = 0.0;
      for (int bb = 0; bb < m; ++bb) t += X(s.dG, a, bb, m) * X(s.K, bb, j, m);
      X(s.dGK, a, j, m) = t;
      X(s.dK, a, j, m) = X(s.dH, a, j, m) + t;
    }
  for (int a = 0; a < m; ++a) {
    double t = w(s.dh + a);
    for (int bb = 0; bb < m; ++bb) t += X(s.dG, a, bb, m) * w(s.k + bb);
    w(s.dk + a) = t;
  }
  chol_solve(w, s.Lg, m, s.dK, np);
  chol_solve(w, s.Lg, m, s.dk, 1);
  for (int i = 0; i < m * np; ++i) w(s.dK + i) = -w(s.dK + i);
  for (int a = 0; a < m; ++a) w(s.dk + a) = -w(s.dk + a);
  // dV_p += dA' Y + Y' dA + A' dWA + dH' K + K' dH + K' dGK (lower, mirrored)
  for (int j = 0; j < np; ++j)
    for (int i = j; i < np; ++i) {
      double t = 0.0, u = 0.0;
      for (int k = 0; k < nc; ++k)
        t += dA(k, i) * X(s.Y, k, j, nc) + X(s.Y, k, i, nc) * dA(k, j) +
             A(k, i) * X(s.dWA, k, j, nc);
      for (int a = 0; a < m; ++a)
        u += X(s.dH, a, i, m) * X(s.K, a, j, m) + X(s.K, a, i, m) * X(s.dH, a, j, m) +
             X(s.K, a, i, m) * X(s.dGK, a, j, m);
      const double x = Vp(vpo + i + j * np) + (t + u);
      Vp(vpo + i + j * np) = x;
      Vp(vpo + j + i * np) = x;
    }
  // dv_p += dA' g + A' dg + dK' h + K' dh
  for (int i = 0; i < np; ++i) {
    double t = 0.0, u = 0.0;
    for (int k = 0; k < nc; ++k) t += dA(k, i) * w(s.g + k) + A(k, i) * w(s.dg + k);
    for (int a = 0; a < m; ++a) u += X(s.dK, a, i, m) * w(s.h + a) + X(s.K, a, i, m) * w(s.dh + a);
    Vp(vpv + i) += t + u;
  }
  if (l.oK)
    for (int i = 0; i < m * np; ++i) l.oK.set(e.mo + i, w(s.dK + i));
  if (l.ok)
    for (int a = 0; a < m; ++a) l.ok.set(e.ru + a, w(s.dk + a));
}

// Element counts of the four output arrays of one problem.
struct OutSizes {
  int K, k, V, v;
};

__device__ void zero_outputs(const Lanes &l, const OutSizes &z) {
  for (int i = 0; i < z.K; ++i) l.oK.set(i, 0.0);
  for (int i = 0; i < z.k; ++i) l.ok.set(i, 0.0);
  for (int i = 0; i < z.V; ++i) l.oV.set(i, 0.0);
  for (int i = 0; i < z.v; ++i) l.ov.set(i, 0.0);
}

__global__ void __launch_bounds__(kThreads)
policy_jvp_generic_kernel(DevTables t, OutSizes z, Slots s, PolicyVjpIn in, LqrIn tan,
                          LqrPolicy out, double *ws, const int *status, int64_t batch,
                          int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const Lanes l = make_lanes(in, tan, out, b, L);
  if (!(b < batch && status[b] == SIPOC_FACTOR_SUCCESS)) {
    zero_outputs(l, z);
    return;
  }
  const GVec w{ws + b, L};
  // dV of node i at s.total + nn_off[i], dv at s.total + nn_off[N] + n_off[i]
  const int vvo = s.total + t.nn_off[t.N];
  for (int order = 0; order < t.N; ++order) {
    const int p = t.postorder[order];
    const int np = t.n[p], pnn = t.nn_off[p], pv = t.n_off[p];
    node_init(l, np, pnn, pv, w, s.total + pnn, vvo + pv);
    for (int ci = t.child_offsets[p]; ci < t.child_offsets[p + 1]; ++ci) {
      const int e = t.child_edges[ci], c = t.children[e];
      const Edge ed{np,          t.n[c],        t.m[e],      t.a_off[e], t.b_off[e],
                    t.nm_off[e], t.mm_off[e],   t.m_off[e],  pv,         pnn,
                    t.n_off[c],  t.nn_off[c]};
      edge_tangent(ed, s, w, l, w, s.total + ed.cnn, vvo + ed.cv, w, s.total + pnn, vvo + pv);
    }
    if (l.oV)
      for (int i = 0; i < np * np; ++i) l.oV.set(pnn + i, w(s.total + pnn + i));
    if (l.ov)
      for (int i = 0; i < np; ++i) l.ov.set(pv + i, w(vvo + pv + i));
  }
}

// ---------------------------------------------------------------------------------------------
// Sub-warp kernel: LP lanes per problem, 32 / LP problems per warp, one warp per block.  Shared
// memory holds, per problem, the staged operands and every matrix of the edge, interleaved
// across the warp's problems (element idx of problem p at idx * PW + p), so the lanes of one
// problem read the same address (a broadcast) and those of different problems adjacent ones.

// Lanes per problem.  The edge's shared footprint (16 KB per problem at (12, 4), 8.7 KB at
// (8, 4)) bounds the problems in flight per SM, so at large n more lanes per problem shorten
// each one and put more warps on an SM: sixteen at n = 12 (two problems and 32 KB per warp,
// seven warps per SM; eight lanes gave three), eight at n = 6 and 8, four at n = 4.
constexpr int sub_lanes(int n) { return n >= 12 ? 16 : n >= 6 ? 8 : 4; }

// Per-problem shared-memory map (doubles) of one edge.  V_c (lower) is staged straight into
// Lf; dW overwrites dV_c of the child once T = dV_c S is formed; dY overwrites P.
struct SubMap {
  int A, B, M, R, r, c, d, v, dA, dB, dM, dR, dr, dc, dd;  // staged
  int Lf, P, W, Y, dWA, buf0, buf1;                        // n x n; buf: dV (n x n), dv (n)
  int sd, sdi, f, g, df, dg;                               // n
  int WB, dWB, K, dH, dGK, dK;                             // n x m
  int Lg, dG;                                              // m x m
  int h, k, dh, dk;                                        // m
  int total;
};

__host__ __device__ constexpr SubMap make_submap(int n, int m) {
  const int nn = n * n, nm = n * m, mm = m * m;
  SubMap s{};
  int o = 0;
  s.A = o; o += nn;
  s.B = o; o += nm;
  s.M = o; o += nm;
  s.R = o; o += mm;
  s.r = o; o += m;
  s.c = o; o += n;
  s.d = o; o += n;
  s.v = o; o += n;
  s.dA = o; o += nn;
  s.dB = o; o += nm;
  s.dM = o; o += nm;
  s.dR = o; o += mm;
  s.dr = o; o += m;
  s.dc = o; o += n;
  s.dd = o; o += n;
  s.Lf = o; o += nn;
  s.P = o; o += nn;
  s.W = o; o += nn;
  s.Y = o; o += nn;
  s.dWA = o; o += nn;
  s.buf0 = o; o += nn + n;
  s.buf1 = o; o += nn + n;
  s.sd = o; o += n;
  s.sdi = o; o += n;
  s.f = o; o += n;
  s.g = o; o += n;
  s.df = o; o += n;
  s.dg = o; o += n;
  s.WB = o; o += nm;
  s.dWB = o; o += nm;
  s.K = o; o += nm;
  s.dH = o; o += nm;
  s.dGK = o; o += nm;
  s.dK = o; o += nm;
  s.Lg = o; o += mm;
  s.dG = o; o += mm;
  s.h = o; o += m;
  s.k = o; o += m;
  s.dh = o; o += m;
  s.dk = o; o += m;
  s.total = o;
  return s;
}

// One problem's view of the warp's shared map.
template <int PW>
struct Sh {
  double *base;  // the warp's region
  int p;         // problem within the warp
  __device__ __forceinline__ double &operator()(int idx) const { return base[idx * PW + p]; }
};

// out(i, j, f(i, j)) for every element of an R x C result, the lane q of LP owning elements
// q, q + LP, ... (column-major).  All values are formed before any is written, so f may read
// what out overwrites.
template <int R, int C, int LP, class F, class O>
__device__ __forceinline__ void for_elems(int q, const F &f, const O &out) {
  constexpr int T = (R * C + LP - 1) / LP;
  double acc[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int e = q + t * LP;
    acc[t] = e < R * C ? f(e % R, e / R) : 0.0;
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int e = q + t * LP;
    if (e < R * C) out(e % R, e / R, acc[t]);
  }
  __syncwarp();
}

// Lower Cholesky of the n x n matrix at off in place, the rows below each pivot spread over
// the lanes.
template <int n, int LP, int PW>
__device__ __forceinline__ void chol_sub(const Sh<PW> &s, int off, int q) {
  constexpr int T = (n + LP - 1) / LP;
#pragma unroll
  for (int k = 0; k < n; ++k) {
    double x = s(off + k + k * n);
#pragma unroll
    for (int j = 0; j < k; ++j) {
      const double l = s(off + k + j * n);
      x -= l * l;
    }
    x = sqrt(x);
    double col[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int i = k + 1 + q + t * LP;
      double y = 0.0;
      if (i < n) {
        y = s(off + i + k * n);
#pragma unroll
        for (int j = 0; j < k; ++j) y -= s(off + i + j * n) * s(off + k + j * n);
        y /= x;
      }
      col[t] = y;
    }
    __syncwarp();
    if (q == 0) s(off + k + k * n) = x;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int i = k + 1 + q + t * LP;
      if (i < n) s(off + i + k * n) = col[t];
    }
    __syncwarp();
  }
}

// X = (L L')^-1 B for C columns (L: n x n lower at loff), lane q owning columns q, q + LP, ...
// each solved in registers.  B(i, j) = init(i, j); out(i, j, X(i, j)).
template <int n, int C, int LP, int PW, class I, class O>
__device__ __forceinline__ void solve_cols(const Sh<PW> &s, int loff, int q, const I &init,
                                           const O &out) {
  constexpr int T = (C + LP - 1) / LP;
  double x[T][n];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int j = q + t * LP;
#pragma unroll
    for (int i = 0; i < n; ++i) x[t][i] = j < C ? init(i, j) : 0.0;
  }
#pragma unroll
  for (int i = 0; i < n; ++i) {
    const double dinv = 1.0 / s(loff + i + i * n);
#pragma unroll
    for (int t = 0; t < T; ++t) {
      double y = x[t][i];
#pragma unroll
      for (int j = 0; j < i; ++j) y -= s(loff + i + j * n) * x[t][j];
      x[t][i] = y * dinv;
    }
  }
#pragma unroll
  for (int i = n - 1; i >= 0; --i) {
    const double dinv = 1.0 / s(loff + i + i * n);
#pragma unroll
    for (int t = 0; t < T; ++t) {
      double y = x[t][i];
#pragma unroll
      for (int j = i + 1; j < n; ++j) y -= s(loff + j + i * n) * x[t][j];
      x[t][i] = y * dinv;
    }
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int j = q + t * LP;
    if (j < C)
#pragma unroll
      for (int i = 0; i < n; ++i) out(i, j, x[t][i]);
  }
  __syncwarp();
}

__device__ __forceinline__ unsigned smem_u32(const void *p) {
  return static_cast<unsigned>(__cvta_generic_to_shared(p));
}

// Stages count consecutive flat elements from goff of an engine-layout array for the warp's
// PW problems (b0 ..) to the per-problem offset soff: PW adjacent doubles per element, one
// cp.async each.  src nullptr stages zeros.
template <int PW>
__device__ __forceinline__ void stage(double *base, int soff, const double *src, int goff,
                                      int count, int64_t b0, size_t ld, int lane) {
  for (int idx = lane; idx < count * PW; idx += 32) {
    const int f = idx / PW, p = idx % PW;
    double *dst = base + (soff + f) * PW + p;
    if (src == nullptr) {
      *dst = 0.0;
    } else {
      const double *g = src + static_cast<size_t>(goff + f) * ld + b0 + p;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_u32(dst)), "l"(g)
                   : "memory");
    }
  }
}

__device__ __forceinline__ void stage_wait() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
  __syncwarp();
}

// Writes count flat elements from soff to an engine-layout array, zeros for the problems whose
// bit of okmask is clear.
template <int PW>
__device__ __forceinline__ void store(double *dst, int goff, const double *base, int soff,
                                      int count, int64_t b0, size_t ld, unsigned okmask,
                                      int lane) {
  if (dst == nullptr) return;
  for (int idx = lane; idx < count * PW; idx += 32) {
    const int f = idx / PW, p = idx % PW;
    const double x = base[(soff + f) * PW + p];
    dst[static_cast<size_t>(goff + f) * ld + b0 + p] = (okmask >> p) & 1u ? x : 0.0;
  }
}

template <int N, int M>
__global__ void __launch_bounds__(32, 1)
policy_jvp_subwarp(PolicyVjpIn in, LqrIn tan, LqrPolicy out, const int *status, int E,
                   int64_t batch, int64_t ld) {
  constexpr int LP = sub_lanes(N), PW = 32 / LP;
  constexpr int NN = N * N, NM = N * M, MM = M * M;
  constexpr SubMap m = make_submap(N, M);
  extern __shared__ double smem[];
  const int lane = threadIdx.x, q = lane % LP;
  const int64_t b0 = static_cast<int64_t>(blockIdx.x) * PW;
  const size_t L = static_cast<size_t>(ld);
  const Sh<PW> s{smem, lane / LP};
  unsigned okmask = 0;
  if (lane < PW) {
    const int64_t b = b0 + lane;
    okmask = b < batch && status[b] == SIPOC_FACTOR_SUCCESS ? 1u : 0u;
  }
  okmask = __ballot_sync(0xffffffffu, okmask != 0);

  auto X = [&](int off, int i, int j, int rows) -> double & { return s(off + i + j * rows); };
  auto sym_node = [&](int buf) {  // dV = sym(dQ) in place
    for_elems<N, N, LP>(
        q, [&](int i, int j) { return 0.5 * (X(buf, i, j, N) + X(buf, j, i, N)); },
        [&](int i, int j, double x) { X(buf, i, j, N) = x; });
  };
  auto store_node = [&](int node, int buf) {
    store<PW>(out.V, node * NN, smem, buf, NN, b0, L, okmask, lane);
    store<PW>(out.v, node * N, smem, buf + NN, N, b0, L, okmask, lane);
    __syncwarp();
  };

  // the last node: dV_E = sym(dQ_E), dv_E = dq_E
  {
    const int buf = E & 1 ? m.buf1 : m.buf0;
    stage<PW>(smem, buf, tan.Q, E * NN, NN, b0, L, lane);
    stage<PW>(smem, buf + NN, tan.q, E * N, N, b0, L, lane);
    stage_wait();
    sym_node(buf);
    store_node(E, buf);
  }
#pragma unroll 1
  for (int e = E - 1; e >= 0; --e) {
    const int c = e + 1;
    const int cur = c & 1 ? m.buf1 : m.buf0, nxt = c & 1 ? m.buf0 : m.buf1;
    // ---- stage the edge's operands, V_c (lower) into Lf, dQ_p / dq_p into the parent's buffer
    stage<PW>(smem, m.A, in.in.A, e * NN, NN, b0, L, lane);
    stage<PW>(smem, m.B, in.in.B, e * NM, NM, b0, L, lane);
    stage<PW>(smem, m.M, in.in.M, e * NM, NM, b0, L, lane);
    stage<PW>(smem, m.R, in.in.R, e * MM, MM, b0, L, lane);
    stage<PW>(smem, m.r, in.in.r, e * M, M, b0, L, lane);
    stage<PW>(smem, m.c, in.in.c, c * N, N, b0, L, lane);
    stage<PW>(smem, m.d, in.in.delta, c * N, N, b0, L, lane);
    stage<PW>(smem, m.v, in.v, c * N, N, b0, L, lane);
#pragma unroll 1
    for (int j = 0; j < N; ++j)
      stage<PW>(smem, m.Lf + j + j * N, in.V, c * NN + j + j * N, N - j, b0, L, lane);
    stage<PW>(smem, m.dA, tan.A, e * NN, NN, b0, L, lane);
    stage<PW>(smem, m.dB, tan.B, e * NM, NM, b0, L, lane);
    stage<PW>(smem, m.dM, tan.M, e * NM, NM, b0, L, lane);
    stage<PW>(smem, m.dR, tan.R, e * MM, MM, b0, L, lane);
    stage<PW>(smem, m.dr, tan.r, e * M, M, b0, L, lane);
    stage<PW>(smem, m.dc, tan.c, c * N, N, b0, L, lane);
    stage<PW>(smem, m.dd, tan.delta, c * N, N, b0, L, lane);
    stage<PW>(smem, nxt, tan.Q, e * NN, NN, b0, L, lane);
    stage<PW>(smem, nxt + NN, tan.q, e * N, N, b0, L, lane);
    stage_wait();
    sym_node(nxt);

    auto A = [&](int i, int j) -> double & { return X(m.A, i, j, N); };
    auto B = [&](int i, int a) -> double & { return X(m.B, i, a, N); };
    auto dA = [&](int i, int j) -> double & { return X(m.dA, i, j, N); };
    auto dB = [&](int i, int a) -> double & { return X(m.dB, i, a, N); };
    auto W = [&](int i, int j) -> double & { return X(m.W, i, j, N); };
    auto Y = [&](int i, int j) -> double & { return X(m.Y, i, j, N); };
    auto P = [&](int i, int j) -> double & { return X(m.P, i, j, N); };
    auto K = [&](int a, int j) -> double & { return X(m.K, a, j, M); };
    auto dH = [&](int a, int j) -> double & { return X(m.dH, a, j, M); };
    auto dW = [&](int i, int j) -> double & { return X(cur, i, j, N); };  // over dV_c
    auto vec = [&](int off, int i) -> double & { return s(off + i); };

    // ---- primal.  sd, sdi;  F = I + D^1/2 V_c D^1/2 (lower), its Cholesky factor
    for_elems<N, 1, LP>(
        q, [&](int i, int) { return sqrt(vec(m.d, i)); },
        [&](int i, int, double x) {
          vec(m.sd, i) = x;
          vec(m.sdi, i) = 1.0 / x;
        });
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          return i >= j ? vec(m.sd, i) * X(m.Lf, i, j, N) * vec(m.sd, j) + (i == j ? 1.0 : 0.0)
                        : 0.0;
        },
        [&](int i, int j, double x) {
          if (i >= j) X(m.Lf, i, j, N) = x;
        });
    chol_sub<N, LP>(s, m.Lf, q);
    // P = F^-1 (its lower triangle mirrored), W = D^-1/2 (I - P) D^-1/2
    solve_cols<N, N, LP>(
        s, m.Lf, q, [](int i, int j) { return i == j ? 1.0 : 0.0; },
        [&](int i, int j, double x) { P(i, j) = x; });
    for_elems<N, N, LP>(
        q, [&](int i, int j) { return i >= j ? P(i, j) : P(j, i); },
        [&](int i, int j, double x) {
          P(i, j) = x;
          W(i, j) = vec(m.sdi, i) * ((i == j ? 1.0 : 0.0) - x) * vec(m.sdi, j);
        });
    // WB = W B;  Y = W A
    for_elems<N, M, LP>(
        q,
        [&](int i, int a) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += W(i, k) * B(k, a);
          return t;
        },
        [&](int i, int a, double x) { X(m.WB, i, a, N) = x; });
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += W(i, k) * A(k, j);
          return t;
        },
        [&](int i, int j, double x) { Y(i, j) = x; });
    // G = R + B' WB, its Cholesky factor;  f = delta .* v - c
    for_elems<M, M, LP>(
        q,
        [&](int a, int bb) {
          double t = X(m.R, a, bb, M);
#pragma unroll
          for (int i = 0; i < N; ++i) t += B(i, a) * X(m.WB, i, bb, N);
          return t;
        },
        [&](int a, int bb, double x) { X(m.Lg, a, bb, M) = x; });
    for_elems<N, 1, LP>(
        q, [&](int i, int) { return vec(m.d, i) * vec(m.v, i) - vec(m.c, i); },
        [&](int i, int, double x) { vec(m.f, i) = x; });
    chol_sub<M, LP>(s, m.Lg, q);
    // g = v - W f
    for_elems<N, 1, LP>(
        q,
        [&](int i, int) {
          double t = vec(m.v, i);
#pragma unroll
          for (int k = 0; k < N; ++k) t -= W(i, k) * vec(m.f, k);
          return t;
        },
        [&](int i, int, double x) { vec(m.g, i) = x; });
    // H = M' + B' Y (over K);  h = r + B' g
    for_elems<M, N, LP>(
        q,
        [&](int a, int j) {
          double t = X(m.M, j, a, N);
#pragma unroll
          for (int i = 0; i < N; ++i) t += B(i, a) * Y(i, j);
          return t;
        },
        [&](int a, int j, double x) { K(a, j) = x; });
    for_elems<M, 1, LP>(
        q,
        [&](int a, int) {
          double t = vec(m.r, a);
#pragma unroll
          for (int i = 0; i < N; ++i) t += B(i, a) * vec(m.g, i);
          return t;
        },
        [&](int a, int, double x) { vec(m.h, a) = x; });
    // K = -G^-1 H;  k = -G^-1 h
    solve_cols<M, N, LP>(
        s, m.Lg, q, [&](int a, int j) { return K(a, j); },
        [&](int a, int j, double x) { K(a, j) = -x; });
    solve_cols<M, 1, LP>(
        s, m.Lg, q, [&](int a, int) { return vec(m.h, a); },
        [&](int a, int, double x) { vec(m.k, a) = -x; });

    // ---- tangent.  T = dV_c S over Lf;  dW = S' T - W dD W over dV_c
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += X(cur, i, k, N) * (vec(m.sd, k) * P(k, j));
          return t * vec(m.sdi, j);
        },
        [&](int i, int j, double x) { X(m.Lf, i, j, N) = x; });
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          double t = 0.0, u = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) {
            t += (vec(m.sd, k) * P(k, i)) * X(m.Lf, k, j, N);
            u += W(i, k) * vec(m.dd, k) * W(k, j);
          }
          return vec(m.sdi, i) * t - u;
        },
        [&](int i, int j, double x) { dW(i, j) = x; });
    // dWB = dW B;  dWA = dW A
    for_elems<N, M, LP>(
        q,
        [&](int i, int a) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += dW(i, k) * B(k, a);
          return t;
        },
        [&](int i, int a, double x) { X(m.dWB, i, a, N) = x; });
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          double t = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += dW(i, k) * A(k, j);
          return t;
        },
        [&](int i, int j, double x) { X(m.dWA, i, j, N) = x; });
    // dG = sym(dR) + dB' WB + WB' dB + B' dWB;  df
    for_elems<M, M, LP>(
        q,
        [&](int a, int bb) {
          double t = 0.5 * (X(m.dR, a, bb, M) + X(m.dR, bb, a, M));
#pragma unroll
          for (int i = 0; i < N; ++i)
            t += dB(i, a) * X(m.WB, i, bb, N) + X(m.WB, i, a, N) * dB(i, bb) +
                 B(i, a) * X(m.dWB, i, bb, N);
          return t;
        },
        [&](int a, int bb, double x) { X(m.dG, a, bb, M) = x; });
    for_elems<N, 1, LP>(
        q,
        [&](int i, int) {
          return vec(m.dd, i) * vec(m.v, i) + vec(m.d, i) * s(cur + NN + i) - vec(m.dc, i);
        },
        [&](int i, int, double x) { vec(m.df, i) = x; });
    // dY = dWA + W dA (over P);  dg = dv_c - dW f - W df
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          double t = X(m.dWA, i, j, N);
#pragma unroll
          for (int k = 0; k < N; ++k) t += W(i, k) * dA(k, j);
          return t;
        },
        [&](int i, int j, double x) { P(i, j) = x; });
    for_elems<N, 1, LP>(
        q,
        [&](int i, int) {
          double t = s(cur + NN + i);
#pragma unroll
          for (int k = 0; k < N; ++k) t -= dW(i, k) * vec(m.f, k) + W(i, k) * vec(m.df, k);
          return t;
        },
        [&](int i, int, double x) { vec(m.dg, i) = x; });
    // dH = dM' + dB' Y + B' dY;  dh = dr + dB' g + B' dg
    for_elems<M, N, LP>(
        q,
        [&](int a, int j) {
          double t = X(m.dM, j, a, N);
#pragma unroll
          for (int i = 0; i < N; ++i) t += dB(i, a) * Y(i, j) + B(i, a) * P(i, j);
          return t;
        },
        [&](int a, int j, double x) { dH(a, j) = x; });
    for_elems<M, 1, LP>(
        q,
        [&](int a, int) {
          double t = vec(m.dr, a);
#pragma unroll
          for (int i = 0; i < N; ++i) t += dB(i, a) * vec(m.g, i) + B(i, a) * vec(m.dg, i);
          return t;
        },
        [&](int a, int, double x) { vec(m.dh, a) = x; });
    // dGK = dG K;  dK = -G^-1 (dH + dGK);  dk = -G^-1 (dh + dG k)
    for_elems<M, N, LP>(
        q,
        [&](int a, int j) {
          double t = 0.0;
#pragma unroll
          for (int bb = 0; bb < M; ++bb) t += X(m.dG, a, bb, M) * K(bb, j);
          return t;
        },
        [&](int a, int j, double x) { X(m.dGK, a, j, M) = x; });
    solve_cols<M, N, LP>(
        s, m.Lg, q, [&](int a, int j) { return dH(a, j) + X(m.dGK, a, j, M); },
        [&](int a, int j, double x) { X(m.dK, a, j, M) = -x; });
    solve_cols<M, 1, LP>(
        s, m.Lg, q,
        [&](int a, int) {
          double t = vec(m.dh, a);
#pragma unroll
          for (int bb = 0; bb < M; ++bb) t += X(m.dG, a, bb, M) * vec(m.k, bb);
          return t;
        },
        [&](int a, int, double x) { vec(m.dk, a) = -x; });
    // dV_p += dA' Y + Y' dA + A' dWA + dH' K + K' dH + K' dGK (lower, mirrored)
    for_elems<N, N, LP>(
        q,
        [&](int i, int j) {
          if (i < j) return 0.0;
          double t = 0.0, u = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k)
            t += dA(k, i) * Y(k, j) + Y(k, i) * dA(k, j) + A(k, i) * X(m.dWA, k, j, N);
#pragma unroll
          for (int a = 0; a < M; ++a)
            u += dH(a, i) * K(a, j) + K(a, i) * dH(a, j) + K(a, i) * X(m.dGK, a, j, M);
          return X(nxt, i, j, N) + (t + u);
        },
        [&](int i, int j, double x) {
          if (i >= j) {
            X(nxt, i, j, N) = x;
            X(nxt, j, i, N) = x;
          }
        });
    // dv_p += dA' g + A' dg + dK' h + K' dh
    for_elems<N, 1, LP>(
        q,
        [&](int i, int) {
          double t = 0.0, u = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) t += dA(k, i) * vec(m.g, k) + A(k, i) * vec(m.dg, k);
#pragma unroll
          for (int a = 0; a < M; ++a) u += X(m.dK, a, i, M) * vec(m.h, a) + K(a, i) * vec(m.dh, a);
          return s(nxt + NN + i) + (t + u);
        },
        [&](int i, int, double x) { s(nxt + NN + i) = x; });

    store<PW>(out.K, e * NM, smem, m.dK, NM, b0, L, okmask, lane);
    store<PW>(out.k, e * M, smem, m.dk, M, b0, L, okmask, lane);
    store_node(e, nxt);
  }
}

template <int N, int M>
bool subwarp(int E, const PolicyVjpIn &in, const LqrIn &tan, const LqrPolicy &out,
             const int *status, int64_t batch, int64_t ld, cudaStream_t s) {
  constexpr int PW = 32 / sub_lanes(N);
  constexpr size_t bytes = sizeof(double) * PW * make_submap(N, M).total;
  // once per instance, on the first (eager) call: the attribute is not a stream operation
  static const cudaError_t attr = cudaFuncSetAttribute(
      policy_jvp_subwarp<N, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
  if (attr != cudaSuccess) return false;
  policy_jvp_subwarp<N, M><<<static_cast<unsigned>(ld / PW), 32, bytes, s>>>(
      in, tan, out, status, E, batch, ld);
  return true;
}

}  // namespace

int64_t policy_jvp_generic_ws_elems(const HostStructure &h) {
  return make_slots(h.max_n, h.max_m).total + h.nn_off[h.N] + h.n_off[h.N];
}

bool policy_jvp_subwarp_shape(int n, int m) {
  return ((n == 4 || n == 6 || n == 8) && m >= 1 && m <= 4) || (n == 12 && m == 4);
}

bool launch_policy_jvp_subwarp(int n, int m, int E, const PolicyVjpIn &in, const LqrIn &tan,
                               const LqrPolicy &out, const int *status, int64_t batch,
                               int64_t ld, cudaStream_t s) {
#define SIPOC_PJVP(NN, MM) \
  if (n == NN && m == MM) return subwarp<NN, MM>(E, in, tan, out, status, batch, ld, s);
  SIPOC_PJVP(4, 1) SIPOC_PJVP(4, 2) SIPOC_PJVP(4, 3) SIPOC_PJVP(4, 4)
  SIPOC_PJVP(6, 1) SIPOC_PJVP(6, 2) SIPOC_PJVP(6, 3) SIPOC_PJVP(6, 4)
  SIPOC_PJVP(8, 1) SIPOC_PJVP(8, 2) SIPOC_PJVP(8, 3) SIPOC_PJVP(8, 4)
  SIPOC_PJVP(12, 4)
#undef SIPOC_PJVP
  return false;
}

void launch_policy_jvp_generic(const DevTables &t, const HostStructure &h, const PolicyVjpIn &in,
                               const LqrIn &tan, const LqrPolicy &out, double *ws,
                               const int *status, int64_t batch, int64_t ld, cudaStream_t s) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  const OutSizes z{h.nm_off[h.E], h.m_off[h.E], h.nn_off[h.N], h.n_off[h.N]};
  policy_jvp_generic_kernel<<<static_cast<unsigned>((ld + threads - 1) / threads), threads, 0,
                              s>>>(t, z, make_slots(h.max_n, h.max_m), in, tan, out, ws, status,
                                   batch, ld);
}

}  // namespace sipoc
