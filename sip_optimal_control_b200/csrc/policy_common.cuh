// Per-edge pieces the two derivative sweeps of the policy share (policy_vjp.cu, policy_jvp.cu):
// optional lanes, the small Cholesky routines, the flat offsets of an edge, and the primal
// recompute of one edge of the Riccati recursion from the inputs and the forward's V_c, v_c.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>

namespace sipoc {
namespace policy_detail {

// Optional read-only lane: nullptr reads as zero, so a NULL array is bitwise a zero one.
struct OptIn {
  const double *p;
  size_t ld;
  __device__ __forceinline__ double operator()(int i) const {
    return p != nullptr ? __ldg(p + static_cast<size_t>(i) * ld) : 0.0;
  }
};

// Optional output lane: nullptr is neither computed nor written.
struct OptOut {
  double *p;
  size_t ld;
  __device__ __forceinline__ explicit operator bool() const { return p != nullptr; }
  __device__ __forceinline__ void set(int i, double v) const {
    if (p != nullptr) p[static_cast<size_t>(i) * ld] = v;
  }
};

// Lower Cholesky in place (left-looking, as chol_lower of generic_kernels.cu).  The forward
// factored the same matrix successfully, so no pivot test.
template <class S>
__device__ __forceinline__ void chol(const S &a, int off, int n) {
  for (int k = 0; k < n; ++k) {
    double x = a(off + k + k * n);
    for (int j = 0; j < k; ++j) {
      const double l = a(off + k + j * n);
      x -= l * l;
    }
    x = sqrt(x);
    a(off + k + k * n) = x;
    for (int i = k + 1; i < n; ++i) {
      double s = a(off + i + k * n);
      for (int j = 0; j < k; ++j) s -= a(off + i + j * n) * a(off + k + j * n);
      a(off + i + k * n) = s / x;
    }
  }
}

// L L' X = B in place, nrhs columns of n rows.
template <class S>
__device__ __forceinline__ void chol_solve(const S &a, int loff, int n, int boff, int nrhs) {
  for (int c = 0; c < nrhs; ++c) {
    const int xo = boff + c * n;
    for (int i = 0; i < n; ++i) {
      double s = a(xo + i);
      for (int j = 0; j < i; ++j) s -= a(loff + i + j * n) * a(xo + j);
      a(xo + i) = s / a(loff + i + i * n);
    }
    for (int i = n - 1; i >= 0; --i) {
      double s = a(xo + i);
      for (int j = i + 1; j < n; ++j) s -= a(loff + j + i * n) * a(xo + j);
      a(xo + i) = s / a(loff + i + i * n);
    }
  }
}

// Flat offsets of one edge and its two nodes.
struct Edge {
  int np, nc, m;
  int a, b, mo, ro, ru;  // A, B, M (and K), R, r (and k)
  int pv, pnn;           // parent: n_off, nn_off
  int cv, cnn;           // child
};

// The primal of edge e, recomputed from the inputs and the forward's V_c (lower), v_c:
//   P_c = (I + D^1/2 V_c D^1/2)^-1   W_c = D^-1/2 (I - P_c) D^-1/2   (D = diag(delta_c))
//   WB = W_c B   G = R + B' W_c B (Cholesky factor at s.Lg)   Y = W_c A   K = -G^-1 (M' + B' Y)
//   f = delta_c .* v_c - c_c   g = v_c - W_c f   h = r + B' g   k = -G^-1 h
// into the scratch w at the slots of s (sd, sdi, Lf, P, W, WB, Lg, Y, K, f, g, h, k; P and W
// both triangles).  l reads A, B, M, R, r, c, delta, V, v.
template <class Sl, class S, class L>
__device__ __forceinline__ void edge_primal(const Edge &e, const Sl &s, const S &w, const L &l) {
  const int np = e.np, nc = e.nc, m = e.m;
  auto A = [&](int i, int j) { return l.A(e.a + i + j * nc); };
  auto B = [&](int i, int a) { return l.B(e.b + i + a * nc); };
  auto X = [&](int slot, int i, int j, int rows) -> double & { return w(slot + i + j * rows); };

  // P_c = F^-1, F = I + D^1/2 V_c D^1/2 (lower of V_c); W_c = D^-1/2 (I - P_c) D^-1/2
  for (int i = 0; i < nc; ++i) {
    const double sd = sqrt(l.delta(e.cv + i));
    w(s.sd + i) = sd;
    w(s.sdi + i) = 1.0 / sd;
  }
  for (int j = 0; j < nc; ++j)
    for (int i = j; i < nc; ++i)
      X(s.Lf, i, j, nc) =
          w(s.sd + i) * l.V(e.cnn + i + j * nc) * w(s.sd + j) + (i == j ? 1.0 : 0.0);
  chol(w, s.Lf, nc);
  for (int j = 0; j < nc; ++j)
    for (int i = 0; i < nc; ++i) X(s.P, i, j, nc) = i == j ? 1.0 : 0.0;
  chol_solve(w, s.Lf, nc, s.P, nc);
  for (int j = 0; j < nc; ++j)
    for (int i = j; i < nc; ++i) {
      const double pij = X(s.P, i, j, nc);
      X(s.P, j, i, nc) = pij;
      const double wij = w(s.sdi + i) * ((i == j ? 1.0 : 0.0) - pij) * w(s.sdi + j);
      X(s.W, i, j, nc) = wij;
      X(s.W, j, i, nc) = wij;
    }
  // WB = W_c B;  G = R + B' W_c B (lower of R), its Cholesky factor
  for (int a = 0; a < m; ++a)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.W, i, k, nc) * B(k, a);
      X(s.WB, i, a, nc) = t;
    }
  for (int bb = 0; bb < m; ++bb)
    for (int a = bb; a < m; ++a) {
      double t = l.R(e.ro + a + bb * m);
      for (int i = 0; i < nc; ++i) t += B(i, a) * X(s.WB, i, bb, nc);
      X(s.Lg, a, bb, m) = t;
    }
  chol(w, s.Lg, m);
  // Y = W_c A;  K = -G^-1 (M' + B' Y)
  for (int j = 0; j < np; ++j)
    for (int i = 0; i < nc; ++i) {
      double t = 0.0;
      for (int k = 0; k < nc; ++k) t += X(s.W, i, k, nc) * A(k, j);
      X(s.Y, i, j, nc) = t;
    }
  for (int j = 0; j < np; ++j)
    for (int a = 0; a < m; ++a) {
      double t = l.M(e.mo + j + a * np);
      for (int i = 0; i < nc; ++i) t += B(i, a) * X(s.Y, i, j, nc);
      X(s.K, a, j, m) = t;
    }
  chol_solve(w, s.Lg, m, s.K, np);
  for (int i = 0; i < m * np; ++i) w(s.K + i) = -w(s.K + i);
  // f, g, h;  k = -G^-1 h
  for (int i = 0; i < nc; ++i)
    w(s.f + i) = l.delta(e.cv + i) * l.v(e.cv + i) - l.c(e.cv + i);
  for (int i = 0; i < nc; ++i) {
    double t = l.v(e.cv + i);
    for (int k = 0; k < nc; ++k) t -= X(s.W, i, k, nc) * w(s.f + k);
    w(s.g + i) = t;
  }
  for (int a = 0; a < m; ++a) {
    double t = l.r(e.ru + a);
    for (int i = 0; i < nc; ++i) t += B(i, a) * w(s.g + i);
    w(s.h + a) = t;
    w(s.k + a) = t;
  }
  chol_solve(w, s.Lg, m, s.k, 1);
  for (int a = 0; a < m; ++a) w(s.k + a) = -w(s.k + a);
}

}  // namespace policy_detail
}  // namespace sipoc
