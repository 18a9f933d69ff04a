// Tangent right-hand sides of the LQR and Newton-KKT JVPs (see jvp.cuh for the formulas).
//
// Mapping, as in the VJP kernels: threads go across problems (engine layout X[flat * ld + b]),
// so every load and store of a warp is 32 consecutive doubles, and a grid-stride loop over
// the rows of the grid (blockIdx.y) walks the items.  An item is one node together with its
// child edges: it owns the rows of t of its node and of those edges (LQR: x_i, and u_e, y_c
// of every child edge e -> c; KKT: the node's and the edges' segments of [x | y | z], y_dyn of
// the children included), and the root's item also owns the root's y / y_dyn rows.  Every
// tangent block then touches only rows its item owns, so one read of the block serves both
// products it enters (D v into its row range, D' w into its column range, gemv2), and each
// thread accumulates into its own lane of t in a fixed order: no atomics, and the result is
// bitwise repeatable.  The KKT theta rows are a sum over every node and edge; the last item
// walks the structure in index order for them, so the theta blocks are read twice (once for
// their rows, once for the theta rows).
#include "jvp.cuh"

#include <algorithm>

#include "kkt_blocks.cuh"
#include "vjp_common.cuh"

namespace sipoc {

namespace {

constexpr int kThreads = 128;
constexpr int kRows = 8;  // rows of a block held in registers
constexpr int kMaxGridY = 65535;

using vjp::Lane;

// A tangent array's lane; a NULL array reads as zero and is never dereferenced.
__device__ __forceinline__ Lane lane(const double *p, int64_t b, size_t ld, bool live) {
  return Lane{p != nullptr ? p + b : nullptr, ld, live && p != nullptr};
}

// Both products of one tangent block D (rows x cols, column-major at element off) from one
// read of it:  out_r[orow + i] += s sum_j D_ij vc(cb + j)  and  out_c[ocol + j] += s sum_i
// D_ij vr(ra + i).  out_r / out_c == nullptr: that product is not accumulated.  out_r and
// out_c may be the same rows (a symmetric block's two halves).
__device__ __forceinline__ void gemv2(const Lane &D, size_t ld, int off, int rows, int cols,
                                      const Lane &vr, int ra, const Lane &vc, int cb,
                                      double *out_r, int orow, double *out_c, int ocol,
                                      double s) {
  for (int i0 = 0; i0 < rows; i0 += kRows) {
    double acc[kRows], vi[kRows];
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      acc[k] = 0.0;
      vi[k] = i0 + k < rows ? vr(ra + i0 + k) : 0.0;
    }
    for (int j = 0; j < cols; ++j) {
      const double vj = vc(cb + j);
      const int col = off + i0 + j * rows;
      double cs = 0.0;
#pragma unroll
      for (int k = 0; k < kRows; ++k)
        if (i0 + k < rows) {
          const double d = D(col + k);
          acc[k] += d * vj;
          cs += d * vi[k];
        }
      if (out_c != nullptr) out_c[static_cast<size_t>(ocol + j) * ld] += s * cs;
    }
    if (out_r != nullptr) {
#pragma unroll
      for (int k = 0; k < kRows; ++k)
        if (i0 + k < rows) out_r[static_cast<size_t>(orow + i0 + k) * ld] += s * acc[k];
    }
  }
}

// ---- LQR ---------------------------------------------------------------------------------

__device__ __forceinline__ void lqr_copy(double *T, size_t ld, int o, int n, const Lane &v) {
  for (int k = 0; k < n; ++k) T[static_cast<size_t>(o + k) * ld] = v(o + k);
}

// The dynamics rows of node c before the blocks: dc_c - ddelta_c .* y_c.
__device__ __forceinline__ void lqr_y_rows(double *T, size_t ld, int o, int n, const Lane &dc,
                                           const Lane &ddelta, const Lane &y) {
  for (int k = 0; k < n; ++k) T[static_cast<size_t>(o + k) * ld] = dc(o + k) - ddelta(o + k) * y(o + k);
}

__global__ void __launch_bounds__(kThreads)
lqr_jvp_kernel(DevTables t, LqrOut sol, LqrTangent d, LqrOut rhs, int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch;
  const Lane x{sol.x + b, L, live}, u{sol.u + b, L, live}, y{sol.y + b, L, live};
  const Lane dq = lane(d.q, b, L, live), dr = lane(d.r, b, L, live), dc = lane(d.c, b, L, live),
             ddelta = lane(d.delta, b, L, live);
  double *tx = rhs.x + b, *tu = rhs.u + b, *ty = rhs.y + b;

  for (int i = blockIdx.y; i < t.N; i += gridDim.y) {
    const int n = t.n[i], o = t.n_off[i];
    const int c0 = t.child_offsets[i], c1 = t.child_offsets[i + 1];
    lqr_copy(tx, L, o, n, dq);
    if (i == t.root) lqr_y_rows(ty, L, o, n, dc, ddelta, y);
    for (int ce = c0; ce < c1; ++ce) {
      const int e = t.child_edges[ce], c = t.children[e];
      lqr_copy(tu, L, t.m_off[e], t.m[e], dr);
      lqr_y_rows(ty, L, t.n_off[c], t.n[c], dc, ddelta, y);
    }
    if (d.Q) gemv2(lane(d.Q, b, L, live), L, t.nn_off[i], n, n, x, o, x, o, tx, o, tx, o, 0.5);
    for (int ce = c0; ce < c1; ++ce) {
      const int e = t.child_edges[ce], c = t.children[e];
      const int m = t.m[e], nc = t.n[c], ou = t.m_off[e], oc = t.n_off[c];
      // M_e at (x_p, u_e), R_e at (u_e, u_e), A_e at (y_c, x_p), B_e at (y_c, u_e)
      if (d.M) gemv2(lane(d.M, b, L, live), L, t.nm_off[e], n, m, x, o, u, ou, tx, o, tu, ou, 1.0);
      if (d.R) gemv2(lane(d.R, b, L, live), L, t.mm_off[e], m, m, u, ou, u, ou, tu, ou, tu, ou, 0.5);
      if (d.A) gemv2(lane(d.A, b, L, live), L, t.a_off[e], nc, n, y, oc, x, o, ty, oc, tx, o, 1.0);
      if (d.B) gemv2(lane(d.B, b, L, live), L, t.b_off[e], nc, m, y, oc, u, ou, ty, oc, tu, ou, 1.0);
    }
  }
}

// ---- Newton-KKT ---------------------------------------------------------------------------

// The rows [o, o + n) of t = db - dK sol before the blocks: db and the regularization term
// of the part of [x | y | z] they lie in (-dr1 .* s, +dr2 .* s or +(dw + dr3) .* s).
__device__ __forceinline__ void kkt_rows(const DevTables &t, double *T, size_t ld, int o, int n,
                                         const Lane &sol, const Lane &db, const Lane &dw,
                                         const Lane &dr1, const Lane &dr2, const Lane &dr3) {
  const int xd = t.x_dim, zd = t.x_dim + t.y_dim;
  for (int k = 0; k < n; ++k) {
    const int r = o + k;
    double v;
    if (r < xd) v = db(r) - dr1(r) * sol(r);
    else if (r < zd) v = db(r) + dr2(r - xd) * sol(r);
    else v = db(r) + (dw(r - zd) + dr3(r - zd)) * sol(r);
    T[static_cast<size_t>(r) * ld] = v;
  }
}

// t[ra:] -= D sol[cb:] (rows) and t[cb:] -= D' sol[ra:] (cols), scaled as the table says.
__device__ __forceinline__ void kkt_block(const KktBlock<const double *> &k, int64_t b, size_t ld,
                                          bool live, const Lane &sol, double *T, bool rows,
                                          bool cols) {
  if (k.G == nullptr || k.rows <= 0 || k.cols <= 0) return;
  gemv2(lane(k.G, b, ld, live), ld, k.off, k.rows, k.cols, sol, k.ra, sol, k.cb,
        rows ? T : nullptr, k.ra, cols ? T : nullptr, k.cb, k.s);
}

__global__ void __launch_bounds__(kThreads)
kkt_jvp_kernel(DevTables t, const double *sol_p, KktTangent d, double *rhs, int64_t batch,
               int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch;
  const Lane sol{sol_p + b, L, live};
  const Lane db = lane(d.b, b, L, live), dw = lane(d.w, b, L, live), dr1 = lane(d.r1, b, L, live),
             dr2 = lane(d.r2, b, L, live), dr3 = lane(d.r3, b, L, live);
  double *T = rhs + b;
  const int xd = t.x_dim, zd = t.x_dim + t.y_dim;

  for (int item = blockIdx.y; item <= t.N; item += gridDim.y) {
    if (item < t.N) {
      const int i = item, c0 = t.child_offsets[i], c1 = t.child_offsets[i + 1];
      kkt_rows(t, T, L, t.x_state[i], t.n[i], sol, db, dw, dr1, dr2, dr3);
      kkt_rows(t, T, L, xd + t.y_node_c[i], t.node_c[i], sol, db, dw, dr1, dr2, dr3);
      kkt_rows(t, T, L, zd + t.z_node[i], t.node_g[i], sol, db, dw, dr1, dr2, dr3);
      if (i == t.root) kkt_rows(t, T, L, xd + t.y_dyn[i], t.n[i], sol, db, dw, dr1, dr2, dr3);
      for (int ce = c0; ce < c1; ++ce) {
        const int e = t.child_edges[ce], c = t.children[e];
        kkt_rows(t, T, L, t.x_control[e], t.m[e], sol, db, dw, dr1, dr2, dr3);
        kkt_rows(t, T, L, xd + t.y_dyn[c], t.n[c], sol, db, dw, dr1, dr2, dr3);
        kkt_rows(t, T, L, xd + t.y_edge_c[e], t.edge_c[e], sol, db, dw, dr1, dr2, dr3);
        kkt_rows(t, T, L, zd + t.z_edge[e], t.edge_g[e], sol, db, dw, dr1, dr2, dr3);
      }
      // the theta blocks add only to their own rows here; theta x theta is the last item's
#pragma unroll 1
      for (int k = 0; k < kKktNodeHtt; ++k)
        kkt_block(kkt_node_block(t, d, k, i), b, L, live, sol, T, true, k < kKktNodeTheta);
      for (int ce = c0; ce < c1; ++ce) {
        const int e = t.child_edges[ce];
#pragma unroll 1
        for (int k = 0; k < kKktEdgeHtt; ++k)
          kkt_block(kkt_edge_block(t, d, k, e), b, L, live, sol, T, true, k < kKktEdgeTheta);
      }
    } else if (t.theta_dim > 0) {  // the theta rows: every theta block, in index order
      kkt_rows(t, T, L, t.sx_dim, t.theta_dim, sol, db, dw, dr1, dr2, dr3);
      for (int i = 0; i < t.N; ++i) {
#pragma unroll 1
        for (int k = kKktNodeTheta; k <= kKktNodeHtt; ++k)
          kkt_block(kkt_node_block(t, d, k, i), b, L, live, sol, T, k == kKktNodeHtt, true);
      }
      for (int e = 0; e < t.E; ++e) {
#pragma unroll 1
        for (int k = kKktEdgeTheta; k <= kKktEdgeHtt; ++k)
          kkt_block(kkt_edge_block(t, d, k, e), b, L, live, sol, T, k == kKktEdgeHtt, true);
      }
    }
  }
}

__global__ void zero_dead_lanes_kernel(double *a, int64_t rows, const int *flag, bool flag_is_ok,
                                       int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  if (b < batch && (flag_is_ok ? flag[b] != 0 : flag[b] == SIPOC_FACTOR_SUCCESS)) return;
  for (int64_t r = 0; r < rows; ++r) a[r * ld + b] = 0.0;
}

dim3 grid_for(int64_t ld, int items, int threads) {
  return dim3(static_cast<unsigned>((ld + threads - 1) / threads),
              static_cast<unsigned>(std::min(items, kMaxGridY)));
}

}  // namespace

void launch_lqr_jvp(const DevTables &t, const LqrOut &sol, const LqrTangent &tan,
                    const LqrOut &rhs, int64_t batch, int64_t ld, cudaStream_t stream) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  lqr_jvp_kernel<<<grid_for(ld, t.N, threads), threads, 0, stream>>>(t, sol, tan, rhs, batch, ld);
}

void launch_kkt_jvp(const DevTables &t, const double *sol, const KktTangent &tan, double *rhs,
                    int64_t batch, int64_t ld, cudaStream_t stream) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));
  kkt_jvp_kernel<<<grid_for(ld, t.N + 1, threads), threads, 0, stream>>>(t, sol, tan, rhs, batch,
                                                                         ld);
}

void launch_zero_dead_lanes(double *a, int64_t rows, const int *flag, bool flag_is_ok,
                            int64_t batch, int64_t ld, cudaStream_t stream) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));
  zero_dead_lanes_kernel<<<static_cast<unsigned>((ld + threads - 1) / threads), threads, 0,
                           stream>>>(a, rows, flag, flag_is_ok, batch, ld);
}

}  // namespace sipoc
