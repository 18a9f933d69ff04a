// Gradient assembly of the Newton-KKT VJP (see kkt_vjp.cuh for the formulas).
//
// Mapping: threads go across problems (engine layout X[flat * ld + b]), so every load and
// store of a warp is 32 consecutive doubles.  Each block row of the grid (blockIdx.y) owns one
// node, one edge, or -- the last row -- the theta rows of the vectors; a grid-stride loop
// over those items keeps gridDim.y within its limit on any tree.  Every model block is an
// outer product of sol and lam on the rows / columns it occupies in K, so the blocks of an
// item are walked as a list of (array, offset, rows, cols, row start, column start, scale)
// through ONE copy of the outer-product loop (vjp_common.cuh) instead of one inlined copy per
// block: sol and lam are read through L1 and the kernel is bound by its gradient stores.
#include "kkt_vjp.cuh"

#include <algorithm>

#include "vjp_common.cuh"

namespace sipoc {

namespace {

constexpr int kThreads = 128;
constexpr int kMaxGridY = 65535;
constexpr int kNodeBlocks = 7;   // node_hxx, node_jc, node_jg, node_hxt, node_jct, node_jgt, node_htt
constexpr int kEdgeBlocks = 15;  // the nine stagewise edge blocks and the six theta ones

using vjp::Lane;
using vjp::copy_vec;
using vjp::outer2;

// G[off + i + j rows] = s (lam_{ra+i} sol_{cb+j} + sol_{ra+i} lam_{cb+j}), rows / columns
// indexed in the full [x | y | z] vector; G == nullptr: not requested.
struct Block {
  double *G;
  int off, rows, cols, ra, cb;
  double s;
};

__device__ __forceinline__ Block node_block(const DevTables &t, const KktGrad &g, int k, int i) {
  const int n = t.n[i], c = t.node_c[i], gg = t.node_g[i], p = t.theta_dim;
  const int xs = t.x_state[i], yc = t.x_dim + t.y_node_c[i], zn = t.x_dim + t.y_dim + t.z_node[i];
  const int th = t.sx_dim;
  switch (k) {
    case 0: return {g.node_hxx, t.nn_off[i], n, n, xs, xs, -0.5};
    case 1: return {g.node_jc, t.jc_node_off[i], c, n, yc, xs, -1.0};
    case 2: return {g.node_jg, t.jg_node_off[i], gg, n, zn, xs, -1.0};
    case 3: return {g.node_hxt, t.n_off[i] * p, n, p, xs, th, -1.0};
    case 4: return {g.node_jct, t.node_c_off[i] * p, c, p, yc, th, -1.0};
    case 5: return {g.node_jgt, t.node_g_off[i] * p, gg, p, zn, th, -1.0};
    default: return {g.node_htt, i * p * p, p, p, th, th, -0.5};
  }
}

__device__ __forceinline__ Block edge_block(const DevTables &t, const KktGrad &g, int k, int e) {
  const int par = t.parents[e], ch = t.children[e], p = t.theta_dim;
  const int np = t.n[par], nc = t.n[ch], m = t.m[e], c = t.edge_c[e], gg = t.edge_g[e];
  const int xp = t.x_state[par], xu = t.x_control[e], yd = t.x_dim + t.y_dyn[ch],
            yc = t.x_dim + t.y_edge_c[e], ze = t.x_dim + t.y_dim + t.z_edge[e];
  const int th = t.sx_dim;
  switch (k) {
    case 0: return {g.edge_hxx, t.hxx_edge_off[e], np, np, xp, xp, -0.5};
    case 1: return {g.edge_hxu, t.nm_off[e], np, m, xp, xu, -1.0};
    case 2: return {g.edge_huu, t.mm_off[e], m, m, xu, xu, -0.5};
    case 3: return {g.edge_A, t.a_off[e], nc, np, yd, xp, -1.0};
    case 4: return {g.edge_B, t.b_off[e], nc, m, yd, xu, -1.0};
    case 5: return {g.edge_jcx, t.jcx_off[e], c, np, yc, xp, -1.0};
    case 6: return {g.edge_jcu, t.jcu_off[e], c, m, yc, xu, -1.0};
    case 7: return {g.edge_jgx, t.jgx_off[e], gg, np, ze, xp, -1.0};
    case 8: return {g.edge_jgu, t.jgu_off[e], gg, m, ze, xu, -1.0};
    case 9: return {g.edge_hxt, t.pn_off[e] * p, np, p, xp, th, -1.0};
    case 10: return {g.edge_hut, t.m_off[e] * p, m, p, xu, th, -1.0};
    case 11: return {g.edge_dynt, t.cn_off[e] * p, nc, p, yd, th, -1.0};
    case 12: return {g.edge_jct, t.edge_c_off[e] * p, c, p, yc, th, -1.0};
    case 13: return {g.edge_jgt, t.edge_g_off[e] * p, gg, p, ze, th, -1.0};
    default: return {g.edge_htt, e * p * p, p, p, th, th, -0.5};
  }
}

// G[go + i] = s lam_{o+i} sol_{o+i}
__device__ __forceinline__ void product(double *G, size_t ld, int go, int o, int n,
                                        const Lane &lam, const Lane &sol, double s) {
  for (int i = 0; i < n; ++i) G[static_cast<size_t>(go + i) * ld] = s * (lam(o + i) * sol(o + i));
}

// The vector gradients of the rows [o, o + n) of [x | y | z]: db, and dr1 / dr2 / (dw, dr3)
// by the part the rows lie in.
__device__ __forceinline__ void vector_rows(const DevTables &t, const KktGrad &g, int64_t b,
                                            size_t ld, int o, int n, const Lane &lam,
                                            const Lane &sol) {
  if (g.b) copy_vec(g.b + b, ld, o, n, lam);
  if (o < t.x_dim) {
    if (g.r1) product(g.r1 + b, ld, o, o, n, lam, sol, -1.0);
  } else if (o < t.x_dim + t.y_dim) {
    if (g.r2) product(g.r2 + b, ld, o - t.x_dim, o, n, lam, sol, 1.0);
  } else {
    const int oz = o - t.x_dim - t.y_dim;
    if (g.w) product(g.w + b, ld, oz, o, n, lam, sol, 1.0);
    if (g.r3) product(g.r3 + b, ld, oz, o, n, lam, sol, 1.0);
  }
}

__global__ void __launch_bounds__(kThreads)
kkt_vjp_kernel(DevTables t, const double *sol_p, const double *lam_p, const int *ok, KktGrad g,
               int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch && ok[b] != 0;
  const Lane sol{sol_p + b, L, live}, lam{lam_p + b, L, live};
  const int xd = t.x_dim, zd = t.x_dim + t.y_dim;

  for (int item = blockIdx.y; item <= t.N + t.E; item += gridDim.y) {
    int nblocks;
    if (item < t.N) {
      const int i = item;
      vector_rows(t, g, b, L, t.x_state[i], t.n[i], lam, sol);
      vector_rows(t, g, b, L, xd + t.y_dyn[i], t.n[i], lam, sol);
      vector_rows(t, g, b, L, xd + t.y_node_c[i], t.node_c[i], lam, sol);
      vector_rows(t, g, b, L, zd + t.z_node[i], t.node_g[i], lam, sol);
      nblocks = kNodeBlocks;
    } else if (item < t.N + t.E) {
      const int e = item - t.N;
      vector_rows(t, g, b, L, t.x_control[e], t.m[e], lam, sol);
      vector_rows(t, g, b, L, xd + t.y_edge_c[e], t.edge_c[e], lam, sol);
      vector_rows(t, g, b, L, zd + t.z_edge[e], t.edge_g[e], lam, sol);
      nblocks = kEdgeBlocks;
    } else {
      vector_rows(t, g, b, L, t.sx_dim, t.theta_dim, lam, sol);  // the theta rows
      nblocks = 0;
    }
#pragma unroll 1
    for (int k = 0; k < nblocks; ++k) {
      const Block d = item < t.N ? node_block(t, g, k, item) : edge_block(t, g, k, item - t.N);
      if (d.G != nullptr && d.rows > 0 && d.cols > 0)
        outer2(d.G + b, L, d.off, d.rows, d.cols, d.ra, lam, sol, d.cb, sol, lam, d.s);
    }
  }
}

}  // namespace

void launch_kkt_vjp(const DevTables &t, const double *sol, const double *lam, const int *ok,
                    const KktGrad &grad, int64_t batch, int64_t ld, cudaStream_t stream) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  const dim3 grid(static_cast<unsigned>((ld + threads - 1) / threads),
                  static_cast<unsigned>(std::min(t.N + t.E + 1, kMaxGridY)));
  kkt_vjp_kernel<<<grid, threads, 0, stream>>>(t, sol, lam, ok, grad, batch, ld);
}

}  // namespace sipoc
