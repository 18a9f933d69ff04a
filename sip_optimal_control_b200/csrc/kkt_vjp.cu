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

#include "kkt_blocks.cuh"
#include "vjp_common.cuh"

namespace sipoc {

namespace {

constexpr int kThreads = 128;
constexpr int kMaxGridY = 65535;

using vjp::Lane;
using vjp::copy_vec;
using vjp::outer2;

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
      nblocks = kKktNodeBlocks;
    } else if (item < t.N + t.E) {
      const int e = item - t.N;
      vector_rows(t, g, b, L, t.x_control[e], t.m[e], lam, sol);
      vector_rows(t, g, b, L, xd + t.y_edge_c[e], t.edge_c[e], lam, sol);
      vector_rows(t, g, b, L, zd + t.z_edge[e], t.edge_g[e], lam, sol);
      nblocks = kKktEdgeBlocks;
    } else {
      vector_rows(t, g, b, L, t.sx_dim, t.theta_dim, lam, sol);  // the theta rows
      nblocks = 0;
    }
#pragma unroll 1
    for (int k = 0; k < nblocks; ++k) {
      const KktBlock<double *> d =
          item < t.N ? kkt_node_block(t, g, k, item) : kkt_edge_block(t, g, k, item - t.N);
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
