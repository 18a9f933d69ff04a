// Gradient assembly of the LQR VJP (see lqr_vjp.cuh for the formulas).
//
// Mapping: threads go across problems (engine layout X[flat * ld + b]), so every load and
// store of a warp is 32 consecutive doubles; each block row of the grid (blockIdx.y) owns
// one node (Q, q, c, delta) or one edge (M, R, r, A, B).  The entries of x, u, y and mu a
// block needs are a few percent of what it writes: they are read through L1 and the rows
// of an outer product are held in registers (vjp_common.cuh), so the kernel is bound by its
// gradient stores.
#include "lqr_vjp.cuh"

#include <algorithm>

#include "vjp_common.cuh"

namespace sipoc {

namespace {

constexpr int kThreads = 128;
constexpr int kMaxGridY = 65535;

using vjp::Lane;
using vjp::copy_vec;
using vjp::outer2;

__global__ void __launch_bounds__(kThreads)
lqr_vjp_kernel(DevTables t, LqrOut sol, LqrOut adj, const int *status, LqrGrad g,
               int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch && status[b] == SIPOC_FACTOR_SUCCESS;
  const Lane x{sol.x + b, L, live}, u{sol.u + b, L, live}, y{sol.y + b, L, live};
  const Lane mx{adj.x + b, L, live}, mu{adj.u + b, L, live}, my{adj.y + b, L, live};

  for (int item = blockIdx.y; item < t.N + t.E; item += gridDim.y) {
    if (item < t.N) {
      const int i = item, n = t.n[i], o = t.n_off[i];
      if (g.q) copy_vec(g.q + b, L, o, n, mx);
      if (g.c) copy_vec(g.c + b, L, o, n, my);
      if (g.delta)
        for (int k = 0; k < n; ++k)
          g.delta[b + static_cast<size_t>(o + k) * L] = live ? -(my(o + k) * y(o + k)) : 0.0;
      if (g.Q) outer2(g.Q + b, L, t.nn_off[i], n, n, o, mx, x, o, x, mx, 0.5);
    } else {
      const int e = item - t.N, p = t.parents[e], c = t.children[e];
      const int np = t.n[p], nc = t.n[c], m = t.m[e];
      const int op = t.n_off[p], oc = t.n_off[c], ou = t.m_off[e];
      if (g.r) copy_vec(g.r + b, L, ou, m, mu);
      if (g.R) outer2(g.R + b, L, t.mm_off[e], m, m, ou, mu, u, ou, u, mu, 0.5);
      if (g.M) outer2(g.M + b, L, t.nm_off[e], np, m, op, mx, x, ou, u, mu, 1.0);
      if (g.A) outer2(g.A + b, L, t.a_off[e], nc, np, oc, y, my, op, mx, x, 1.0);
      if (g.B) outer2(g.B + b, L, t.b_off[e], nc, m, oc, y, my, ou, mu, u, 1.0);
    }
  }
}

}  // namespace

void launch_lqr_vjp(const DevTables &t, const LqrOut &sol, const LqrOut &adjoint,
                    const int *status, const LqrGrad &grad, int64_t batch, int64_t ld,
                    cudaStream_t stream) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  const dim3 grid(static_cast<unsigned>((ld + threads - 1) / threads),
                  static_cast<unsigned>(std::min(t.N + t.E, kMaxGridY)));
  lqr_vjp_kernel<<<grid, threads, 0, stream>>>(t, sol, adjoint, status, grad, batch, ld);
}

}  // namespace sipoc
