// Device helpers shared by the gradient-assembly kernels of the VJPs (lqr_vjp.cu, kkt_vjp.cu).
//
// Both kernels run one thread per problem on the engine layout X[flat * ld + b] and write
// gradient blocks that are outer products of a solution and its adjoint; the entries of
// those vectors are a few percent of what a kernel writes, so they are read through L1 and
// the rows of an outer product are held in registers, kVjpRows at a time.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>

namespace sipoc {
namespace vjp {

constexpr int kVjpRows = 8;  // rows of an outer-product block held in registers

// One problem's lane of an engine-layout vector; reads 0 where the problem is not live
// (padding lane or failed factorization), so every gradient there comes out as zero.
struct Lane {
  const double *p;
  size_t ld;
  bool live;
  __device__ __forceinline__ double operator()(int off) const {
    return live ? __ldg(p + static_cast<size_t>(off) * ld) : 0.0;
  }
};

__device__ __forceinline__ void copy_vec(double *G, size_t ld, int off, int n, const Lane &v) {
  for (int i = 0; i < n; ++i) G[static_cast<size_t>(off + i) * ld] = v(off + i);
}

// G[off + i + j rows] = s (a_i b_j + c_i d_j): a rows x cols column-major block; a, c are
// read at ra + i, b, d at cb + j.
__device__ __forceinline__ void outer2(double *G, size_t ld, int off, int rows, int cols,
                                       int ra, const Lane &a, const Lane &c, int cb,
                                       const Lane &b, const Lane &d, double s) {
  for (int i0 = 0; i0 < rows; i0 += kVjpRows) {
    double av[kVjpRows], cv[kVjpRows];
#pragma unroll
    for (int k = 0; k < kVjpRows; ++k) {
      const bool in = i0 + k < rows;
      av[k] = in ? a(ra + i0 + k) : 0.0;
      cv[k] = in ? c(ra + i0 + k) : 0.0;
    }
    for (int j = 0; j < cols; ++j) {
      const double bj = b(cb + j), dj = d(cb + j);
      double *col = G + static_cast<size_t>(off + i0 + j * rows) * ld;
#pragma unroll
      for (int k = 0; k < kVjpRows; ++k)
        if (i0 + k < rows) col[k * ld] = s * (av[k] * bj + cv[k] * dj);
    }
  }
}

}  // namespace vjp
}  // namespace sipoc
