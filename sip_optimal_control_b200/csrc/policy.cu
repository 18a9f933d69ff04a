// Policy export kernels (see policy.cuh): a masked block gather out of a plan's kept store
// and spill, and the per-edge rebuild of V for the plans that keep P = F^-1 instead of V.
#include "policy.cuh"

#include <algorithm>

namespace sipoc {

namespace {

constexpr int kThreads = 128;
constexpr int kMaxGridY = 65535;

__host__ __device__ constexpr int tri(int n) { return n * (n + 1) / 2; }
// Column-major packed lower index, i >= j (the kept P of riccati_fast.cu / riccati_cta.cu).
__host__ __device__ constexpr int pk(int i, int j, int n) { return j * n - j * (j - 1) / 2 + (i - j); }

__device__ __forceinline__ double src_at(const PolicySrc &s, int64_t flat, int64_t b, size_t L) {
  return s.pm_stride != 0 ? s.p[b * s.pm_stride + flat] : s.p[static_cast<size_t>(flat) * L + b];
}

__global__ void __launch_bounds__(kThreads)
policy_gather_kernel(DevTables t, PolicyArray which, PolicySrc src, double *dst,
                     const int *status, int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch && status[b] == SIPOC_FACTOR_SUCCESS;
  const bool per_edge = which == PolicyArray::K || which == PolicyArray::k;
  const int count = per_edge ? t.E : t.N;
  for (int j = blockIdx.y; j < count; j += gridDim.y) {
    int rows, cols, o;
    switch (which) {
      case PolicyArray::K: rows = t.m[j]; cols = t.n[t.parents[j]]; o = t.nm_off[j]; break;
      case PolicyArray::k: rows = t.m[j]; cols = 1; o = t.m_off[j]; break;
      case PolicyArray::V: rows = t.n[j]; cols = rows; o = t.nn_off[j]; break;
      default: rows = t.n[j]; cols = 1; o = t.n_off[j]; break;
    }
    int64_t base = o;
    int lead = rows;
    if (!src.same_as_out) {
      int s = 0, local = j;
      if (src.seg_len > 0) {
        s = min(j / src.seg_len, src.segs - 1);
        local = j - s * src.seg_len;
      }
      base = s * src.seg_stride + src.off + local * src.block;
      lead = src.rows;
    }
    for (int c = 0; c < cols; ++c)
      for (int r = 0; r < rows; ++r)
        dst[static_cast<size_t>(o + r + c * rows) * L + b] =
            live ? src_at(src, base + r + c * lead, b, L) : 0.0;
  }
}

template <int N, int M>
__global__ void __launch_bounds__(kThreads)
policy_rebuild_v_kernel(LqrIn in, PolicySrc P, PolicySrc K, double *V, const int *status, int E,
                        int64_t batch, int64_t ld) {
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  const size_t L = static_cast<size_t>(ld);
  const bool live = b < batch && status[b] == SIPOC_FACTOR_SUCCESS;
  for (int p = blockIdx.y; p <= E; p += gridDim.y) {  // node p, and edge p (child p + 1)
    double *Vo = V + static_cast<size_t>(p) * N * N * L + b;
    const double *Q = in.Q + static_cast<size_t>(p) * N * N * L + b;
    if (!live) {
      for (int t = 0; t < N * N; ++t) Vo[static_cast<size_t>(t) * L] = 0.0;
      continue;
    }
    if (p == E) {  // terminal node: V = Q (lqr.cpp:658)
      for (int j = 0; j < N; ++j)
        for (int i = j; i < N; ++i) {
          const double q = Q[static_cast<size_t>(i + j * N) * L];
          Vo[static_cast<size_t>(i + j * N) * L] = q;
          Vo[static_cast<size_t>(j + i * N) * L] = q;
        }
      continue;
    }
    int64_t seg = 0;
    int le = p;
    if (P.seg_len > 0) {
      const int s = p / P.seg_len;
      le = p - s * P.seg_len;
      seg = s;
    }
    const int64_t pbase = seg * P.seg_stride + P.off + static_cast<int64_t>(le + 1) * P.block;
    const int64_t kbase = seg * K.seg_stride + K.off + static_cast<int64_t>(le) * K.block;
    const double *A = in.A + static_cast<size_t>(p) * N * N * L + b;
    const double *B = in.B + static_cast<size_t>(p) * N * M * L + b;
    const double *Mm = in.M + static_cast<size_t>(p) * N * M * L + b;
    const double *dl = in.delta + static_cast<size_t>(p + 1) * N * L + b;
    double sdi[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sdi[i] = rsqrt(dl[static_cast<size_t>(i) * L]);
#pragma unroll 1
    for (int j = 0; j < N; ++j) {
      // w = W_c a_j = D^-1/2 (s - P s), s = D^-1/2 a_j  (apply_node of riccati_fast.cu)
      double w[N], f[N];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        w[i] = sdi[i] * A[static_cast<size_t>(i + j * N) * L];
        f[i] = 0.0;
      }
#pragma unroll
      for (int jj = 0; jj < N; ++jj)
#pragma unroll
        for (int i = jj; i < N; ++i) {
          const double pv = src_at(P, pbase + pk(i, jj, N), b, L);
          f[i] += pv * w[jj];
          if (i != jj) f[jj] += pv * w[i];
        }
#pragma unroll
      for (int i = 0; i < N; ++i) w[i] = sdi[i] * (w[i] - f[i]);
      // h = H(:, j) = M(j, :)' + B' w  (lqr.cpp:704-705)
      double h[M];
#pragma unroll
      for (int a = 0; a < M; ++a) {
        double s = Mm[static_cast<size_t>(j + a * N) * L];
#pragma unroll
        for (int i = 0; i < N; ++i) s += B[static_cast<size_t>(i + a * N) * L] * w[i];
        h[a] = s;
      }
      // V(i, j), i >= j: Q(i, j) + a_i' w + K(:, i)' h  (lqr.cpp:715-719)
#pragma unroll 1
      for (int i = j; i < N; ++i) {
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < N; ++r) s += A[static_cast<size_t>(r + i * N) * L] * w[r];
        double kh = 0.0;
#pragma unroll
        for (int a = 0; a < M; ++a) kh += src_at(K, kbase + a + i * M, b, L) * h[a];
        const double v = Q[static_cast<size_t>(i + j * N) * L] + s + kh;
        Vo[static_cast<size_t>(i + j * N) * L] = v;
        Vo[static_cast<size_t>(j + i * N) * L] = v;
      }
    }
  }
}

dim3 grid_for(int64_t ld, int items, int threads) {
  return dim3(static_cast<unsigned>((ld + threads - 1) / threads),
              static_cast<unsigned>(std::max(1, std::min(items, kMaxGridY))));
}

template <int N, int M>
void rebuild(const LqrIn &in, const PolicySrc &P, const PolicySrc &K, double *V,
             const int *status, int E, int64_t batch, int64_t ld, cudaStream_t s) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));  // ld: multiple of 32
  policy_rebuild_v_kernel<N, M><<<grid_for(ld, E + 1, threads), threads, 0, s>>>(
      in, P, K, V, status, E, batch, ld);
}

}  // namespace

void launch_policy_gather(const DevTables &t, PolicyArray which, const PolicySrc &src,
                          double *dst, const int *status, int64_t batch, int64_t ld,
                          cudaStream_t s) {
  const int threads = static_cast<int>(std::min<int64_t>(kThreads, ld));
  const int items = (which == PolicyArray::K || which == PolicyArray::k) ? t.E : t.N;
  policy_gather_kernel<<<grid_for(ld, items, threads), threads, 0, s>>>(t, which, src, dst,
                                                                        status, batch, ld);
}

// The shapes of the plans that keep P instead of V: riccati_fast.cu (n in {4, 6, 8} x
// m in {1..4}, (12, 4)) and riccati_cta.cu ((16, 4), (32, 8), (64, 24)).
bool launch_policy_rebuild_v(int n, int m, const LqrIn &in, const PolicySrc &P,
                             const PolicySrc &K, double *V, const int *status, int E,
                             int64_t batch, int64_t ld, cudaStream_t s) {
#define SIPOC_REBUILD(NN, MM)                                    \
  if (n == NN && m == MM) {                                      \
    rebuild<NN, MM>(in, P, K, V, status, E, batch, ld, s);       \
    return true;                                                 \
  }
  SIPOC_REBUILD(4, 1) SIPOC_REBUILD(4, 2) SIPOC_REBUILD(4, 3) SIPOC_REBUILD(4, 4)
  SIPOC_REBUILD(6, 1) SIPOC_REBUILD(6, 2) SIPOC_REBUILD(6, 3) SIPOC_REBUILD(6, 4)
  SIPOC_REBUILD(8, 1) SIPOC_REBUILD(8, 2) SIPOC_REBUILD(8, 3) SIPOC_REBUILD(8, 4)
  SIPOC_REBUILD(12, 4) SIPOC_REBUILD(16, 4) SIPOC_REBUILD(32, 8) SIPOC_REBUILD(64, 24)
#undef SIPOC_REBUILD
  return false;
}

PolicySources policy_sources(PolicyStore kind, int n, int m, int T, const double *store,
                             const double *scratch) {
  PolicySources o;
  const int64_t T1 = T + 1;
  o.K.p = o.V_or_P.p = store;
  o.k.p = o.v.p = scratch;
  o.K.rows = m;
  o.K.block = int64_t(n) * m;
  o.k.rows = m;
  o.k.block = m;
  o.k.off = T1 * n;  // FastSizes / CtaSizes / StrictSizes::ok
  o.v.rows = n;
  o.v.block = n;
  if (kind == PolicyStore::STRICT) {  // StrictSizes: V, F, sqrt(delta), 1/sqrt(delta), W, K, G
    o.V_or_P.rows = n;
    o.V_or_P.block = int64_t(n) * n;
    o.K.off = T1 * (2 * n * n + 2 * n) + int64_t(T) * n * n;
  } else {  // FastSizes / CtaSizes: P packed, K, G
    o.V_or_P.block = tri(n);
    o.K.off = T1 * tri(n);
    if (kind == PolicyStore::CTA) {  // problem-major, CtaSizes::store / scratch per problem
      const int64_t st = o.K.off + int64_t(T) * n * m + int64_t(T) * tri(m);
      const int64_t sc = o.k.off + int64_t(T) * m;
      o.K.pm_stride = o.V_or_P.pm_stride = st;
      o.k.pm_stride = o.v.pm_stride = sc;
    }
  }
  return o;
}

}  // namespace sipoc
