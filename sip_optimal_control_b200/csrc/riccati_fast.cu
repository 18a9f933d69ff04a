// Shape-specialised Riccati kernels for uniform chains (n, m compile-time).
//
// Three kernels per shape, all sm_100a, FP64:
//
//   riccati_backward_subwarp<N, M>   backward Riccati sweep (reference
//       lqr.cpp:645-731) fused with the backward affine sweep of the solve
//       (lqr.cpp:738-796).  FOUR LANES PER PROBLEM, eight problems per warp.
//       Each stage's A, B, Q, M, R, q, r, c, delta are staged into shared
//       memory with cp.async (16 B per lane, 64 B contiguous per matrix element
//       = the 8 problems of the warp in the batch-interleaved HBM layout);
//       the next stage's copy is issued as soon as the current stage has
//       consumed its operands and lands while the factorizations run.
//   riccati_backward_thread<N, M>    the same mathematics, one thread per
//       problem with every matrix in registers, for tiny n (cartpole).
//   affine_backward<N, M>            backward affine sweep alone (solve after
//       a kept factorization), one thread per problem, streaming.
//   rollout_forward<N, M>            root solve + forward rollout + costates
//       (lqr.cpp:798-870), one thread per problem, streaming: every operand is
//       read exactly once with fully coalesced 256 B warp requests.
//
// Per stage (edge k, parent node k, child node k+1) the backward kernels use
// the "augmented Hessian" form of the recursion, algebraically identical to
// the reference's statements but with ~35 % fewer flops:
//     Z   = [B_k | A_k]                         (n x (m+n))
//     S   = W_{k+1} Z                           W = V (I + D V)^-1, symmetric
//     Psi = [R M'; M Q] + Z' S                  ((m+n) x (m+n), lower)
//     G   = Psi_uu = L_G L_G'                   fail -> G_FACTORIZATION_FAILURE
//     Lam = Psi_xu L_G^-T ;  K_k = -L_G^-T Lam'
//     V_k = Psi_xx - Lam Lam'
//     F   = I + D^1/2 V_k D^1/2 = L L'          fail -> F_FACTORIZATION_FAILURE
//     W_k = D^-1/2 (I - L^-T L^-1) D^-1/2       (lqr.cpp:511-529)
// and, for the affine part,
//     g = v' - W'(delta' o v' - c') ;  [h; w] = [r; q] + Z' g
//     t = L_G^-1 h ;  k_k = -L_G^-T t ;  v_k = w - Lam t.
// The forward pass needs only (W, v) per node and (K, k) per edge:
//     y' = v' + W' f ,  x' = f - delta' o (W' f) ,  f = c' - delta' o v' + A x + B u
// because (I + D V)^-1 = I - D W.
#include "riccati_fast.cuh"

#include <cstdio>
#include <cstdlib>
#include <type_traits>

namespace sipoc {
namespace {

#ifndef SIPOC_FUSED_PF
#define SIPOC_FUSED_PF 0
#endif
constexpr int kGroup = 4;  // lanes per problem
constexpr int kTile = 8;   // problems per warp

__host__ __device__ constexpr int tri(int n) { return n * (n + 1) / 2; }
// Column-major packed lower index, i >= j.
__host__ __device__ constexpr int pk(int i, int j, int n) {
  return j * n - j * (j - 1) / 2 + (i - j);
}
__host__ __device__ constexpr int cdiv(int a, int b) { return (a + b - 1) / b; }
// Packed lower, column-major: first row of column j minus j, so that (i, j) is colbase(j) + i.
__host__ __device__ constexpr int colbase(int j, int n) { return j * n - j * (j - 1) / 2 - j; }

// Per-problem element counts of the kept factorization and the rollout spill.
template <int N, int M>
struct FastSizes {
  static __host__ __device__ constexpr int64_t oW(int) { return 0; }
  static __host__ __device__ constexpr int64_t oK(int T) { return int64_t(T + 1) * tri(N); }
  static __host__ __device__ constexpr int64_t oG(int T) { return oK(T) + int64_t(T) * N * M; }
  static __host__ __device__ constexpr int64_t store(int T) { return oG(T) + int64_t(T) * tri(M); }
  static __host__ __device__ constexpr int64_t ov(int) { return 0; }
  static __host__ __device__ constexpr int64_t ok(int T) { return int64_t(T + 1) * N; }
  static __host__ __device__ constexpr int64_t scratch(int T) { return ok(T) + int64_t(T) * M; }
};

__device__ __forceinline__ void cp_async16(double *smem, const double *gmem) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(double *smem, const double *gmem) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const double *gmem) {
  asm volatile("prefetch.global.L2 [%0];\n" ::"l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() {
  asm volatile("cp.async.commit_group;\n" ::: "memory");
}
template <int PENDING>
__device__ __forceinline__ void cp_async_wait_group() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(PENDING) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

// Streaming loads / stores: every operand is touched once per pass.
__device__ __forceinline__ double ldcs(const double *p) { return __ldcs(p); }
__device__ __forceinline__ void stcs(double *p, double v) { __stcs(p, v); }

// What the kept factorization holds per node is P = F^-1 = (I + D^1/2 V D^1/2)^-1 (packed
// lower), not W: with s = D^-1/2 z and t = P s,
//     (I + D V)^-1 z = D^1/2 t             the reference's F-solve form, lqr.cpp:531-549
//     W z            = D^-1/2 (s - t)      W = D^-1/2 (I - P) D^-1/2, lqr.cpp:511-529
// The rollout's x' = (I + D V)^-1 f formed as f - delta o (W f) cancels at large delta
// (Newton-KKT: r2 up to 1e9 -> 1e-7 relative); D^1/2 P D^-1/2 f does not.
// On return z holds W z and fz holds (I + D V)^-1 z.
template <int N, class LoadP>
__device__ __forceinline__ void apply_node(double (&z)[N], const double (&dd)[N], LoadP loadP,
                                           double (&fz)[N]) {
  double sdi[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    sdi[i] = rsqrt(dd[i]);
    z[i] *= sdi[i];
    fz[i] = 0.0;
  }
#pragma unroll
  for (int j = 0; j < N; ++j)
#pragma unroll
    for (int i = j; i < N; ++i) {
      const double p = loadP(pk(i, j, N));
      fz[i] += p * z[j];
      if (i != j) fz[j] += p * z[i];
    }
#pragma unroll
  for (int i = 0; i < N; ++i) {
    z[i] = sdi[i] * (z[i] - fz[i]);
    fz[i] *= dd[i] * sdi[i];
  }
}

// ===========================================================================
// Shared-memory map of one warp (rows of kTile doubles = 64 B).
// ===========================================================================
// PACKW: W packed and no pitch padding -- 494 rows at (12, 4), seven warps per SM -- for
// grids of a few waves (and the fused rollout); otherwise W full with an odd column pitch,
// 592 rows, six warps per SM, the faster map when the grid is many waves deep.
template <int N, int M, bool PACKW>
struct Smem {
  static constexpr int NZ = N + M;
  // Column pitch of every array whose columns are read by different lanes of a problem
  // at the same time (Z, M, W, Psi_xu): an ODD number of 64-byte rows, so the four
  // lanes' rows alternate between the two halves of the 32 banks (pitch N = 12 puts them
  // all in one half: 4 wavefronts per load instead of 2).  No padding in the packed map.
  static constexpr int P = (N % 2 == 0 && !PACKW) ? N + 1 : N;
  static constexpr int rZ = 0;                // [B | A], column-major, pitch P
  static constexpr int rQ = rZ + NZ * P;      // Q_k, packed lower
  static constexpr int rM = rQ + tri(N);      // M_k, N x M column-major, pitch P
  static constexpr int rR = rM + M * P;       // R_k, packed lower
  static constexpr int rq = rR + tri(M);      // q_k
  static constexpr int rr = rq + N;           // r_k
  static constexpr int rc = rr + M;           // c_{k+1}
  static constexpr int rd = rc + N;           // delta_k (as staged)
  static constexpr int kStaged = rd + N;
  // W of the last processed node: full (pitch P), or PACKED lower (column-major): entry
  // (i, j), i >= j, at row colbase(j) + i, colbase(j) = pk(j, j) - j.
  static constexpr int rW = kStaged;
  static constexpr int rG = rc;               // g overwrites c (dead once f is formed)
  static constexpr int rV = rW + (PACKW ? tri(N) : N * P);  // v of the last processed node
  static constexpr int rDl = rV + N;          // delta of the last processed node
  static constexpr int rSd = rDl + N;         // sqrt(delta), 1/sqrt(delta) of the node in flight
  static constexpr int rSdi = rSd + N;
  // Exchange region, ALIASED onto the Q | M | R staging rows (their contents are
  // consumed before the first exchange of a stage and re-fetched after the last):
  // first [Psi_uu packed | Psi_xu (overwritten in place by Lambda) | h], later F packed.
  static constexpr int rX = rQ;
  static constexpr int xGuu = rX;
  static constexpr int xPxu = xGuu + tri(M);
  static constexpr int xH = xPxu + M * P;
  static constexpr int xLam = xPxu;
  static_assert(tri(M) + M * P + M <= tri(N) + M * P + tri(M), "exchange region fits");
  static constexpr int kRows = rSdi + N;
  static constexpr int kBytes = kRows * kTile * int(sizeof(double));
};

// Copies `count` consecutive flat elements (rows of 8 problems) into shared
// memory: lane l moves 16 B (problems 2(l&3), 2(l&3)+1) of row (l>>2) + 8 i.
// `dst` and `src` already include the lane's own row / chunk offset; ld8 = 8 ld.
__device__ __forceinline__ void stage_run(double *dst, const double *src, int64_t ld8,
                                          int count, int rr) {
#pragma unroll
  for (int i0 = 0; i0 < count; i0 += 8) {
    if (i0 + 8 <= count || i0 + rr < count) cp_async16(dst + i0 * kTile, src);
    src += ld8;
  }
}

// `count` consecutive flat elements of a column-major block with N rows per column
// -> shared-memory columns of pitch P rows.
template <int N, int P>
__device__ __forceinline__ void stage_cols(double *dst0, const double *src, int64_t ld8,
                                           int count, int lane) {
  const int sub = lane & 3, rr = lane >> 2;
#pragma unroll
  for (int i0 = 0; i0 < count; i0 += 8) {
    const int e = i0 + rr;
    const int row = e + (P - N) * (e / N);
    if (i0 + 8 <= count || e < count) cp_async16(dst0 + row * kTile + sub * 2, src);
    src += ld8;
  }
}

// Lower triangle of a column-major N x N block -> packed lower rows.
template <int N>
__device__ __forceinline__ void stage_lower(double *dst, const double *src, int64_t ld,
                                            int64_t ld8, int rr) {
#pragma unroll
  for (int j = 0; j < N; ++j) {
    stage_run(dst + pk(j, j, N) * kTile, src, ld8, N - j, rr);
    src += (N + 1) * ld;
  }
}

// ===========================================================================
// Backward sweep, four lanes per problem, WARPS warps (8 problems each) per CTA.
// ===========================================================================
//
// FUSED (factor + solve in one call): the warp rolls its own eight problems forward
// right after their backward sweep -- root solve, rollout, costates (lqr.cpp:798-870) --
// with the four lanes of a problem sharing the matrix-vector products and the operands
// of every stage (A, B from the inputs; K, k, P, v from the spill the sweep has just
// written; c, delta) brought in by cp.async one half-stage ahead of their use.  The
// rollout of one tile hides under the DFMA-bound sweeps of the other tiles of the SM:
// the step costs the backward sweep plus a few per cent instead of sweep + rollout, and
// a shard of a few thousand problems no longer pays a latency-bound rollout kernel.
//
// SEGMENTED (parallel in time, scan.cu): blockIdx.y is a segment of T edges of a longer
// horizon.  The tile sweeps its segment from the boundary value function (V, v at the
// segment's last node, from the scan) instead of (Q, q) of that node, and rolls forward from
// the boundary state instead of the root solve; every array is addressed at the segment's
// offset, the kept factorization and the status are per (segment, problem).
struct SegmentArgs {
  const double *Vb, *vb, *xb;  // [S + 1][N N | N | N][ld], engine layout
};

template <int N, int M, bool SOLVE, int WARPS, bool FUSED = false, bool PACKW = FUSED,
          bool SEGMENTED = false>
__global__ void __launch_bounds__(32 * WARPS)
riccati_backward_subwarp(LqrIn in, LqrOut out, int *status_out, double *store, double *scratch,
                         int64_t batch, int64_t ld, int T, SegmentArgs sg) {
  static_assert(SOLVE || !FUSED, "the fused rollout needs the affine sweep");
  static_assert(FUSED || !SEGMENTED, "segments run the fused sweep + rollout");
  using S = Smem<N, M, PACKW>;
  using Z = FastSizes<N, M>;
  const int seg = SEGMENTED ? blockIdx.y : 0;
  if constexpr (SEGMENTED) {
    const int64_t node0 = static_cast<int64_t>(seg) * T;  // first node / edge of the segment
    in.Q += node0 * N * N * ld;
    in.q += node0 * N * ld;
    in.c += node0 * N * ld;
    in.delta += node0 * N * ld;
    in.A += node0 * N * N * ld;
    in.B += node0 * N * M * ld;
    in.M += node0 * N * M * ld;
    in.R += node0 * M * M * ld;
    in.r += node0 * M * ld;
    out.x += node0 * N * ld;
    out.y += node0 * N * ld;
    out.u += node0 * M * ld;
    store += static_cast<int64_t>(seg) * Z::store(T) * ld;
    scratch += static_cast<int64_t>(seg) * Z::scratch(T) * ld;
    status_out += static_cast<int64_t>(seg) * ld;
  }
  constexpr int SX = cdiv(N, kGroup);  // own state columns per lane
  constexpr int SU = cdiv(M, kGroup);  // own control columns per lane
  extern __shared__ __align__(16) double sm_all[];

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  double *sm = sm_all + warp * (S::kRows * kTile);
  const int prob = lane & (kTile - 1);
  const int r = lane >> 3;
  int64_t b0 = (static_cast<int64_t>(blockIdx.x) * WARPS + warp) * kTile;
  const bool tile_ok = b0 < batch;
  if (b0 + kTile > ld) b0 = ld - kTile;  // spare warp of the last CTA: stay in bounds
  const int64_t b = b0 + prob;
  const bool valid = tile_ok && b < batch;
  const unsigned group_mask = 0x01010101u << prob;

  // Own columns (cyclic): state column xj[s] = r + 4 s, control column uj[s].
  int xj[SX], uj[SU], qcol[SX], rcol[SU];
  bool xok[SX], uok[SU];
#pragma unroll
  for (int s = 0; s < SX; ++s) {
    const int j = r + kGroup * s;
    xok[s] = j < N;
    xj[s] = xok[s] ? j : N - 1;
    qcol[s] = xj[s] * N - xj[s] * (xj[s] - 1) / 2 - xj[s];  // packed row of (i, xj) = qcol + i
  }
#pragma unroll
  for (int s = 0; s < SU; ++s) {
    const int j = r + kGroup * s;
    uok[s] = j < M;
    uj[s] = uok[s] ? j : M - 1;
    rcol[s] = uj[s] * M - uj[s] * (uj[s] - 1) / 2 - uj[s];
  }

#define SM(row) sm[(row) * kTile + prob]

  // Staging: per-array running pointers to the block of the stage to fetch next
  // (already offset by this lane's row / 16-byte chunk); they walk backward.
  const int rr = lane >> 2;
  const int64_t ld8 = ld * 8;
  const int64_t lane_goff = rr * ld + (lane & 3) * 2 + b0;
  double *sdst = sm + rr * kTile + (lane & 3) * 2;
  const double *pQ = in.Q + static_cast<int64_t>(T) * N * N * ld + lane_goff;
  const double *pd = in.delta + static_cast<int64_t>(T) * N * ld + lane_goff;
  const double *pq = SOLVE ? in.q + static_cast<int64_t>(T) * N * ld + lane_goff : nullptr;
  const double *pc = SOLVE ? in.c + static_cast<int64_t>(T) * N * ld + lane_goff : nullptr;
  const double *pA = in.A + static_cast<int64_t>(T - 1) * N * N * ld + lane_goff;
  const double *pB = in.B + static_cast<int64_t>(T - 1) * N * M * ld + lane_goff;
  const double *pM = in.M + static_cast<int64_t>(T - 1) * N * M * ld + lane_goff;
  const double *pR = in.R + static_cast<int64_t>(T - 1) * M * M * ld + lane_goff;
  const double *pr = SOLVE ? in.r + static_cast<int64_t>(T - 1) * M * ld + lane_goff : nullptr;

  // Z = [B | A] and the vectors of the stage the pointers stand on (q, delta of its
  // node, r of its edge, c of the edge's child), then step back.  Issued as soon as
  // the current stage has consumed its own copies.
  auto issue_z_vec = [&](bool with_edge) {
    stage_run(sdst + S::rd * kTile, pd, ld8, N, rr);
    pd -= static_cast<int64_t>(N) * ld;
    if (SOLVE) {
      stage_run(sdst + S::rq * kTile, pq, ld8, N, rr);
      pq -= static_cast<int64_t>(N) * ld;
    }
    if (with_edge) {
      stage_cols<N, S::P>(sm + S::rZ * kTile, pB, ld8, N * M, lane);
      stage_cols<N, S::P>(sm + (S::rZ + M * S::P) * kTile, pA, ld8, N * N, lane);
      pB -= static_cast<int64_t>(N) * M * ld;
      pA -= static_cast<int64_t>(N) * N * ld;
      if (SOLVE) {
        stage_run(sdst + S::rr * kTile, pr, ld8, M, rr);
        stage_run(sdst + S::rc * kTile, pc, ld8, N, rr);
        pr -= static_cast<int64_t>(M) * ld;
        pc -= static_cast<int64_t>(N) * ld;
      }
    }
  };
  // Q (lower), M, R (lower) of the stage the pointers stand on, then step back.  Their
  // rows double as the exchange region, so they are fetched only after the last
  // exchange of the current stage (the read of F).
  auto issue_qmr = [&](bool with_edge) {
    stage_lower<N>(sdst + S::rQ * kTile, pQ, ld, ld8, rr);
    pQ -= static_cast<int64_t>(N) * N * ld;
    if (with_edge) {
      stage_cols<N, S::P>(sm + S::rM * kTile, pM, ld8, N * M, lane);
      stage_lower<M>(sdst + S::rR * kTile, pR, ld, ld8, rr);
      pM -= static_cast<int64_t>(N) * M * ld;
      pR -= static_cast<int64_t>(M) * M * ld;
    }
  };

  // Output pointers of the stage in flight (problem b), walking backward too.
  double *Wst = store + (Z::oW(T) + static_cast<int64_t>(T) * tri(N)) * ld + b;
  double *Kst = store + (Z::oK(T) + static_cast<int64_t>(T - 1) * N * M) * ld + b;
  double *Gst = store + (Z::oG(T) + static_cast<int64_t>(T - 1) * tri(M)) * ld + b;
  double *vst = SOLVE ? scratch + (Z::ov(T) + static_cast<int64_t>(T) * N) * ld + b : nullptr;
  double *kst = SOLVE ? scratch + (Z::ok(T) + static_cast<int64_t>(T - 1) * M) * ld + b : nullptr;

  int status = SIPOC_FACTOR_SUCCESS;
  bool bad_delta = false;

  // delta_k -> rDl, sqrt -> rSd, 1/sqrt -> rSdi, own rows  (lqr.cpp:475-485)
  auto update_delta = [&]() {
    bad_delta = false;
#pragma unroll
    for (int s = 0; s < SX; ++s) {
      const double d = SM(S::rd + xj[s]);
      if (xok[s]) {
        bad_delta = bad_delta || !(d > 0.0);
        // 1 / sqrt(d) by rsqrt, sqrt(d) = d * that: the FP64 sqrt + division chain it replaces
        // was 4.6 % of the sweep's stall samples (ncu); a couple of ulps, far inside 1e-9
        const double sdi = rsqrt(d);
        SM(S::rDl + xj[s]) = d;
        SM(S::rSd + xj[s]) = d * sdi;
        SM(S::rSdi + xj[s]) = sdi;
      }
    }
  };

  if constexpr (SEGMENTED) {
    // terminal node of the segment: the boundary value function stands in for (Q, q)
    pQ = sg.Vb + static_cast<int64_t>(seg + 1) * N * N * ld + lane_goff;
    pq = sg.vb + static_cast<int64_t>(seg + 1) * N * ld + lane_goff;
  }
  issue_z_vec(false);
  issue_qmr(false);
  cp_async_commit();
  if constexpr (SEGMENTED) {
    pQ = in.Q + static_cast<int64_t>(T - 1) * N * N * ld + lane_goff;
    pq = in.q + static_cast<int64_t>(T - 1) * N * ld + lane_goff;
  }

  for (int k = T; k >= 0; --k) {
    cp_async_wait_all();
    // One CTA-wide barrier per stage keeps the warps of the CTA inside the same
    // stretch of code, so they share instruction-cache lines.
    if (WARPS > 1) __syncthreads(); else __syncwarp();

    // V_k (own columns, rows >= 4 s) and v_k (own entries).
    double V[SX][N], vv[SX];
    if (k == T) {
      // ---- terminal node: V = Q_T, v = q_T ----------------------------------
#pragma unroll
      for (int s = 0; s < SX; ++s) {
#pragma unroll
        for (int i = kGroup * s; i < N; ++i) V[s][i] = SM(S::rQ + qcol[s] + i);
        vv[s] = SOLVE ? SM(S::rq + xj[s]) : 0.0;
      }
      update_delta();
      __syncwarp();
      if (T > 0) {
        issue_z_vec(true);
        cp_async_commit();
      }
    } else {
      // ---- edge k: parent node k, child node k + 1 ---------------------------
      // g = v' - W'(delta' o v' - c'), own rows  (lqr.cpp:778-782)
      if (SOLVE) {
        double f[N];
#pragma unroll
        for (int i = 0; i < N; ++i) f[i] = SM(S::rDl + i) * SM(S::rV + i) - SM(S::rc + i);
        __syncwarp();  // g is written over c
#pragma unroll
        for (int s = 0; s < SX; ++s) {
          double acc = 0.0;
#pragma unroll
          for (int q = 0; q < N; ++q) {  // W'(xj, q): symmetric / from the packed lower triangle
            const int idx = !PACKW ? q * S::P + xj[s]
                                   : ((q < xj[s]) ? colbase(q, N) + xj[s] : qcol[s] + q);
            acc += SM(S::rW + idx) * f[q];
          }
          if (xok[s]) SM(S::rG + xj[s]) = SM(S::rV + xj[s]) - acc;
        }
      }
      // Own columns of Z = [B | A] stay in registers for the whole stage.
      double zu[SU][N], zx[SX][N];
#pragma unroll
      for (int s = 0; s < SU; ++s)
#pragma unroll
        for (int q = 0; q < N; ++q) zu[s][q] = SM(S::rZ + uj[s] * S::P + q);
#pragma unroll
      for (int s = 0; s < SX; ++s)
#pragma unroll
        for (int q = 0; q < N; ++q) zx[s][q] = SM(S::rZ + (M + xj[s]) * S::P + q);
      __syncwarp();  // g complete; every lane is done with v', delta'

      update_delta();  // node k

      // Psi = [R M'; M Q] + Z' (W' Z), own columns (block-lower), and
      // [h; w] = [r; q] + Z' g.  One ROLLED loop over the rows p of S = W' Z keeps
      // the instruction footprint small: row p of S (own columns) is formed from
      // row p of W' and immediately consumed by the rank-1 update of Psi.
      double Puu[SU][M], Pxu[SU][N], hu[SU];
#pragma unroll
      for (int s = 0; s < SU; ++s) {
#pragma unroll
        for (int i = 0; i < M; ++i) Puu[s][i] = 0.0;
#pragma unroll
        for (int x = 0; x < N; ++x) Pxu[s][x] = 0.0;
        hu[s] = 0.0;
      }
#pragma unroll
      for (int s = 0; s < SX; ++s) {
#pragma unroll
        for (int i = 0; i < N; ++i) V[s][i] = 0.0;
        vv[s] = 0.0;
      }
      if (SOLVE) {  // [h; w] = Z' g with the own columns of Z already in registers
#pragma unroll
        for (int q = 0; q < N; ++q) {
          const double gq = SM(S::rG + q);
#pragma unroll
          for (int s = 0; s < SU; ++s) hu[s] += zu[s][q] * gq;
#pragma unroll
          for (int s = 0; s < SX; ++s) vv[s] += zx[s][q] * gq;
        }
      }
      if constexpr (PACKW) {
        // The first half of each W' row is fetched one iteration ahead (wpre), so the
        // dot products start without waiting on shared memory; the second half and the
        // Z row are in flight while they run.  W' is packed: entry (p, q) sits at row
        // colbase(q) + p left of the diagonal and at colbase(p) + q from the diagonal on, so
        // the rolled loop over p runs in blocks of four rows -- for every q outside the block
        // the side of the diagonal is known at compile time, inside it is one select.
        constexpr int H = N / 2;
        double wpre[H];
#pragma unroll
        for (int q = 0; q < H; ++q) wpre[q] = sm[(S::rW + q) * kTile + prob];  // row 0
        const double *smW = sm + S::rW * kTile + prob;
        auto p_block = [&](auto pb_tag) {
          constexpr int LO = 4 * decltype(pb_tag)::value;
          constexpr int HI = LO + 3 < N - 1 ? LO + 3 : N - 1;  // rows LO .. HI
          int cb = colbase(LO, N);                              // colbase(p)
#pragma unroll 1
          for (int p = LO; p <= HI; ++p) {
            const double *zrow = sm + (S::rZ + p) * kTile + prob;
            double wlate[N - H];
#pragma unroll
            for (int q = H; q < N; ++q) {
              const int idx = (q < LO) ? colbase(q, N) + p
                                       : ((q >= HI) ? cb + q : (q < p ? colbase(q, N) + p : cb + q));
              wlate[q - H] = smW[idx * kTile];
            }
            double su[SU], sx[SX], su2[SU], sx2[SX];
#pragma unroll
            for (int s = 0; s < SU; ++s) su[s] = su2[s] = 0.0;
#pragma unroll
            for (int s = 0; s < SX; ++s) sx[s] = sx2[s] = 0.0;
#pragma unroll
            for (int q = 0; q < H; ++q) {
              const double w = wpre[q];
              if (q & 1) {
#pragma unroll
                for (int s = 0; s < SU; ++s) su2[s] += w * zu[s][q];
#pragma unroll
                for (int s = 0; s < SX; ++s) sx2[s] += w * zx[s][q];
              } else {
#pragma unroll
                for (int s = 0; s < SU; ++s) su[s] += w * zu[s][q];
#pragma unroll
                for (int s = 0; s < SX; ++s) sx[s] += w * zx[s][q];
              }
            }
            if (p + 1 < N) {  // prefetch the head of the next row, pn = p + 1 in LO + 1 .. HI + 1
              const int pn = p + 1, cbn = cb + (N - 1 - p);
#pragma unroll
              for (int q = 0; q < H; ++q) {
                const int idx = (q < LO + 1) ? colbase(q, N) + pn
                                             : ((q >= HI + 1) ? cbn + q
                                                              : (q < pn ? colbase(q, N) + pn : cbn + q));
                wpre[q] = smW[idx * kTile];
              }
            }
#pragma unroll
            for (int q = H; q < N; ++q) {
              const double w = wlate[q - H];
              if (q & 1) {
#pragma unroll
                for (int s = 0; s < SU; ++s) su2[s] += w * zu[s][q];
#pragma unroll
                for (int s = 0; s < SX; ++s) sx2[s] += w * zx[s][q];
              } else {
#pragma unroll
                for (int s = 0; s < SU; ++s) su[s] += w * zu[s][q];
#pragma unroll
                for (int s = 0; s < SX; ++s) sx[s] += w * zx[s][q];
              }
            }
#pragma unroll
            for (int s = 0; s < SU; ++s) su[s] += su2[s];
#pragma unroll
            for (int s = 0; s < SX; ++s) sx[s] += sx2[s];
#pragma unroll
            for (int i = 0; i < M; ++i) {  // B(p, i)
              const double z = zrow[i * S::P * kTile];
#pragma unroll
              for (int s = 0; s < SU; ++s)
                if (i >= kGroup * s) Puu[s][i] += z * su[s];
            }
#pragma unroll
            for (int x = 0; x < N; ++x) {  // A(p, x)
              const double z = zrow[(M + x) * S::P * kTile];
#pragma unroll
              for (int s = 0; s < SU; ++s) Pxu[s][x] += z * su[s];
#pragma unroll
              for (int s = 0; s < SX; ++s)
                if (x >= kGroup * s) V[s][x] += z * sx[s];
            }
            cb += N - 1 - p;
          }
        };
        p_block(std::integral_constant<int, 0>{});
        if constexpr (N > 4) p_block(std::integral_constant<int, 1>{});
        if constexpr (N > 8) p_block(std::integral_constant<int, 2>{});
        if constexpr (N > 12) p_block(std::integral_constant<int, 3>{});
        static_assert(N <= 16, "p loop blocks cover N <= 16");
      } else {
        // The first half of each W' row is fetched one iteration ahead (wpre), so the
        // dot products start without waiting on shared memory; the second half and the
        // Z row are in flight while they run.
        constexpr int H = N / 2;
        double wpre[H];
#pragma unroll
        for (int q = 0; q < H; ++q) wpre[q] = sm[(S::rW + q) * kTile + prob];
#pragma unroll 1
        for (int p = 0; p < N; ++p) {
          const double *wrow = sm + (S::rW + p * S::P) * kTile + prob;
          const double *zrow = sm + (S::rZ + p) * kTile + prob;
          double wlate[N - H];
#pragma unroll
          for (int q = H; q < N; ++q) wlate[q - H] = wrow[q * kTile];
          double su[SU], sx[SX], su2[SU], sx2[SX];
#pragma unroll
          for (int s = 0; s < SU; ++s) su[s] = su2[s] = 0.0;
#pragma unroll
          for (int s = 0; s < SX; ++s) sx[s] = sx2[s] = 0.0;
#pragma unroll
          for (int q = 0; q < H; ++q) {
            const double w = wpre[q];
            if (q & 1) {
#pragma unroll
              for (int s = 0; s < SU; ++s) su2[s] += w * zu[s][q];
#pragma unroll
              for (int s = 0; s < SX; ++s) sx2[s] += w * zx[s][q];
            } else {
#pragma unroll
              for (int s = 0; s < SU; ++s) su[s] += w * zu[s][q];
#pragma unroll
              for (int s = 0; s < SX; ++s) sx[s] += w * zx[s][q];
            }
          }
          {  // prefetch the head of the next row (row 0 again on the last iteration)
            const double *wnext = sm + (S::rW + (p + 1 < N ? p + 1 : 0) * S::P) * kTile + prob;
#pragma unroll
            for (int q = 0; q < H; ++q) wpre[q] = wnext[q * kTile];
          }
#pragma unroll
          for (int q = H; q < N; ++q) {
            const double w = wlate[q - H];
            if (q & 1) {
#pragma unroll
              for (int s = 0; s < SU; ++s) su2[s] += w * zu[s][q];
#pragma unroll
              for (int s = 0; s < SX; ++s) sx2[s] += w * zx[s][q];
            } else {
#pragma unroll
              for (int s = 0; s < SU; ++s) su[s] += w * zu[s][q];
#pragma unroll
              for (int s = 0; s < SX; ++s) sx[s] += w * zx[s][q];
            }
          }
#pragma unroll
          for (int s = 0; s < SU; ++s) su[s] += su2[s];
#pragma unroll
          for (int s = 0; s < SX; ++s) sx[s] += sx2[s];
#pragma unroll
          for (int i = 0; i < M; ++i) {  // B(p, i)
            const double z = zrow[i * S::P * kTile];
#pragma unroll
            for (int s = 0; s < SU; ++s)
              if (i >= kGroup * s) Puu[s][i] += z * su[s];
          }
#pragma unroll
          for (int x = 0; x < N; ++x) {  // A(p, x)
            const double z = zrow[(M + x) * S::P * kTile];
#pragma unroll
            for (int s = 0; s < SU; ++s) Pxu[s][x] += z * su[s];
#pragma unroll
            for (int s = 0; s < SX; ++s)
              if (x >= kGroup * s) V[s][x] += z * sx[s];
          }
        }
      }
#pragma unroll
      for (int s = 0; s < SU; ++s) {
#pragma unroll
        for (int i = kGroup * s; i < M; ++i) Puu[s][i] += SM(S::rR + rcol[s] + i);
#pragma unroll
        for (int x = 0; x < N; ++x) Pxu[s][x] += SM(S::rM + uj[s] * S::P + x);
        if (SOLVE) hu[s] += SM(S::rr + uj[s]);
      }
#pragma unroll
      for (int s = 0; s < SX; ++s) {
#pragma unroll
        for (int i = kGroup * s; i < N; ++i) V[s][i] += SM(S::rQ + qcol[s] + i);
        if (SOLVE) vv[s] += SM(S::rq + xj[s]);
      }
      __syncwarp();  // every lane has taken its Q / M / R entries: their rows become X
      // Publish the control block: Psi_uu (packed lower), Psi_xu, h.
#pragma unroll
      for (int s = 0; s < SU; ++s) {
        if (uok[s]) {
#pragma unroll
          for (int i = kGroup * s; i < M; ++i)
            if (i >= uj[s]) SM(S::xGuu + rcol[s] + i) = Puu[s][i];
#pragma unroll
          for (int x = 0; x < N; ++x) SM(S::xPxu + uj[s] * S::P + x) = Pxu[s][x];
          if (SOLVE) SM(S::xH + uj[s]) = hu[s];
        }
      }
      __syncwarp();  // control block visible; staged operands of stage k consumed

      if (k > 0) {
        issue_z_vec(true);
        cp_async_commit();
      }

      // Cholesky of G (replicated), Lambda (own rows), K (own columns), t, k.
      double Lg[tri(M)], dg[M];
#pragma unroll
      for (int t = 0; t < tri(M); ++t) Lg[t] = SM(S::xGuu + t);
      bool g_ok = true;
#pragma unroll
      for (int j = 0; j < M; ++j) {
        double x = Lg[pk(j, j, M)];
#pragma unroll
        for (int q = 0; q < j; ++q) x -= Lg[pk(j, q, M)] * Lg[pk(j, q, M)];
        g_ok = g_ok && (x > 0.0);
        const double d = rsqrt(x);
        dg[j] = d;
#pragma unroll
        for (int i = j + 1; i < M; ++i) {
          double t = Lg[pk(i, j, M)];
#pragma unroll
          for (int q = 0; q < j; ++q) t -= Lg[pk(i, q, M)] * Lg[pk(j, q, M)];
          Lg[pk(i, j, M)] = t * d;
        }
      }
      if (!g_ok && status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_G_FACTORIZATION_FAILURE;

      double tt[M];
      if (SOLVE) {
#pragma unroll
        for (int a = 0; a < M; ++a) {
          double t = SM(S::xH + a);
#pragma unroll
          for (int c = 0; c < a; ++c) t -= Lg[pk(a, c, M)] * tt[c];
          tt[a] = t * dg[a];
        }
        // k_k = -L_G^-T t
        double kk[M];
#pragma unroll
        for (int a = M - 1; a >= 0; --a) {
          double t = tt[a];
#pragma unroll
          for (int c = a + 1; c < M; ++c) t -= Lg[pk(c, a, M)] * kk[c];
          kk[a] = t * dg[a];
        }
        if (valid && r == 0) {
          double *dst = kst;
#pragma unroll
          for (int a = 0; a < M; ++a) {
            stcs(dst, -kk[a]);
            dst += ld;
          }
        }
        kst -= static_cast<int64_t>(M) * ld;
      }
      {
        // G^-1 = L_G^-T L_G^-1 (packed lower) for later solves against this factor.
        double Gi[tri(M)];
#pragma unroll
        for (int j = 0; j < M; ++j)
#pragma unroll
          for (int i = j; i < M; ++i) {
            double t = (i == j) ? 1.0 : 0.0;
#pragma unroll
            for (int q = j; q < i; ++q) t -= Lg[pk(i, q, M)] * Gi[pk(q, j, M)];
            Gi[pk(i, j, M)] = t * dg[i];
          }
        if (valid && r == 0) {
          double *dst = Gst;
#pragma unroll
          for (int j = 0; j < M; ++j)
#pragma unroll
            for (int i = j; i < M; ++i) {
              double t = 0.0;
#pragma unroll
              for (int q = i; q < M; ++q) t += Gi[pk(q, i, M)] * Gi[pk(q, j, M)];
              stcs(dst, t);
              dst += ld;
            }
        }
        Gst -= static_cast<int64_t>(tri(M)) * ld;
      }

      double lam[SX][M];
#pragma unroll
      for (int s = 0; s < SX; ++s) {
#pragma unroll
        for (int a = 0; a < M; ++a) {
          double t = SM(S::xPxu + a * S::P + xj[s]);
#pragma unroll
          for (int c = 0; c < a; ++c) t -= lam[s][c] * Lg[pk(a, c, M)];
          lam[s][a] = t * dg[a];
        }
        if (xok[s]) {
#pragma unroll
          for (int a = 0; a < M; ++a) SM(S::xLam + a * S::P + xj[s]) = lam[s][a];
        }
        // K(:, xj) = -L_G^-T Lambda(xj, :)'
        double kap[M];
#pragma unroll
        for (int a = M - 1; a >= 0; --a) {
          double t = lam[s][a];
#pragma unroll
          for (int c = a + 1; c < M; ++c) t -= Lg[pk(c, a, M)] * kap[c];
          kap[a] = t * dg[a];
        }
        if (valid && xok[s]) {
          double *dst = Kst + static_cast<int64_t>(xj[s] * M) * ld;
#pragma unroll
          for (int a = 0; a < M; ++a) {
            stcs(dst, -kap[a]);
            dst += ld;
          }
        }
      }
      Kst -= static_cast<int64_t>(N) * M * ld;
      __syncwarp();  // Lambda visible

      // V_k = Psi_xx - Lambda Lambda', v_k = w - Lambda t (own columns).
#pragma unroll
      for (int s = 0; s < SX; ++s) {
#pragma unroll
        for (int i = kGroup * s; i < N; ++i) {
          double t = V[s][i];
#pragma unroll
          for (int a = 0; a < M; ++a) t -= SM(S::xLam + a * S::P + i) * lam[s][a];
          V[s][i] = t;
        }
        if (SOLVE) {
          double t = vv[s];
#pragma unroll
          for (int a = 0; a < M; ++a) t -= lam[s][a] * tt[a];
          vv[s] = t;
        }
      }
    }

    // ---- node k: compute_delta_sqrt + factor_F + compute_regularized_W --------
    // (lqr.cpp:475-529): V, v in registers -> W_k in shared memory and in the
    // store, v_k in shared memory and in the spill.
    double sdo[SX], sdio[SX], sd[N];
#pragma unroll
    for (int s = 0; s < SX; ++s) {
      sdo[s] = SM(S::rSd + xj[s]);
      sdio[s] = SM(S::rSdi + xj[s]);
    }
#pragma unroll
    for (int i = 0; i < N; ++i) sd[i] = SM(S::rSd + i);
    // Own columns of F = I + D^1/2 V D^1/2 (rows >= 4 s).
#pragma unroll
    for (int s = 0; s < SX; ++s)
#pragma unroll
      for (int i = kGroup * s; i < N; ++i)
        V[s][i] = sd[i] * V[s][i] * sdo[s] + (i == xj[s] ? 1.0 : 0.0);
    __syncwarp();  // every lane is done with the exchange region (Lambda)
    // F goes through the W rows (W_{k+1} is consumed), so the exchange rows can take the
    // next stage's Q, M, R right away and the copy lands while F is factored.
    if (k > 0) {
      issue_qmr(true);
      cp_async_commit();
    }
#pragma unroll
    for (int s = 0; s < SX; ++s) {
      if (SOLVE && xok[s]) {
        SM(S::rV + xj[s]) = vv[s];
        if (valid) stcs(vst + static_cast<int64_t>(xj[s]) * ld, vv[s]);
      }
    }
    if (SOLVE) vst -= static_cast<int64_t>(N) * ld;
    if (__ballot_sync(0xffffffffu, bad_delta) & group_mask) {
      if (status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_INVALID_DELTA;
    }

    // Cholesky of F = L L' (the diagonal of L keeps the pivots, dinv their rsqrt), blocked
    // by kGroup columns: diagonal block b holds own column xj[b] of every lane.  Per block
    // the lanes publish their columns of the block, every lane factors the diagonal block
    // (replicated, so the rsqrt -> mul -> FMA chain needs no exchange), each lane solves
    // its own rows xj[s] of the panel below and publishes them, and each lane applies the
    // block's update to its own later columns.  Every entry takes its updates in ascending
    // pivot order and the same scaling as the unblocked right-looking form, so L is the
    // same to the bit; the trailing FMAs are split four ways instead of replicated.
    double L[tri(N)], dinv[N];
    bool f_ok = true;
    // One call per block with b a compile-time constant: a partial last block (n = 6) kept a
    // plain unrolled loop from resolving the indices of L, which then went to local memory.
    auto f_block = [&](auto b_tag) {
      constexpr int b = decltype(b_tag)::value;
      constexpr int j0 = kGroup * b, j1 = j0 + kGroup < N ? j0 + kGroup : N;
      if (xok[b]) {
#pragma unroll
        for (int i = j0; i < N; ++i)
          if (i >= xj[b]) SM(S::rW + qcol[b] + i) = V[b][i];
      }
      __syncwarp();  // columns j0 .. j1 - 1 of F, all updates of earlier blocks applied
#pragma unroll
      for (int j = j0; j < j1; ++j)
#pragma unroll
        for (int i = j; i < j1; ++i) L[pk(i, j, N)] = SM(S::rW + pk(i, j, N));
#pragma unroll
      for (int j = j0; j < j1; ++j) {
        const double x = L[pk(j, j, N)];
        f_ok = f_ok && (x > 0.0);
        const double d = rsqrt(x);
        dinv[j] = d;
#pragma unroll
        for (int i = j + 1; i < j1; ++i) L[pk(i, j, N)] *= d;
#pragma unroll
        for (int c = j + 1; c < j1; ++c)
#pragma unroll
          for (int i = c; i < j1; ++i) L[pk(i, c, N)] -= L[pk(i, j, N)] * L[pk(c, j, N)];
      }
      if constexpr (b + 1 < SX) {
        // Own rows xj[s] of the panel: L(xj, j) for the block's columns j.
        double lr[SX][kGroup];
#pragma unroll
        for (int s = b + 1; s < SX; ++s) {
#pragma unroll
          for (int j = j0; j < j1; ++j) {
            double t = SM(S::rW + colbase(j, N) + xj[s]);
#pragma unroll
            for (int q = j0; q < j; ++q) t -= lr[s][q - j0] * L[pk(j, q, N)];
            lr[s][j - j0] = t * dinv[j];
          }
          if (xok[s]) {
#pragma unroll
            for (int j = j0; j < j1; ++j) SM(S::rW + colbase(j, N) + xj[s]) = lr[s][j - j0];
          }
        }
        __syncwarp();  // the panel of the block is solved
#pragma unroll
        for (int j = j0; j < j1; ++j)
#pragma unroll
          for (int i = j1; i < N; ++i) L[pk(i, j, N)] = SM(S::rW + pk(i, j, N));
#pragma unroll
        for (int s = b + 1; s < SX; ++s)
#pragma unroll
          for (int j = j0; j < j1; ++j)
#pragma unroll
            for (int i = kGroup * s; i < N; ++i) V[s][i] -= L[pk(i, j, N)] * lr[s][j - j0];
      }
    };
    f_block(std::integral_constant<int, 0>{});
    if constexpr (SX > 1) f_block(std::integral_constant<int, 1>{});
    if constexpr (SX > 2) f_block(std::integral_constant<int, 2>{});
    if constexpr (SX > 3) f_block(std::integral_constant<int, 3>{});
    __syncwarp();  // every lane has read F: the W rows take W_k
    if (!f_ok && status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_F_FACTORIZATION_FAILURE;
    // Own columns of F^-1 = L^-T L^-1: forward substitution on e_xj, then backward
    // substitution, both against the lane's register copy of L (no exchange).
    // W = D^-1/2 (I - F^-1) D^-1/2, rows >= 4 s of the own columns.
    double sdi[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sdi[i] = SM(S::rSdi + i);
#pragma unroll
    for (int s = 0; s < SX; ++s) {
      // Column-oriented (axpy) substitutions: each solved entry immediately updates
      // the remaining right-hand side with independent FMAs.
      double y[N];
#pragma unroll
      for (int i = kGroup * s; i < N; ++i) y[i] = (i == xj[s]) ? 1.0 : 0.0;
#pragma unroll
      for (int i = kGroup * s; i < N; ++i) {  // L y = e_xj
        y[i] *= dinv[i];
#pragma unroll
        for (int q = i + 1; q < N; ++q) y[q] -= L[pk(q, i, N)] * y[i];
      }
#pragma unroll
      for (int i = N - 1; i >= kGroup * s; --i) {  // L' x = y
        y[i] *= dinv[i];
#pragma unroll
        for (int q = kGroup * s; q < i; ++q) y[q] -= L[pk(i, q, N)] * y[i];
      }
      double *dst = Wst + static_cast<int64_t>(qcol[s] + kGroup * s) * ld;
#pragma unroll
      for (int i = kGroup * s; i < N; ++i) {
        const double w = sdi[i] * ((i == xj[s] ? 1.0 : 0.0) - y[i]) * sdio[s];
        if (xok[s] && i >= xj[s]) {
          if constexpr (PACKW) {
            SM(S::rW + qcol[s] + i) = w;
          } else {
            SM(S::rW + xj[s] * S::P + i) = w;
            SM(S::rW + i * S::P + xj[s]) = w;
          }
          if (valid) stcs(dst, y[i]);  // the store keeps P = F^-1
        }
        dst += ld;
      }
    }
    Wst -= static_cast<int64_t>(tri(N)) * ld;
    __syncwarp();
  }

  if (status_out != nullptr && valid && r == 0) status_out[b] = status;

  if constexpr (FUSED) {
    // ---- forward phase ------------------------------------------------------------
    // Shared-memory rows (of 8 problems), over the staging area of the sweep:
    // block 1 = what u and A x + B u need, block 2 = what the node solve needs.
    constexpr int fA = 0, fB = fA + N * N, fK = fB + N * M, fk = fK + N * M;
    constexpr int fP = fk + M, fv = fP + tri(N), fd = fv + N, fc = fd + N;
    constexpr int fx = fc + N, fu = fx + N, fs = fu + M;
    static_assert(fs + N <= S::kRows, "rollout operands fit the sweep's shared memory");
    __threadfence_block();
    __syncwarp();  // the spill of every lane is visible to the copies below
    const double *gA = in.A + lane_goff, *gB = in.B + lane_goff;
    const double *gc = in.c + lane_goff, *gd = in.delta + lane_goff;
    const double *gK = store + Z::oK(T) * ld + lane_goff;
    const double *gP = store + Z::oW(T) * ld + lane_goff;
    const double *gv = scratch + Z::ov(T) * ld + lane_goff;
    const double *gk = scratch + Z::ok(T) * ld + lane_goff;
    // The copies have half a stage of lead; what they fetch is pulled into L2 kPF stages
    // earlier (prefetch.global.L2: no registers, no shared memory), so that they pay an
    // L2 round trip, not an HBM one.
    constexpr int kPF = SIPOC_FUSED_PF;
    auto l2_run = [&](const double *src, int count) {
#pragma unroll
      for (int i0 = 0; i0 < count; i0 += 8) {
        if ((lane & 1) == 0 && (i0 + 8 <= count || i0 + rr < count)) prefetch_l2(src);
        src += ld8;
      }
    };
    auto prefetch_edge = [&]() {  // edge kPF stages past the one the pointers stand on
      l2_run(gA + static_cast<int64_t>(kPF) * N * N * ld, N * N);
      l2_run(gB + static_cast<int64_t>(kPF) * N * M * ld, N * M);
      l2_run(gK + static_cast<int64_t>(kPF) * N * M * ld, N * M);
      l2_run(gk + static_cast<int64_t>(kPF) * M * ld, M);
    };
    auto prefetch_node = [&]() {
      l2_run(gP + static_cast<int64_t>(kPF) * tri(N) * ld, tri(N));
      l2_run(gv + static_cast<int64_t>(kPF) * N * ld, N);
      l2_run(gd + static_cast<int64_t>(kPF) * N * ld, N);
      l2_run(gc + static_cast<int64_t>(kPF) * N * ld, N);
    };
    auto issue_edge = [&]() {  // A_k, B_k, K_k, k_k; then step to edge k + 1
      stage_run(sdst + fA * kTile, gA, ld8, N * N, rr);
      stage_run(sdst + fB * kTile, gB, ld8, N * M, rr);
      stage_run(sdst + fK * kTile, gK, ld8, N * M, rr);
      stage_run(sdst + fk * kTile, gk, ld8, M, rr);
      gA += static_cast<int64_t>(N) * N * ld;
      gB += static_cast<int64_t>(N) * M * ld;
      gK += static_cast<int64_t>(N) * M * ld;
      gk += static_cast<int64_t>(M) * ld;
    };
    auto issue_node = [&]() {  // P, v, delta, c of the node the pointers stand on
      stage_run(sdst + fP * kTile, gP, ld8, tri(N), rr);
      stage_run(sdst + fv * kTile, gv, ld8, N, rr);
      stage_run(sdst + fd * kTile, gd, ld8, N, rr);
      stage_run(sdst + fc * kTile, gc, ld8, N, rr);
      gP += static_cast<int64_t>(tri(N)) * ld;
      gv += static_cast<int64_t>(N) * ld;
      gd += static_cast<int64_t>(N) * ld;
      gc += static_cast<int64_t>(N) * ld;
    };
    // Node solve on the own rows i = xj[s], given f (own rows) in fo[]:
    //   s = D^-1/2 f, t = P s, (I + D V)^-1 f = D^1/2 t, W f = D^-1/2 (s - t)
    // (the F-solve form of lqr.cpp:531-549; P = F^-1 from the store).  Returns t and
    // leaves s in fo; ends with the exchange rows free again.
    double fo[SX], to[SX], sdi_o[SX];
    auto node_solve = [&]() {
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        sdi_o[s] = rsqrt(SM(fd + xj[s]));
        fo[s] *= sdi_o[s];
        if (xok[s]) SM(fs + xj[s]) = fo[s];
      }
      __syncwarp();
      double sv[N];
#pragma unroll
      for (int j = 0; j < N; ++j) sv[j] = SM(fs + j);
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        double acc = 0.0, acc2 = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
          // packed lower index of (xj, j): below the diagonal j * N - j (j - 1) / 2 + xj - j
          const int below = j * N - j * (j - 1) / 2 - j + xj[s];
          const int idx = (j < xj[s]) ? below : qcol[s] + j;
          if (j & 1) acc2 += SM(fP + idx) * sv[j]; else acc += SM(fP + idx) * sv[j];
        }
        to[s] = acc + acc2;
      }
    };
    double *xo = out.x + b, *uo = out.u + b, *yo = out.y + b;

    if (kPF > 0) {
      // edges 1 .. kPF and nodes 2 .. kPF + 1 (the loop below keeps the distance)
      for (int j = 1; j <= kPF; ++j) {
        if (j < T) {
          l2_run(gA + static_cast<int64_t>(j) * N * N * ld, N * N);
          l2_run(gB + static_cast<int64_t>(j) * N * M * ld, N * M);
          l2_run(gK + static_cast<int64_t>(j) * N * M * ld, N * M);
          l2_run(gk + static_cast<int64_t>(j) * M * ld, M);
        }
        if (j + 1 <= T) {
          l2_run(gP + static_cast<int64_t>(j + 1) * tri(N) * ld, tri(N));
          l2_run(gv + static_cast<int64_t>(j + 1) * N * ld, N);
          l2_run(gd + static_cast<int64_t>(j + 1) * N * ld, N);
          l2_run(gc + static_cast<int64_t>(j + 1) * N * ld, N);
        }
      }
    }
    issue_node();  // root
    cp_async_commit();
    if (T > 0) issue_edge();
    cp_async_commit();
    cp_async_wait_group<1>();
    __syncwarp();
    if (SEGMENTED && seg > 0) {
      // the segment starts from the boundary state; its first node's x, y are the previous
      // segment's last and are written there
#pragma unroll
      for (int s = 0; s < SX; ++s)
        if (xok[s])
          SM(fx + xj[s]) = __ldg(sg.xb + (static_cast<int64_t>(seg) * N + xj[s]) * ld + b);
    } else {
      // root: f = delta v - c, x = -(I + D V)^-1 f, y = v - W f     (lqr.cpp:798-819)
#pragma unroll
      for (int s = 0; s < SX; ++s)
        fo[s] = SM(fd + xj[s]) * SM(fv + xj[s]) - SM(fc + xj[s]);
      node_solve();
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        const double xi = -SM(fd + xj[s]) * sdi_o[s] * to[s];
        const double yi = SM(fv + xj[s]) - sdi_o[s] * (fo[s] - to[s]);
        if (xok[s]) {
          SM(fx + xj[s]) = xi;
          if (valid) {
            stcs(xo + static_cast<int64_t>(xj[s]) * ld, xi);
            stcs(yo + static_cast<int64_t>(xj[s]) * ld, yi);
          }
        }
      }
    }
    __syncwarp();  // x_0 visible; every lane is done with the node block
    if (T > 0) issue_node();
    cp_async_commit();
    xo += static_cast<int64_t>(N) * ld;
    yo += static_cast<int64_t>(N) * ld;

#ifdef SIPOC_EXP_SKIP_FWD
    if (T > 0) { cp_async_wait_all(); return; }
#endif
    for (int k = 0; k < T; ++k) {
#ifndef SIPOC_EXP_NOWAIT
      cp_async_wait_group<1>();  // edge block of stage k
#endif
      __syncwarp();
      double xr[N];
#pragma unroll
      for (int j = 0; j < N; ++j) xr[j] = SM(fx + j);
      // u = k + K x, own controls                                   (lqr.cpp:856-857)
#pragma unroll
      for (int s = 0; s < SU; ++s) {
        double acc = SM(fk + uj[s]), acc2 = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
          if (j & 1) acc2 += SM(fK + j * M + uj[s]) * xr[j]; else acc += SM(fK + j * M + uj[s]) * xr[j];
        }
        acc += acc2;
        if (uok[s]) {
          SM(fu + uj[s]) = acc;
          if (valid) stcs(uo + static_cast<int64_t>(uj[s]) * ld, acc);
        }
      }
      uo += static_cast<int64_t>(M) * ld;
      // A x, own rows (needs x only: runs while the lanes' u meet below)
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        double acc = 0.0, acc2 = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
          if (j & 1) acc2 += SM(fA + j * N + xj[s]) * xr[j]; else acc += SM(fA + j * N + xj[s]) * xr[j];
        }
        fo[s] = acc + acc2;
      }
      __syncwarp();  // u visible
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        double acc = 0.0;
#pragma unroll
        for (int a = 0; a < M; ++a) acc += SM(fB + a * N + xj[s]) * SM(fu + a);
        fo[s] += acc;
      }
      __syncwarp();  // every lane is done with the edge block
      if (kPF > 0 && k + 1 + kPF < T) prefetch_edge();
      if (k + 1 < T) issue_edge();
      cp_async_commit();
#ifndef SIPOC_EXP_NOWAIT
      cp_async_wait_group<1>();  // node block of stage k (node k + 1)
#endif
      __syncwarp();
      // f = c' - delta' o v' + A x + B u ; x' = (I + D V)^-1 f ; y' = v' + W f   (:859-868)
#pragma unroll
      for (int s = 0; s < SX; ++s)
        fo[s] += SM(fc + xj[s]) - SM(fd + xj[s]) * SM(fv + xj[s]);
      node_solve();
#pragma unroll
      for (int s = 0; s < SX; ++s) {
        const double xi = SM(fd + xj[s]) * sdi_o[s] * to[s];
        const double yi = SM(fv + xj[s]) + sdi_o[s] * (fo[s] - to[s]);
        if (xok[s]) {
          SM(fx + xj[s]) = xi;
          if (valid) {
            stcs(xo + static_cast<int64_t>(xj[s]) * ld, xi);
            stcs(yo + static_cast<int64_t>(xj[s]) * ld, yi);
          }
        }
      }
      xo += static_cast<int64_t>(N) * ld;
      yo += static_cast<int64_t>(N) * ld;
      __syncwarp();  // x' visible; node block free
      if (kPF > 0 && k + 2 + kPF <= T) prefetch_node();  // pointers stand on node k + 2
      if (k + 1 < T) issue_node();
      cp_async_commit();
    }
    cp_async_wait_all();
  }
#undef SM
}

// ===========================================================================
// Backward sweep, one thread per problem, registers only (tiny n).
// ===========================================================================
template <int N, int M, bool SOLVE>
__global__ void __launch_bounds__(64)
riccati_backward_thread(LqrIn in, int *status_out, double *store, double *scratch,
                        int64_t batch, int64_t ld, int T) {
  using Z = FastSizes<N, M>;
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const size_t L_ = static_cast<size_t>(ld);
#define G(ptr, e) ldcs((ptr) + static_cast<size_t>(e) * L_ + b)
  double *Wst = store + Z::oW(T) * ld + b;
  double *Kst = store + Z::oK(T) * ld + b;
  double *Gst = store + Z::oG(T) * ld + b;
  double *vst = SOLVE ? scratch + Z::ov(T) * ld + b : nullptr;
  double *kst = SOLVE ? scratch + Z::ok(T) * ld + b : nullptr;

  int status = SIPOC_FACTOR_SUCCESS;
  double W[tri(N)], v[N], dl[N];

  // V (packed lower), vv, delta of node k -> W, v, dl; stores W_k, v_k.
  auto process_node = [&](int k, double (&V)[tri(N)], double (&vv)[N], const double (&dk)[N]) {
    double sd[N], sdi[N];
    bool d_ok = true;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double d = dk[i];
      d_ok = d_ok && (d > 0.0);
      dl[i] = d;
      sdi[i] = rsqrt(d);   // (sqrt + division were 21 % of this kernel's stall samples)
      sd[i] = d * sdi[i];
    }
    if (!d_ok && status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_INVALID_DELTA;
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = j; i < N; ++i)
        V[pk(i, j, N)] = sd[i] * V[pk(i, j, N)] * sd[j] + (i == j ? 1.0 : 0.0);
    double dinv[N];
    bool f_ok = true;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double x = V[pk(j, j, N)];
#pragma unroll
      for (int p = 0; p < j; ++p) x -= V[pk(j, p, N)] * V[pk(j, p, N)];
      f_ok = f_ok && (x > 0.0);
      const double d = rsqrt(x);
      dinv[j] = d;
#pragma unroll
      for (int i = j + 1; i < N; ++i) {
        double t = V[pk(i, j, N)];
#pragma unroll
        for (int p = 0; p < j; ++p) t -= V[pk(i, p, N)] * V[pk(j, p, N)];
        V[pk(i, j, N)] = t * d;
      }
    }
    if (!f_ok && status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_F_FACTORIZATION_FAILURE;
    double Li[tri(N)];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = j; i < N; ++i) {
        double t = (i == j) ? 1.0 : 0.0;
#pragma unroll
        for (int p = j; p < i; ++p) t -= V[pk(i, p, N)] * Li[pk(p, j, N)];
        Li[pk(i, j, N)] = t * dinv[i];
      }
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = j; i < N; ++i) {
        double fin = 0.0;
#pragma unroll
        for (int p = i; p < N; ++p) fin += Li[pk(p, i, N)] * Li[pk(p, j, N)];
        const double w = sdi[i] * ((i == j ? 1.0 : 0.0) - fin) * sdi[j];
        W[pk(i, j, N)] = w;
        stcs(Wst + (static_cast<int64_t>(k) * tri(N) + pk(i, j, N)) * ld, fin);  // P = F^-1
      }
#pragma unroll
    for (int i = 0; i < N; ++i) {
      v[i] = vv[i];
      if (SOLVE) stcs(vst + static_cast<int64_t>(k * N + i) * ld, vv[i]);
    }
  };

  // Inputs of the stage to process next, fetched one stage ahead: the loads are issued
  // in the middle of the previous stage (once its products are formed and their
  // registers are free) and land while its factorizations run.
  double nA[N * N], nB[N * M], nQ[tri(N)], nM[N * M], nR[tri(M)], nq[N], nr[M], nc[N], nd[N];
  auto fetch_stage = [&](int k) {
#pragma unroll
    for (int t = 0; t < N * M; ++t) {
      nB[t] = G(in.B, k * N * M + t);
      nM[t] = G(in.M, k * N * M + t);
    }
#pragma unroll
    for (int t = 0; t < N * N; ++t) nA[t] = G(in.A, k * N * N + t);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = j; i < N; ++i) nQ[pk(i, j, N)] = G(in.Q, (k * N + j) * N + i);
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
      for (int i = j; i < M; ++i) nR[pk(i, j, M)] = G(in.R, (k * M + j) * M + i);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      nd[i] = G(in.delta, k * N + i);
      nq[i] = SOLVE ? G(in.q, k * N + i) : 0.0;
      nc[i] = SOLVE ? G(in.c, (k + 1) * N + i) : 0.0;
    }
#pragma unroll
    for (int a = 0; a < M; ++a) nr[a] = SOLVE ? G(in.r, k * M + a) : 0.0;
  };

  {
    double V[tri(N)], vv[N], dT[N];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = j; i < N; ++i) V[pk(i, j, N)] = G(in.Q, (T * N + j) * N + i);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = SOLVE ? G(in.q, T * N + i) : 0.0;
      dT[i] = G(in.delta, T * N + i);
    }
    if (T > 0) fetch_stage(T - 1);
    process_node(T, V, vv, dT);
  }

  for (int k = T - 1; k >= 0; --k) {
    // Z = [B | A] and the rest of the stage, from the prefetch registers.
    double Zm[N + M][N], dk[N];
#pragma unroll
    for (int a = 0; a < M; ++a)
#pragma unroll
      for (int p = 0; p < N; ++p) Zm[a][p] = nB[a * N + p];
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int p = 0; p < N; ++p) Zm[M + j][p] = nA[j * N + p];
#pragma unroll
    for (int i = 0; i < N; ++i) dk[i] = nd[i];
    double g[N];
    if (SOLVE) {
      double f[N];
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] = dl[i] * v[i] - nc[i];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < N; ++q) acc += W[q <= i ? pk(i, q, N) : pk(q, i, N)] * f[q];
        g[i] = v[i] - acc;
      }
    }
    // S = W' Z
    double Sm[N + M][N];
#pragma unroll
    for (int c = 0; c < N + M; ++c)
#pragma unroll
      for (int i = 0; i < N; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < N; ++q) acc += W[q <= i ? pk(i, q, N) : pk(q, i, N)] * Zm[c][q];
        Sm[c][i] = acc;
      }
    // Psi (lower) and [h; w]
    double Puu[tri(M)], Pxu[M][N], Pxx[tri(N)], hu[M], wx[N];
#pragma unroll
    for (int j = 0; j < M; ++j) {
#pragma unroll
      for (int i = j; i < M; ++i) {
        double acc = nR[pk(i, j, M)];
#pragma unroll
        for (int p = 0; p < N; ++p) acc += Zm[i][p] * Sm[j][p];
        Puu[pk(i, j, M)] = acc;
      }
#pragma unroll
      for (int x = 0; x < N; ++x) {
        double acc = nM[j * N + x];
#pragma unroll
        for (int p = 0; p < N; ++p) acc += Zm[M + x][p] * Sm[j][p];
        Pxu[j][x] = acc;
      }
      double acc = 0.0;
      if (SOLVE) {
        acc = nr[j];
#pragma unroll
        for (int p = 0; p < N; ++p) acc += Zm[j][p] * g[p];
      }
      hu[j] = acc;
    }
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
      for (int i = j; i < N; ++i) {
        double acc = nQ[pk(i, j, N)];
#pragma unroll
        for (int p = 0; p < N; ++p) acc += Zm[M + i][p] * Sm[M + j][p];
        Pxx[pk(i, j, N)] = acc;
      }
      double acc = 0.0;
      if (SOLVE) {
        acc = nq[j];
#pragma unroll
        for (int p = 0; p < N; ++p) acc += Zm[M + j][p] * g[p];
      }
      wx[j] = acc;
    }
    if (k > 0) fetch_stage(k - 1);  // products formed: their registers take the next stage
    // Cholesky of G
    double dg[M];
    bool g_ok = true;
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double x = Puu[pk(j, j, M)];
#pragma unroll
      for (int p = 0; p < j; ++p) x -= Puu[pk(j, p, M)] * Puu[pk(j, p, M)];
      g_ok = g_ok && (x > 0.0);
      const double d = rsqrt(x);
      dg[j] = d;
#pragma unroll
      for (int i = j + 1; i < M; ++i) {
        double t = Puu[pk(i, j, M)];
#pragma unroll
        for (int p = 0; p < j; ++p) t -= Puu[pk(i, p, M)] * Puu[pk(j, p, M)];
        Puu[pk(i, j, M)] = t * d;
      }
    }
    if (!g_ok && status == SIPOC_FACTOR_SUCCESS) status = SIPOC_FACTOR_G_FACTORIZATION_FAILURE;
    double tt[M];
    if (SOLVE) {
#pragma unroll
      for (int a = 0; a < M; ++a) {
        double t = hu[a];
#pragma unroll
        for (int c = 0; c < a; ++c) t -= Puu[pk(a, c, M)] * tt[c];
        tt[a] = t * dg[a];
      }
      double kk[M];
#pragma unroll
      for (int a = M - 1; a >= 0; --a) {
        double t = tt[a];
#pragma unroll
        for (int c = a + 1; c < M; ++c) t -= Puu[pk(c, a, M)] * kk[c];
        kk[a] = t * dg[a];
        stcs(kst + static_cast<int64_t>(k * M + a) * ld, -kk[a]);
      }
    }
    {
      double Gi[tri(M)];
#pragma unroll
      for (int j = 0; j < M; ++j)
#pragma unroll
        for (int i = j; i < M; ++i) {
          double t = (i == j) ? 1.0 : 0.0;
#pragma unroll
          for (int p = j; p < i; ++p) t -= Puu[pk(i, p, M)] * Gi[pk(p, j, M)];
          Gi[pk(i, j, M)] = t * dg[i];
        }
#pragma unroll
      for (int j = 0; j < M; ++j)
#pragma unroll
        for (int i = j; i < M; ++i) {
          double t = 0.0;
#pragma unroll
          for (int p = i; p < M; ++p) t += Gi[pk(p, i, M)] * Gi[pk(p, j, M)];
          stcs(Gst + (static_cast<int64_t>(k) * tri(M) + pk(i, j, M)) * ld, t);
        }
    }
    // Lambda, K, V, v
    double lam[N][M];
#pragma unroll
    for (int x = 0; x < N; ++x) {
#pragma unroll
      for (int a = 0; a < M; ++a) {
        double t = Pxu[a][x];
#pragma unroll
        for (int c = 0; c < a; ++c) t -= lam[x][c] * Puu[pk(a, c, M)];
        lam[x][a] = t * dg[a];
      }
      double kap[M];
#pragma unroll
      for (int a = M - 1; a >= 0; --a) {
        double t = lam[x][a];
#pragma unroll
        for (int c = a + 1; c < M; ++c) t -= Puu[pk(c, a, M)] * kap[c];
        kap[a] = t * dg[a];
        stcs(Kst + (static_cast<int64_t>(k) * N * M + x * M + a) * ld, -kap[a]);
      }
    }
    double vv[N];
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
      for (int i = j; i < N; ++i) {
        double t = Pxx[pk(i, j, N)];
#pragma unroll
        for (int a = 0; a < M; ++a) t -= lam[i][a] * lam[j][a];
        Pxx[pk(i, j, N)] = t;
      }
      double t = wx[j];
      if (SOLVE) {
#pragma unroll
        for (int a = 0; a < M; ++a) t -= lam[j][a] * tt[a];
      }
      vv[j] = t;
    }
    process_node(k, Pxx, vv, dk);
  }
  if (status_out != nullptr) status_out[b] = status;
#undef G
}

// ===========================================================================
// Backward affine sweep against a kept factorization (lqr.cpp:738-796), small batches:
// one thread per problem, one warp per block, every operand of a stage copied to shared
// memory with cp.async NBUF - 1 stages ahead of its use ([row][lane]: conflict-free, and
// a thread only ever reads what it copied itself, so no barrier is involved).  At a few
// thousand problems there are not enough threads to hide HBM latency by occupancy -- the
// register-staged kernel below pays three dependent round trips per stage -- so the
// latency is taken off the chain instead: a stage costs its arithmetic, not its loads.
// ===========================================================================
template <int N, int M>
struct AffineRows {
  static constexpr int rW = 0, rD = rW + tri(N), rC = rD + N, rB = rC + N, rK = rB + N * M,
                       rG = rK + N * M, rR = rG + tri(M), rA = rR + M, rQ = rA + N * N,
                       kRows = rQ + N;
  // stages in flight: as many 32-lane buffers as fit in ~96 KB (two blocks per SM), 2..4
  static constexpr int kBuf =
      (96 * 1024) / (kRows * 32 * 8) >= 4 ? 4 : ((96 * 1024) / (kRows * 32 * 8) >= 3 ? 3 : 2);
  static constexpr int kBytes = kBuf * kRows * 32 * int(sizeof(double));
};

template <int N, int M>
__global__ void __launch_bounds__(32)
affine_backward_staged(LqrIn in, const double *store, double *scratch, int64_t batch, int64_t ld,
                       int T) {
  using Z = FastSizes<N, M>;
  using R = AffineRows<N, M>;
  constexpr int NBUF = R::kBuf;
  extern __shared__ __align__(16) double sm_affine[];
  const int lane = threadIdx.x;
  const int64_t b_raw = static_cast<int64_t>(blockIdx.x) * 32 + lane;
  const bool valid = b_raw < batch;
  const int64_t b = valid ? b_raw : batch - 1;
  const size_t L_ = static_cast<size_t>(ld);
  const double *Wst = store + Z::oW(T) * ld + b;
  const double *Kst = store + Z::oK(T) * ld + b;
  const double *Gst = store + Z::oG(T) * ld + b;
  double *vst = scratch + Z::ov(T) * ld + b;
  double *kst = scratch + Z::ok(T) * ld + b;

  auto fetch = [&](int k, int buf) {
    double *dst = sm_affine + static_cast<size_t>(buf) * R::kRows * 32 + lane;
    const size_t kk = static_cast<size_t>(k);
#pragma unroll
    for (int t = 0; t < tri(N); ++t) cp_async8(dst + (R::rW + t) * 32, Wst + ((kk + 1) * tri(N) + t) * L_);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      cp_async8(dst + (R::rD + i) * 32, in.delta + ((kk + 1) * N + i) * L_ + b);
      cp_async8(dst + (R::rC + i) * 32, in.c + ((kk + 1) * N + i) * L_ + b);
      cp_async8(dst + (R::rQ + i) * 32, in.q + (kk * N + i) * L_ + b);
    }
#pragma unroll
    for (int t = 0; t < N * M; ++t) {
      cp_async8(dst + (R::rB + t) * 32, in.B + (kk * N * M + t) * L_ + b);
      cp_async8(dst + (R::rK + t) * 32, Kst + (kk * N * M + t) * L_);
    }
#pragma unroll
    for (int t = 0; t < tri(M); ++t) cp_async8(dst + (R::rG + t) * 32, Gst + (kk * tri(M) + t) * L_);
#pragma unroll
    for (int a = 0; a < M; ++a) cp_async8(dst + (R::rR + a) * 32, in.r + (kk * M + a) * L_ + b);
#pragma unroll
    for (int t = 0; t < N * N; ++t) cp_async8(dst + (R::rA + t) * 32, in.A + (kk * N * N + t) * L_ + b);
  };

  // stages T-1 .. T-NBUF+1 in flight before the loop; one commit per slot keeps the group
  // count uniform when the horizon is shorter than the pipeline
#pragma unroll
  for (int j = 0; j < NBUF - 1; ++j) {
    if (T - 1 - j >= 0) fetch(T - 1 - j, j);
    cp_async_commit();
  }
  double v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    v[i] = ldcs(in.q + (static_cast<size_t>(T) * N + i) * L_ + b);
    if (valid) stcs(vst + static_cast<int64_t>(T * N + i) * ld, v[i]);
  }
  int buf = 0;  // buffer of stage k = (T - 1 - k) % NBUF
  for (int k = T - 1; k >= 0; --k) {
    {
      const int kf = k - (NBUF - 1);  // goes into the buffer stage k + 1 has just left
      const int bf = buf == 0 ? NBUF - 1 : buf - 1;
      if (kf >= 0) fetch(kf, bf);
      cp_async_commit();
    }
    cp_async_wait_group<NBUF - 1>();
    const double *S = sm_affine + static_cast<size_t>(buf) * R::kRows * 32 + lane;
#define SR(row) S[(row) * 32]
    double f[N], g[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      dd[i] = SR(R::rD + i);
      f[i] = dd[i] * v[i] - SR(R::rC + i);
    }
    {
      double fz[N];
      apply_node<N>(f, dd, [&](int t) { return SR(R::rW + t); }, fz);  // f <- W f
    }
#pragma unroll
    for (int i = 0; i < N; ++i) g[i] = v[i] - f[i];
    double h[M];
#pragma unroll
    for (int a = 0; a < M; ++a) {
      double acc = SR(R::rR + a);
#pragma unroll
      for (int p = 0; p < N; ++p) acc += SR(R::rB + a * N + p) * g[p];
      h[a] = acc;
    }
    double kk[M];
#pragma unroll
    for (int a = 0; a < M; ++a) kk[a] = 0.0;
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
      for (int i = j; i < M; ++i) {
        const double gi = SR(R::rG + pk(i, j, M));
        kk[i] -= gi * h[j];
        if (i != j) kk[j] -= gi * h[i];
      }
#pragma unroll
    for (int a = 0; a < M; ++a)
      if (valid) stcs(kst + static_cast<int64_t>(k * M + a) * ld, kk[a]);
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double acc = SR(R::rQ + j);
#pragma unroll
      for (int p = 0; p < N; ++p) acc += SR(R::rA + j * N + p) * g[p];
#pragma unroll
      for (int a = 0; a < M; ++a) acc += SR(R::rK + j * M + a) * h[a];
      v[j] = acc;
    }
#undef SR
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (valid) stcs(vst + static_cast<int64_t>(k * N + i) * ld, v[i]);
    buf = buf + 1 == NBUF ? 0 : buf + 1;
  }
}

// ===========================================================================
// Backward affine sweep against a kept factorization (lqr.cpp:738-796).
// ===========================================================================
template <int N, int M>
__global__ void __launch_bounds__(128)
affine_backward(LqrIn in, const double *store, double *scratch, int64_t batch, int64_t ld,
                int T) {
  using Z = FastSizes<N, M>;
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const size_t L_ = static_cast<size_t>(ld);
#define G(ptr, e) ldcs((ptr) + static_cast<size_t>(e) * L_ + b)
  const double *Wst = store + Z::oW(T) * ld;
  const double *Kst = store + Z::oK(T) * ld;
  const double *Gst = store + Z::oG(T) * ld;
  double *vst = scratch + Z::ov(T) * ld + b;
  double *kst = scratch + Z::ok(T) * ld + b;

  double v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    v[i] = G(in.q, T * N + i);
    stcs(vst + static_cast<int64_t>(T * N + i) * ld, v[i]);
  }
  for (int k = T - 1; k >= 0; --k) {
    // Operands are pulled into register arrays in three groups BEFORE the arithmetic
    // that needs them, so each thread keeps ~100 independent loads in flight: at the
    // small batches this kernel serves (one Newton-KKT solve after a kept factor) the
    // latency of the dependent chain is hidden by memory-level parallelism, not by
    // occupancy.
    double wv[tri(N)], dv[N], cv[N];
#pragma unroll
    for (int t = 0; t < tri(N); ++t) wv[t] = G(Wst, (k + 1) * tri(N) + t);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      dv[i] = G(in.delta, (k + 1) * N + i);
      cv[i] = G(in.c, (k + 1) * N + i);
    }
    double f[N], g[N];
#pragma unroll
    for (int i = 0; i < N; ++i) f[i] = dv[i] * v[i] - cv[i];
    {
      double fz[N];
      apply_node<N>(f, dv, [&](int t) { return wv[t]; }, fz);  // f <- W f
    }
#pragma unroll
    for (int i = 0; i < N; ++i) g[i] = v[i] - f[i];
    double bv[N * M], kv[N * M], gv[tri(M)], rv[M];
#pragma unroll
    for (int t = 0; t < N * M; ++t) {
      bv[t] = G(in.B, k * N * M + t);
      kv[t] = G(Kst, k * N * M + t);
    }
#pragma unroll
    for (int t = 0; t < tri(M); ++t) gv[t] = G(Gst, k * tri(M) + t);
#pragma unroll
    for (int a = 0; a < M; ++a) rv[a] = G(in.r, k * M + a);
    double h[M];
#pragma unroll
    for (int a = 0; a < M; ++a) {
      double acc = rv[a];
#pragma unroll
      for (int p = 0; p < N; ++p) acc += bv[a * N + p] * g[p];
      h[a] = acc;
    }
    double kk[M];
#pragma unroll
    for (int a = 0; a < M; ++a) kk[a] = 0.0;
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
      for (int i = j; i < M; ++i) {
        const double gi = gv[pk(i, j, M)];
        kk[i] -= gi * h[j];
        if (i != j) kk[j] -= gi * h[i];
      }
#pragma unroll
    for (int a = 0; a < M; ++a) stcs(kst + static_cast<int64_t>(k * M + a) * ld, kk[a]);
    constexpr int HALF = (N + 1) / 2;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      double av[HALF * N], qv[HALF];
#pragma unroll
      for (int jj = 0; jj < HALF; ++jj) {
        const int j = half * HALF + jj;
        if (j < N) {
          qv[jj] = G(in.q, k * N + j);
#pragma unroll
          for (int p = 0; p < N; ++p) av[jj * N + p] = G(in.A, (k * N + j) * N + p);
        }
      }
#pragma unroll
      for (int jj = 0; jj < HALF; ++jj) {
        const int j = half * HALF + jj;
        if (j < N) {
          double acc = qv[jj];
#pragma unroll
          for (int p = 0; p < N; ++p) acc += av[jj * N + p] * g[p];
#pragma unroll
          for (int a = 0; a < M; ++a) acc += kv[j * M + a] * h[a];
          v[j] = acc;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) stcs(vst + static_cast<int64_t>(k * N + i) * ld, v[i]);
  }
#undef G
}

// ===========================================================================
// Root solve + forward rollout + costates (lqr.cpp:798-870), small batches: the same
// arithmetic as rollout_forward below with the operands of a stage copied to shared
// memory by cp.async kBuf - 1 stages ahead ([row][lane], one warp per block, a thread
// reads only what it copied).  At a few thousand problems -- or 64 with a horizon of
// 4 096 -- occupancy cannot hide the HBM latency of a stage's loads; the pipeline does.
// ===========================================================================
template <int N, int M>
struct ForwardRows {
  static constexpr int rA = 0, rB = rA + N * N, rK = rB + N * M, rW = rK + N * M, rv = rW + tri(N),
                       rd = rv + N, rc = rd + N, rk = rc + N, kRows = rk + M;
  static constexpr int kFit = (184 * 1024) / (kRows * 32 * 8);
  static constexpr int kBuf = kFit >= 4 ? 4 : (kFit >= 3 ? 3 : 2);
  static constexpr int kBytes = kBuf * kRows * 32 * int(sizeof(double));
  static_assert(kFit >= 2, "two stages of operands must fit shared memory");
};

template <int N, int M>
__global__ void __launch_bounds__(32)
rollout_forward_staged(LqrIn in, LqrOut out, const double *store, const double *scratch,
                       int64_t batch, int64_t ld, int T) {
  using Z = FastSizes<N, M>;
  using R = ForwardRows<N, M>;
  constexpr int NBUF = R::kBuf;
  extern __shared__ __align__(16) double sm_forward[];
  const int lane = threadIdx.x;
  const int64_t b_raw = static_cast<int64_t>(blockIdx.x) * 32 + lane;
  const bool valid = b_raw < batch;
  const int64_t b = valid ? b_raw : batch - 1;
  const size_t L_ = static_cast<size_t>(ld);
  const double *Wst = store + Z::oW(T) * ld + b;
  const double *Kst = store + Z::oK(T) * ld + b;
  const double *vst = scratch + Z::ov(T) * ld + b;
  const double *kst = scratch + Z::ok(T) * ld + b;
  double *xo = out.x + b, *uo = out.u + b, *yo = out.y + b;

  auto fetch = [&](int k, int buf) {  // operands of edge k / node k + 1
    double *dst = sm_forward + static_cast<size_t>(buf) * R::kRows * 32 + lane;
    const size_t kk = static_cast<size_t>(k);
#pragma unroll
    for (int t = 0; t < N * N; ++t) cp_async8(dst + (R::rA + t) * 32, in.A + (kk * N * N + t) * L_ + b);
#pragma unroll
    for (int t = 0; t < N * M; ++t) {
      cp_async8(dst + (R::rB + t) * 32, in.B + (kk * N * M + t) * L_ + b);
      cp_async8(dst + (R::rK + t) * 32, Kst + (kk * N * M + t) * L_);
    }
#pragma unroll
    for (int t = 0; t < tri(N); ++t) cp_async8(dst + (R::rW + t) * 32, Wst + ((kk + 1) * tri(N) + t) * L_);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      cp_async8(dst + (R::rv + i) * 32, vst + ((kk + 1) * N + i) * L_);
      cp_async8(dst + (R::rd + i) * 32, in.delta + ((kk + 1) * N + i) * L_ + b);
      cp_async8(dst + (R::rc + i) * 32, in.c + ((kk + 1) * N + i) * L_ + b);
    }
#pragma unroll
    for (int a = 0; a < M; ++a) cp_async8(dst + (R::rk + a) * 32, kst + (kk * M + a) * L_);
  };
#pragma unroll
  for (int j = 0; j < NBUF - 1; ++j) {
    if (j < T) fetch(j, j);
    cp_async_commit();
  }

  double x[N];
  {  // root: x_0 = -(I - D W)(delta o v - c), y_0 = v - W (delta o v - c)
    double f[N], fz[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = ldcs(vst + static_cast<size_t>(i) * L_);
      dd[i] = ldcs(in.delta + static_cast<size_t>(i) * L_ + b);
      f[i] = dd[i] * vv[i] - ldcs(in.c + static_cast<size_t>(i) * L_ + b);
    }
    apply_node<N>(f, dd, [&](int t) { return ldcs(Wst + static_cast<size_t>(t) * L_); }, fz);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      x[i] = -fz[i];
      if (valid) {
        stcs(xo + static_cast<size_t>(i) * L_, x[i]);
        stcs(yo + static_cast<size_t>(i) * L_, vv[i] - f[i]);
      }
    }
  }
  int buf = 0;
  for (int k = 0; k < T; ++k) {
    {
      const int kf = k + (NBUF - 1);  // goes into the buffer stage k - 1 has just left
      if (kf < T) fetch(kf, buf == 0 ? NBUF - 1 : buf - 1);
      cp_async_commit();
    }
    cp_async_wait_group<NBUF - 1>();
    const double *S = sm_forward + static_cast<size_t>(buf) * R::kRows * 32 + lane;
#define SR(row) S[(row) * 32]
    double u[M];
#pragma unroll
    for (int a = 0; a < M; ++a) u[a] = SR(R::rk + a);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int a = 0; a < M; ++a) u[a] += SR(R::rK + j * M + a) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a)
      if (valid) stcs(uo + static_cast<size_t>(k * M + a) * L_, u[a]);
    double f[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = SR(R::rv + i);
      dd[i] = SR(R::rd + i);
      f[i] = SR(R::rc + i) - dd[i] * vv[i];
    }
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] += SR(R::rA + j * N + i) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a)
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] += SR(R::rB + a * N + i) * u[a];
    apply_node<N>(f, dd, [&](int t) { return SR(R::rW + t); }, x);  // x' = (I + D V)^-1 f, f <- W f
#undef SR
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (valid) {
        stcs(xo + static_cast<size_t>((k + 1) * N + i) * L_, x[i]);
        stcs(yo + static_cast<size_t>((k + 1) * N + i) * L_, vv[i] + f[i]);
      }
    }
    buf = buf + 1 == NBUF ? 0 : buf + 1;
  }
}

// ===========================================================================
// Root solve + forward rollout + costates (lqr.cpp:798-870).
// ===========================================================================
template <int N, int M, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
rollout_forward(LqrIn in, LqrOut out, const double *store, const double *scratch,
                int64_t batch, int64_t ld, int T) {
  using Z = FastSizes<N, M>;
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const size_t L_ = static_cast<size_t>(ld);
#define G(ptr, e) ldcs((ptr) + static_cast<size_t>(e) * L_ + b)
  const double *Wst = store + Z::oW(T) * ld;
  const double *Kst = store + Z::oK(T) * ld;
  const double *vst = scratch + Z::ov(T) * ld;
  const double *kst = scratch + Z::ok(T) * ld;
  double *xo = out.x + b, *uo = out.u + b, *yo = out.y + b;

  double x[N];
  {  // root: x_0 = -(I - D W)(delta o v - c), y_0 = v - W (delta o v - c)
    double f[N], fz[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = G(vst, i);
      dd[i] = G(in.delta, i);
      f[i] = dd[i] * vv[i] - G(in.c, i);
    }
    apply_node<N>(f, dd, [&](int t) { return G(Wst, t); }, fz);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      x[i] = -fz[i];
      stcs(xo + static_cast<size_t>(i) * L_, x[i]);
      stcs(yo + static_cast<size_t>(i) * L_, vv[i] - f[i]);
    }
  }
  // Small shapes (the whole stage fits the register file twice): operands of stage
  // k + 1 are fetched while stage k is computed — none of them depends on x, so the
  // only exposed latency is the first stage's.  Large shapes rely on the compiler
  // hoisting a stage's loads (HBM-bound at 254 registers already).
  constexpr bool PREFETCH = (N * N + 2 * N * M + tri(N) + 3 * N + M) <= 64;
  constexpr int PA = PREFETCH ? N * N : 1, PB = PREFETCH ? N * M : 1, PW = PREFETCH ? tri(N) : 1,
                PN = PREFETCH ? N : 1, PM = PREFETCH ? M : 1;
  double nA[PA], nB[PB], nK[PB], nW[PW], nv[PN], nd[PN], nc[PN], nk[PM];
  auto fetch = [&](int k) {
    if constexpr (PREFETCH) {
#pragma unroll
      for (int t = 0; t < N * N; ++t) nA[t] = G(in.A, k * N * N + t);
#pragma unroll
      for (int t = 0; t < N * M; ++t) {
        nB[t] = G(in.B, k * N * M + t);
        nK[t] = G(Kst, k * N * M + t);
      }
#pragma unroll
      for (int t = 0; t < tri(N); ++t) nW[t] = G(Wst, (k + 1) * tri(N) + t);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        nv[i] = G(vst, (k + 1) * N + i);
        nd[i] = G(in.delta, (k + 1) * N + i);
        nc[i] = G(in.c, (k + 1) * N + i);
      }
#pragma unroll
      for (int a = 0; a < M; ++a) nk[a] = G(kst, k * M + a);
    }
  };
  if (T > 0) fetch(0);
  for (int k = 0; k < T; ++k) {
    double cA[PA], cB[PB], cK[PB], cW[PW], cv[PN], cd[PN], cc[PN], ck[PM];
    if constexpr (PREFETCH) {
#pragma unroll
      for (int t = 0; t < N * N; ++t) cA[t] = nA[t];
#pragma unroll
      for (int t = 0; t < N * M; ++t) {
        cB[t] = nB[t];
        cK[t] = nK[t];
      }
#pragma unroll
      for (int t = 0; t < tri(N); ++t) cW[t] = nW[t];
#pragma unroll
      for (int i = 0; i < N; ++i) {
        cv[i] = nv[i];
        cd[i] = nd[i];
        cc[i] = nc[i];
      }
#pragma unroll
      for (int a = 0; a < M; ++a) ck[a] = nk[a];
      if (k + 1 < T) fetch(k + 1);
    }
    double u[M];
#pragma unroll
    for (int a = 0; a < M; ++a) u[a] = PREFETCH ? ck[a] : G(kst, k * M + a);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int a = 0; a < M; ++a)
        u[a] += (PREFETCH ? cK[j * M + a] : G(Kst, (k * N + j) * M + a)) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a) stcs(uo + static_cast<size_t>(k * M + a) * L_, u[a]);
    double f[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = PREFETCH ? cv[i] : G(vst, (k + 1) * N + i);
      dd[i] = PREFETCH ? cd[i] : G(in.delta, (k + 1) * N + i);
      f[i] = (PREFETCH ? cc[i] : G(in.c, (k + 1) * N + i)) - dd[i] * vv[i];
    }
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i)
        f[i] += (PREFETCH ? cA[j * N + i] : G(in.A, (k * N + j) * N + i)) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a)
#pragma unroll
      for (int i = 0; i < N; ++i)
        f[i] += (PREFETCH ? cB[a * N + i] : G(in.B, (k * M + a) * N + i)) * u[a];
    // x' = (I + D V)^-1 f, f <- W f
    apply_node<N>(
        f, dd,
        [&](int t) {
          if constexpr (PREFETCH) return cW[t];
          else return G(Wst, (k + 1) * tri(N) + t);
        },
        x);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      stcs(xo + static_cast<size_t>((k + 1) * N + i) * L_, x[i]);
      stcs(yo + static_cast<size_t>((k + 1) * N + i) * L_, vv[i] + f[i]);
    }
  }
#undef G
}

// ===========================================================================
// Newton-KKT solve against a kept factorization, uniform chains (helpers.cpp:749-894):
// the rhs build is fused into the backward affine sweep and the dual recovery into the
// forward rollout, which writes the flat [x | y | z] solution directly.
// One thread per problem; constraint dimensions are runtime (per node / per edge).
// ===========================================================================
struct KktView {
  DevTables t;
  KktModel mdl;
  KktWs ws;
  const double *b;
  double *sol;
};

template <int N, int M>
__global__ void __launch_bounds__(128)
affine_backward_kkt(KktView kv, const double *store, double *scratch, int64_t batch, int64_t ld,
                    int T) {
  using Z = FastSizes<N, M>;
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const size_t L_ = static_cast<size_t>(ld);
  const DevTables &t = kv.t;
#define G(ptr, e) __ldg((ptr) + static_cast<size_t>(e) * L_ + b)
  const double *Wst = store + Z::oW(T) * ld;
  const double *Kst = store + Z::oK(T) * ld;
  const double *Gst = store + Z::oG(T) * ld;
  double *vst = scratch + Z::ov(T) * ld + b;
  double *kst = scratch + Z::ok(T) * ld + b;
  const int xd = t.x_dim, yd = t.y_dim;

  // q_mod of node k (node part): -b_x - Jc' Lc b_yc - Jg' Lg b_z      (helpers.cpp:752-778)
  auto node_q = [&](int k, double (&qv)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) qv[i] = -G(kv.b, t.x_state[k] + i);
    const int c = t.node_c[k], g = t.node_g[k];
    for (int r = 0; r < c; ++r) {
      const double wr = G(kv.ws.node_c_r2_inv, t.node_c_off[k] + r) * G(kv.b, xd + t.y_node_c[k] + r);
#pragma unroll
      for (int i = 0; i < N; ++i) qv[i] -= G(kv.mdl.node_jc, t.jc_node_off[k] + r + i * c) * wr;
    }
    for (int r = 0; r < g; ++r) {
      const double wr =
          G(kv.ws.node_mod_w_inv, t.node_g_off[k] + r) * G(kv.b, xd + yd + t.z_node[k] + r);
#pragma unroll
      for (int i = 0; i < N; ++i) qv[i] -= G(kv.mdl.node_jg, t.jg_node_off[k] + r + i * g) * wr;
    }
  };
  // edge part of q_mod[parent] and r_mod of edge e                      (helpers.cpp:780-812)
  auto edge_qr = [&](int e, double (&qv)[N], double (&rv)[M]) {
#pragma unroll
    for (int a = 0; a < M; ++a) rv[a] = -G(kv.b, t.x_control[e] + a);
    const int c = t.edge_c[e], g = t.edge_g[e];
    for (int r = 0; r < c; ++r) {
      const double wr = G(kv.ws.edge_c_r2_inv, t.edge_c_off[e] + r) * G(kv.b, xd + t.y_edge_c[e] + r);
#pragma unroll
      for (int i = 0; i < N; ++i) qv[i] -= G(kv.mdl.edge_jcx, t.jcx_off[e] + r + i * c) * wr;
#pragma unroll
      for (int a = 0; a < M; ++a) rv[a] -= G(kv.mdl.edge_jcu, t.jcu_off[e] + r + a * c) * wr;
    }
    for (int r = 0; r < g; ++r) {
      const double wr =
          G(kv.ws.edge_mod_w_inv, t.edge_g_off[e] + r) * G(kv.b, xd + yd + t.z_edge[e] + r);
#pragma unroll
      for (int i = 0; i < N; ++i) qv[i] -= G(kv.mdl.edge_jgx, t.jgx_off[e] + r + i * g) * wr;
#pragma unroll
      for (int a = 0; a < M; ++a) rv[a] -= G(kv.mdl.edge_jgu, t.jgu_off[e] + r + a * g) * wr;
    }
  };

  double v[N];
  node_q(T, v);
#pragma unroll
  for (int i = 0; i < N; ++i) stcs(vst + static_cast<int64_t>(T * N + i) * ld, v[i]);
  for (int k = T - 1; k >= 0; --k) {
    double wv[tri(N)], f[N], g[N], dd[N];
#pragma unroll
    for (int u = 0; u < tri(N); ++u) wv[u] = G(Wst, (k + 1) * tri(N) + u);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      // c_mod = -b_ydyn (helpers.cpp:777), delta = dyn_r2
      dd[i] = G(kv.ws.dyn_r2, (k + 1) * N + i);
      f[i] = dd[i] * v[i] + G(kv.b, xd + t.y_dyn[k + 1] + i);
    }
    {
      double fz[N];
      apply_node<N>(f, dd, [&](int u) { return wv[u]; }, fz);  // f <- W f
    }
#pragma unroll
    for (int i = 0; i < N; ++i) g[i] = v[i] - f[i];
    double qv[N], rv[M];
    node_q(k, qv);
    edge_qr(k, qv, rv);
    double bv[N * M], kvv[N * M], gv[tri(M)];
#pragma unroll
    for (int u = 0; u < N * M; ++u) {
      bv[u] = G(kv.mdl.edge_B, k * N * M + u);
      kvv[u] = G(Kst, k * N * M + u);
    }
#pragma unroll
    for (int u = 0; u < tri(M); ++u) gv[u] = G(Gst, k * tri(M) + u);
    double h[M], kk[M];
#pragma unroll
    for (int a = 0; a < M; ++a) {
      double acc = rv[a];
#pragma unroll
      for (int p = 0; p < N; ++p) acc += bv[a * N + p] * g[p];
      h[a] = acc;
      kk[a] = 0.0;
    }
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
      for (int i = j; i < M; ++i) {
        const double gi = gv[pk(i, j, M)];
        kk[i] -= gi * h[j];
        if (i != j) kk[j] -= gi * h[i];
      }
#pragma unroll
    for (int a = 0; a < M; ++a) stcs(kst + static_cast<int64_t>(k * M + a) * ld, kk[a]);
#pragma unroll
    for (int j = 0; j < N; ++j) {
      double acc = qv[j];
#pragma unroll
      for (int p = 0; p < N; ++p) acc += G(kv.mdl.edge_A, (k * N + j) * N + p) * g[p];
#pragma unroll
      for (int a = 0; a < M; ++a) acc += kvv[j * M + a] * h[a];
      v[j] = acc;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) stcs(vst + static_cast<int64_t>(k * N + i) * ld, v[i]);
  }
#undef G
}

template <int N, int M>
__global__ void __launch_bounds__(128)
rollout_forward_kkt(KktView kv, const double *store, const double *scratch, int64_t batch,
                    int64_t ld, int T) {
  using Z = FastSizes<N, M>;
  const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const size_t L_ = static_cast<size_t>(ld);
  const DevTables &t = kv.t;
#define G(ptr, e) __ldg((ptr) + static_cast<size_t>(e) * L_ + b)
#define SOL(e) kv.sol[static_cast<size_t>(e) * L_ + b]
  const double *Wst = store + Z::oW(T) * ld;
  const double *Kst = store + Z::oK(T) * ld;
  const double *vst = scratch + Z::ov(T) * ld;
  const double *kst = scratch + Z::ok(T) * ld;
  const int xd = t.x_dim, yd = t.y_dim;

  // y_c = Lc (Jc x - b_yc), z = Lg (Jg x - b_z) of node k                (helpers.cpp:828-856)
  auto recover_node = [&](int k, const double (&x)[N]) {
    const int c = t.node_c[k], g = t.node_g[k];
    for (int r = 0; r < c; ++r) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) s += G(kv.mdl.node_jc, t.jc_node_off[k] + r + j * c) * x[j];
      s -= G(kv.b, xd + t.y_node_c[k] + r);
      SOL(xd + t.y_node_c[k] + r) = G(kv.ws.node_c_r2_inv, t.node_c_off[k] + r) * s;
    }
    for (int r = 0; r < g; ++r) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) s += G(kv.mdl.node_jg, t.jg_node_off[k] + r + j * g) * x[j];
      s -= G(kv.b, xd + yd + t.z_node[k] + r);
      SOL(xd + yd + t.z_node[k] + r) = G(kv.ws.node_mod_w_inv, t.node_g_off[k] + r) * s;
    }
  };
  // the same for the constraints of edge e (parent state x, control u)    (helpers.cpp:858-893)
  auto recover_edge = [&](int e, const double (&x)[N], const double (&u)[M]) {
    const int c = t.edge_c[e], g = t.edge_g[e];
    for (int r = 0; r < c; ++r) {
      double s = 0.0, s2 = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) s += G(kv.mdl.edge_jcx, t.jcx_off[e] + r + j * c) * x[j];
#pragma unroll
      for (int a = 0; a < M; ++a) s2 += G(kv.mdl.edge_jcu, t.jcu_off[e] + r + a * c) * u[a];
      s += s2;
      s -= G(kv.b, xd + t.y_edge_c[e] + r);
      SOL(xd + t.y_edge_c[e] + r) = G(kv.ws.edge_c_r2_inv, t.edge_c_off[e] + r) * s;
    }
    for (int r = 0; r < g; ++r) {
      double s = 0.0, s2 = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) s += G(kv.mdl.edge_jgx, t.jgx_off[e] + r + j * g) * x[j];
#pragma unroll
      for (int a = 0; a < M; ++a) s2 += G(kv.mdl.edge_jgu, t.jgu_off[e] + r + a * g) * u[a];
      s += s2;
      s -= G(kv.b, xd + yd + t.z_edge[e] + r);
      SOL(xd + yd + t.z_edge[e] + r) = G(kv.ws.edge_mod_w_inv, t.edge_g_off[e] + r) * s;
    }
  };

  double x[N];
  {  // root
    double f[N], fz[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = G(vst, i);
      dd[i] = G(kv.ws.dyn_r2, i);
      f[i] = dd[i] * vv[i] + G(kv.b, xd + t.y_dyn[0] + i);  // delta o v - c, c = -b_ydyn
    }
    apply_node<N>(f, dd, [&](int u) { return G(Wst, u); }, fz);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      x[i] = -fz[i];
      SOL(t.x_state[0] + i) = x[i];
      SOL(xd + t.y_dyn[0] + i) = vv[i] - f[i];
    }
  }
  for (int k = 0; k < T; ++k) {
    double u[M];
#pragma unroll
    for (int a = 0; a < M; ++a) u[a] = G(kst, k * M + a);
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int a = 0; a < M; ++a) u[a] += G(Kst, (k * N + j) * M + a) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a) SOL(t.x_control[k] + a) = u[a];
    recover_node(k, x);
    recover_edge(k, x, u);
    double f[N], vv[N], dd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      vv[i] = G(vst, (k + 1) * N + i);
      dd[i] = G(kv.ws.dyn_r2, (k + 1) * N + i);
      f[i] = -G(kv.b, xd + t.y_dyn[k + 1] + i) - dd[i] * vv[i];  // c' - delta' o v'
    }
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] += G(kv.mdl.edge_A, (k * N + j) * N + i) * x[j];
#pragma unroll
    for (int a = 0; a < M; ++a)
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] += G(kv.mdl.edge_B, (k * M + a) * N + i) * u[a];
    // x' = (I + D V)^-1 f, f <- W f
    apply_node<N>(f, dd, [&](int u) { return G(Wst, (k + 1) * tri(N) + u); }, x);
#pragma unroll
    for (int i = 0; i < N; ++i) {
      SOL(t.x_state[k + 1] + i) = x[i];
      SOL(xd + t.y_dyn[k + 1] + i) = vv[i] + f[i];
    }
  }
  recover_node(T, x);
#undef SOL
#undef G
}

// ===========================================================================
// Plans
// ===========================================================================
// Below this many problems a thread-per-problem kernel launches one-warp blocks.
constexpr int64_t kSmallBatch = 148 * 128 * 2;
// Up to this many problems factor + solve runs as the fused sweep + rollout kernel.
#ifndef SIPOC_FUSED_MAX_BATCH
#define SIPOC_FUSED_MAX_BATCH 40960
#endif
constexpr int64_t kFusedMaxBatch = SIPOC_FUSED_MAX_BATCH;

template <int N, int M, bool SUBWARP>
struct Plan {
  static int64_t store_elems(int T) { return FastSizes<N, M>::store(T); }
  static int64_t scratch_elems(int T) { return FastSizes<N, M>::scratch(T); }

  template <bool SOLVE, int W, bool FUSED = false, bool PACKW = FUSED>
  static void launch_subwarp(const FastArgs &a, cudaStream_t s) {
    auto kern = riccati_backward_subwarp<N, M, SOLVE, W, FUSED, PACKW>;
    using Sm = Smem<N, M, PACKW>;
    constexpr int bytes = Sm::kBytes * W;
    if (bytes > 48 * 1024)
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    const unsigned grid = static_cast<unsigned>((a.batch + kTile * W - 1) / (kTile * W));
    ProfScope ps(a.prof, FUSED ? "riccati_fused_subwarp" : "riccati_backward_subwarp", s);
    kern<<<grid, 32 * W, bytes, s>>>(a.in, a.out, a.status, a.store, a.scratch, a.batch, a.ld,
                                     a.num_edges, SegmentArgs{});
  }

  template <bool SOLVE>
  static void backward(const FastArgs &a, cudaStream_t s) {
    if constexpr (SUBWARP) {
      // One warp (8 problems) per CTA: warps of different CTAs drift apart, so the
      // DFMA-heavy and the latency-bound phases of different tiles overlap on an SM
      // (measured: 1 warp / CTA 5.97 ms, 4 warps / CTA in lockstep 7.40 ms).
      // Up to ~3 waves of tiles: the packed map, seven warps per SM (8 192 problems are
      // one wave); deeper grids: the padded map at six.
      if (a.batch <= kFusedMaxBatch) launch_subwarp<SOLVE, 1, false, true>(a, s);
      else launch_subwarp<SOLVE, 1, false, false>(a, s);
    } else {
      const unsigned grid = static_cast<unsigned>((a.batch + 63) / 64);
      ProfScope ps(a.prof, "riccati_backward_thread", s);
      riccati_backward_thread<N, M, SOLVE>
          <<<grid, 64, 0, s>>>(a.in, a.status, a.store, a.scratch, a.batch, a.ld, a.num_edges);
    }
  }
  template <int THREADS, int MINB>
  static void launch_forward(const FastArgs &a, cudaStream_t s) {
    const unsigned grid = static_cast<unsigned>((a.batch + THREADS - 1) / THREADS);
    ProfScope ps(a.prof, "rollout_forward", s);
    rollout_forward<N, M, THREADS, MINB>
        <<<grid, THREADS, 0, s>>>(a.in, a.out, a.store, a.scratch, a.batch, a.ld, a.num_edges);
  }
  static void forward(const FastArgs &a, cudaStream_t s) {
    // No register cap: the compiler then hoists a whole stage's loads (254 registers),
    // which is what keeps HBM busy (capped variants were slower).  Small batches use
    // one-warp blocks so that every SM gets work (8 192 problems are 64 blocks of 128).
    if (a.batch >= kSmallBatch) {
      launch_forward<128, 1>(a, s);
    } else {
      auto kern = rollout_forward_staged<N, M>;
      constexpr int bytes = ForwardRows<N, M>::kBytes;
      if (bytes > 48 * 1024)
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      ProfScope ps(a.prof, "rollout_forward_staged", s);
      kern<<<static_cast<unsigned>((a.batch + 31) / 32), 32, bytes, s>>>(
          a.in, a.out, a.store, a.scratch, a.batch, a.ld, a.num_edges);
    }
  }
  static int factor(const FastArgs &a, cudaStream_t s) {
    backward<false>(a, s);
    return 1;
  }
  static int solve(const FastArgs &a, cudaStream_t s) {
    if (a.batch < kSmallBatch) {
      auto kern = affine_backward_staged<N, M>;
      constexpr int bytes = AffineRows<N, M>::kBytes;
      if (bytes > 48 * 1024)
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      ProfScope ps(a.prof, "affine_backward_staged", s);
      kern<<<static_cast<unsigned>((a.batch + 31) / 32), 32, bytes, s>>>(
          a.in, a.store, a.scratch, a.batch, a.ld, a.num_edges);
    } else {
      ProfScope ps(a.prof, "affine_backward", s);
      affine_backward<N, M><<<static_cast<unsigned>((a.batch + 127) / 128), 128, 0, s>>>(
          a.in, a.store, a.scratch, a.batch, a.ld, a.num_edges);
    }
    forward(a, s);
    return 2;
  }
  static int factor_solve(const FastArgs &a, cudaStream_t s) {
    if (SUBWARP && a.batch <= kFusedMaxBatch) {
      // One kernel: each warp rolls its tile forward right after its backward sweep.  Pays
      // up to about four waves of tiles (quadrotor: 3.10 against 3.56 ms at 32 768 problems,
      // 1.50 against 1.64 ms at 16 384, 0.74 against 1.10 ms at 8 192 -- the per-GPU shard of
      // the 65 536-problem batch on eight GPUs, one wave at seven warps per SM); at 65 536
      // the sweep + the streaming thread-per-problem rollout is faster (5.8 against 6.1 ms:
      // a tile's rollout costs its warp ~4 us per stage during which the slot does no sweep
      // work, and the sweep runs faster on the padded map at six warps per SM).
      if constexpr (SUBWARP) launch_subwarp<true, 1, true>(a, s);
      return 1;
    } else {
      backward<true>(a, s);
      forward(a, s);
      return 2;
    }
  }
  // Parallel in time: S segments of a.num_edges edges each, from the scan's boundary data.
  // a.status is [S][ld]; a.store / a.scratch hold S segment-sized regions.
  static int factor_solve_segments(const FastArgs &a, const double *Vb, const double *vb,
                                   const double *xb, int S, cudaStream_t s) {
    if constexpr (SUBWARP) {
      auto kern = riccati_backward_subwarp<N, M, true, 1, true, true, true>;
      using Sm = Smem<N, M, true>;
      constexpr int bytes = Sm::kBytes;
      if (bytes > 48 * 1024)
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      const dim3 grid(static_cast<unsigned>((a.batch + kTile - 1) / kTile), static_cast<unsigned>(S));
      ProfScope ps(a.prof, "riccati_fused_subwarp_segments", s);
      kern<<<grid, 32, bytes, s>>>(a.in, a.out, a.status, a.store, a.scratch, a.batch, a.ld,
                                   a.num_edges, SegmentArgs{Vb, vb, xb});
      return 1;
    } else {
      return -1;
    }
  }
  static int kkt_solve(const FastKktArgs &k, cudaStream_t s) {
    const unsigned grid = static_cast<unsigned>((k.batch + 127) / 128);
    const KktView view{*k.tables, *k.model, *k.ws, k.b, k.sol};
    {
      ProfScope ps(k.prof, "affine_backward_kkt", s);
      affine_backward_kkt<N, M>
          <<<grid, 128, 0, s>>>(view, k.store, k.scratch, k.batch, k.ld, k.num_edges);
    }
    {
      ProfScope ps(k.prof, "rollout_forward_kkt", s);
      rollout_forward_kkt<N, M>
          <<<grid, 128, 0, s>>>(view, k.store, k.scratch, k.batch, k.ld, k.num_edges);
    }
    return 2;
  }
};

template <int N, int M, bool SUBWARP>
const FastPlan *make_plan(const char *name) {
  using P = Plan<N, M, SUBWARP>;
  static const FastPlan plan{name,         N,           M,         &P::store_elems,
                             &P::scratch_elems, &P::factor, &P::solve, &P::factor_solve,
                             &P::kkt_solve, false,
                             SUBWARP ? &P::factor_solve_segments : nullptr};
  return &plan;
}

}  // namespace

// The shapes are compiled in four parts (the same file with -DSIPOC_FAST_PART=0..3, see the
// Makefile) so that the translation units build in parallel.  Together they cover the
// reference benchmark grid for n <= 8 (lqr_benchmark.cpp:537-545: n in {4, 6, 8} x
// m in {1, 2, 3, 4}) plus the quadrotor shape; n = 16 runs on the CTA-per-problem plans
// (riccati_cta.cu), every other uniform shape is padded up to the next shape of either set.
#ifndef SIPOC_FAST_PART
#define SIPOC_FAST_PART 0
#endif
#define SIPOC_CAT2(a, b) a##b
#define SIPOC_CAT(a, b) SIPOC_CAT2(a, b)
const FastPlan *select_fast_plan_part1(int n, int m);
const FastPlan *select_fast_plan_part2(int n, int m);
const FastPlan *select_fast_plan_part3(int n, int m);

#if SIPOC_FAST_PART == 0
const FastPlan *select_fast_plan(int n, int m) {
  if (n == 12 && m == 4) return make_plan<12, 4, true>("subwarp4_n12_m4");
  if (n == 4 && m == 1) return make_plan<4, 1, false>("thread_per_problem_n4_m1");
  if (n == 4 && m == 2) return make_plan<4, 2, false>("thread_per_problem_n4_m2");
  if (n == 4 && m == 3) return make_plan<4, 3, false>("thread_per_problem_n4_m3");
  if (n == 4 && m == 4) return make_plan<4, 4, false>("thread_per_problem_n4_m4");
  if (const FastPlan *p = select_fast_plan_part1(n, m)) return p;
  if (const FastPlan *p = select_fast_plan_part2(n, m)) return p;
  return select_fast_plan_part3(n, m);
}
#elif SIPOC_FAST_PART == 1
const FastPlan *select_fast_plan_part1(int n, int m) {
  if (n == 6 && m == 1) return make_plan<6, 1, true>("subwarp4_n6_m1");
  if (n == 6 && m == 2) return make_plan<6, 2, true>("subwarp4_n6_m2");
  if (n == 6 && m == 3) return make_plan<6, 3, true>("subwarp4_n6_m3");
  return nullptr;
}
#elif SIPOC_FAST_PART == 2
const FastPlan *select_fast_plan_part2(int n, int m) {
  if (n == 6 && m == 4) return make_plan<6, 4, true>("subwarp4_n6_m4");
  if (n == 8 && m == 1) return make_plan<8, 1, true>("subwarp4_n8_m1");
  if (n == 8 && m == 2) return make_plan<8, 2, true>("subwarp4_n8_m2");
  return nullptr;
}
#else
const FastPlan *select_fast_plan_part3(int n, int m) {
  if (n == 8 && m == 3) return make_plan<8, 3, true>("subwarp4_n8_m3");
  if (n == 8 && m == 4) return make_plan<8, 4, true>("subwarp4_n8_m4");
  return nullptr;
}
#endif

}  // namespace sipoc
