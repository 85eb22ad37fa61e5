// gemm.cu — FP64 tensor-core GEMM for sm_100a.
//
// Blackwell's tcgen05 path has no FP64 kind; the FP64 tensor pipe is reached
// through mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4 — every larger PTX f64 shape is
// split into it by ptxas on sm_100a).  The kernel is therefore a multi-stage
// cp.async (LDGSTS) pipeline feeding register accumulators:
//   * CTA tile BM x BN x 16, STAGES-deep shared-memory ring, one barrier per
//     k-tile;
//   * both operands in either orientation (K-contiguous or M/N-contiguous), so
//     the index permutes of the contraction engine are absorbed by the loads;
//   * 64-bit fragments cannot use ldmatrix: tiles are padded by 4 doubles per
//     row, which makes every half-warp LDS.64 fragment read conflict-free;
//   * batched (free index or reduction index) and split-K launches write
//     partial products that reduce.cu sums deterministically;
//   * grouped tile rasterisation keeps an A row-panel group L2-resident.
// C = alpha * op(A) op(B) + beta * C, row-major C.
#include "kernels.h"

#include <cstdlib>

namespace ecw {

namespace {

constexpr int PAD = 4;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Load a tile whose contiguous direction is the K direction: smem[r][k], r < ROWS.
template <int ROWS, int THREADS, int BK>
__device__ __forceinline__ void load_kmajor(double* sm, const double* __restrict__ g, int64_t ld,
                                            int64_t row0, int64_t nrows, int64_t k0, int64_t kend,
                                            int vec, int tid) {
  constexpr int LDS = BK + PAD;
  if (vec) {
    constexpr int CH = ROWS * (BK / 2);
#pragma unroll
    for (int c = tid; c < CH; c += THREADS) {
      int r = c / (BK / 2), kc = (c % (BK / 2)) * 2;
      int64_t gr = row0 + r, gk = k0 + kc;
      int bytes = 0;
      if (gr < nrows && gk < kend) bytes = (gk + 1 < kend) ? 16 : 8;
      const double* src = bytes ? g + gr * ld + gk : g;
      cp_async16(sm + r * LDS + kc, src, bytes);
    }
  } else {
    constexpr int CH = ROWS * BK;
#pragma unroll
    for (int c = tid; c < CH; c += THREADS) {
      int r = c / BK, kc = c % BK;
      int64_t gr = row0 + r, gk = k0 + kc;
      int bytes = (gr < nrows && gk < kend) ? 8 : 0;
      const double* src = bytes ? g + gr * ld + gk : g;
      cp_async8(sm + r * LDS + kc, src, bytes);
    }
  }
}

// Load a tile whose contiguous direction is the M/N direction: smem[k][c], c < COLS.
template <int COLS, int THREADS, int BK>
__device__ __forceinline__ void load_mnmajor(double* sm, const double* __restrict__ g, int64_t ld,
                                             int64_t col0, int64_t ncols, int64_t k0, int64_t kend,
                                             int vec, int tid) {
  constexpr int LDS = COLS + PAD;
  if (vec) {
    constexpr int CPR = COLS / 2;
    constexpr int CH = BK * CPR;
#pragma unroll
    for (int c = tid; c < CH; c += THREADS) {
      int kr = c / CPR, cc = (c % CPR) * 2;
      int64_t gk = k0 + kr, gc = col0 + cc;
      int bytes = 0;
      if (gk < kend && gc < ncols) bytes = (gc + 1 < ncols) ? 16 : 8;
      const double* src = bytes ? g + gk * ld + gc : g;
      cp_async16(sm + kr * LDS + cc, src, bytes);
    }
  } else {
    constexpr int CH = BK * COLS;
#pragma unroll
    for (int c = tid; c < CH; c += THREADS) {
      int kr = c / COLS, cc = c % COLS;
      int64_t gk = k0 + kr, gc = col0 + cc;
      int bytes = (gk < kend && gc < ncols) ? 8 : 0;
      const double* src = bytes ? g + gk * ld + gc : g;
      cp_async8(sm + kr * LDS + cc, src, bytes);
    }
  }
}

template <int BM, int BN, int BK, int TA, int TB>
struct SmemLayout {
  static constexpr int A_ELEMS = TA ? BK * (BM + PAD) : BM * (BK + PAD);
  static constexpr int B_ELEMS = TB ? BN * (BK + PAD) : BK * (BN + PAD);
  static constexpr int STAGE = A_ELEMS + B_ELEMS;
};

template <int BM, int BN, int WM, int WN, int BK, int TA, int TB, int STAGES, int ILV>
__global__ void __launch_bounds__((BM / WM) * (BN / WN) * 32, (BK == 8) ? ((BM * BN <= 80 * 80) ? 3 : 2) : ((BM * BN <= 128 * 48) ? 2 : 1))
dgemm_kernel(GemmArgs p) {
  constexpr int THREADS = (BM / WM) * (BN / WN) * 32;
  constexpr int MI = WM / 8, NI = WN / 8;
  using L = SmemLayout<BM, BN, BK, TA, TB>;
  extern __shared__ __align__(16) double smem[];

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, tig = lane & 3;
  const int wm0 = (warp % (BM / WM)) * WM;
  const int wn0 = (warp / (BM / WM)) * WN;

  // ---- tile coordinates (grouped rasterisation: GROUP row-tiles share column sweeps)
  const int64_t tiles_m = (p.M + BM - 1) / BM, tiles_n = (p.N + BN - 1) / BN;
  int64_t tile = blockIdx.x;
  int64_t tm, tn;
  {
    const int64_t GROUP = 8;
    int64_t per_group = GROUP * tiles_n;
    int64_t gid = tile / per_group;
    int64_t first_m = gid * GROUP;
    int64_t gsz = min(tiles_m - first_m, GROUP);
    tm = first_m + (tile % per_group) % gsz;
    tn = (tile % per_group) / gsz;
  }
  const int64_t m0 = tm * BM, n0 = tn * BN;

  // ---- batch / split-K slice
  const int64_t zb = blockIdx.y;
  const int64_t r = zb / p.splitk, s = zb % p.splitk;
  const int64_t kbeg = s * p.kchunk;
  const int64_t kend = min(p.K, kbeg + p.kchunk);
  const double* __restrict__ A = p.A + r * p.sA;
  const double* __restrict__ B = p.B + r * p.sB;
  double* __restrict__ C = p.C + zb * p.sC;

  double acc[MI][NI][2];
#pragma unroll
  for (int i = 0; i < MI; ++i)
#pragma unroll
    for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int64_t ktiles = (kend - kbeg + BK - 1) / BK;
  static_assert(BK % 4 == 0, "BK");

  auto load_stage = [&](int stage, int64_t kt) {
    double* sa = smem + stage * L::STAGE;
    double* sb = sa + L::A_ELEMS;
    const int64_t k0 = kbeg + kt * BK;
    if (TA == 0) load_kmajor<BM, THREADS, BK>(sa, A, p.lda, m0, p.M, k0, kend, p.vecA, tid);
    else load_mnmajor<BM, THREADS, BK>(sa, A, p.lda, m0, p.M, k0, kend, p.vecA, tid);
    if (TB == 0) load_mnmajor<BN, THREADS, BK>(sb, B, p.ldb, n0, p.N, k0, kend, p.vecB, tid);
    else load_kmajor<BN, THREADS, BK>(sb, B, p.ldb, n0, p.N, k0, kend, p.vecB, tid);
  };

#pragma unroll
  for (int st = 0; st < STAGES - 1; ++st) {
    if (st < ktiles) load_stage(st, st);
    cp_async_commit();
  }

  for (int64_t kt = 0; kt < ktiles; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    if (!ILV) {
      int64_t nk = kt + STAGES - 1;
      if (nk < ktiles) load_stage((int)(nk % STAGES), nk);
      cp_async_commit();
    }
    const double* sa = smem + (kt % STAGES) * L::STAGE;
    const double* sb = sa + L::A_ELEMS;
#pragma unroll
    for (int k4 = 0; k4 < BK / 4; ++k4) {
      double af[MI], bf[NI];
      const int kk = k4 * 4 + tig;
#pragma unroll
      for (int i = 0; i < MI; ++i) {
        const int m = wm0 + i * 8 + g;
        af[i] = TA ? sa[kk * (BM + PAD) + m] : sa[m * (BK + PAD) + kk];
      }
#pragma unroll
      for (int j = 0; j < NI; ++j) {
        const int n = wn0 + j * 8 + g;
        bf[j] = TB ? sb[n * (BK + PAD) + kk] : sb[kk * (BN + PAD) + n];
      }
#pragma unroll
      for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
      if (ILV && k4 == 0) {
        // issue the next stage's copies in the shadow of the DMMAs just queued: the slot being
        // refilled was last read in iteration kt-1, i.e. before the barrier above
        int64_t nk = kt + STAGES - 1;
        if (nk < ktiles) load_stage((int)(nk % STAGES), nk);
        cp_async_commit();
      }
    }
  }
  cp_async_wait<0>();

  // ---- epilogue.  With beta != 0 the old values of a group of fragment rows are all fetched before the first store of
  // the group (RG * NI independent loads in flight per thread): a load-add-store chain per fragment would serialise on
  // the memory latency, which is the whole run time of the K = nocc rank updates (huge M*N, three k-tiles).
  const double alpha = p.alpha, beta = p.beta;
  const bool vecC = p.vecC;
  constexpr int RG = (MI >= 2 && THREADS < 512) ? 2 : 1;     // 512-thread tiles run under a 128-register cap
#pragma unroll
  for (int i0 = 0; i0 < MI; i0 += RG) {
    double2 old[RG][NI];
    if (beta != 0.0) {
#pragma unroll
      for (int ii = 0; ii < RG; ++ii) {
        const int64_t m = m0 + wm0 + (i0 + ii) * 8 + g;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          const int64_t n = n0 + wn0 + j * 8 + 2 * tig;
          old[ii][j] = make_double2(0.0, 0.0);
          if (i0 + ii < MI && m < p.M && n < p.N) {
            const double* c = C + m * p.ldc + n;
            if (vecC && n + 1 < p.N) {
              old[ii][j] = *reinterpret_cast<const double2*>(c);
            } else {
              old[ii][j].x = c[0];
              if (n + 1 < p.N) old[ii][j].y = c[1];
            }
          }
        }
      }
    }
#pragma unroll
    for (int ii = 0; ii < RG; ++ii) {
      if (i0 + ii >= MI) continue;
      const int i = i0 + ii;
      const int64_t m = m0 + wm0 + i * 8 + g;
      if (m >= p.M) continue;
#pragma unroll
      for (int j = 0; j < NI; ++j) {
        const int64_t n = n0 + wn0 + j * 8 + 2 * tig;
        if (n >= p.N) continue;
        double* c = C + m * p.ldc + n;
        double v0 = alpha * acc[i][j][0], v1 = alpha * acc[i][j][1];
        if (beta != 0.0) {
          v0 += beta * old[ii][j].x;
          v1 += beta * old[ii][j].y;
        }
        if (vecC && n + 1 < p.N) {
          *reinterpret_cast<double2*>(c) = make_double2(v0, v1);
        } else {
          c[0] = v0;
          if (n + 1 < p.N) c[1] = v1;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// N == 1: matrix-vector products (the ovvv / oovv_ph contractions with a singles-sized operand, CCSD.py:363, 377, 499
// and the rdm1 'vo' block).  Bound by the one pass over A: every thread keeps 8 independent 16-byte loads in flight.
// x[k] = B[k * xs]; partial sums of the batch / split-K slices are written like the GEMM kernel writes them
// (C + zb * sC), the plan's OP_REDUCE adds them in a fixed order.
// ta == 1: A[k * lda + m].  CTA = 4 k-lanes x 64 threads, thread = two adjacent m.
__global__ void __launch_bounds__(256) dgemv_mcontig_kernel(GemmArgs p, int64_t xs) {
  __shared__ double2 red[4][64];
  const int tx = threadIdx.x & 63, ky = threadIdx.x >> 6;
  const int64_t zb = blockIdx.y, r = zb / p.splitk, s = zb % p.splitk;
  const int64_t kbeg = s * p.kchunk, kend = min(p.K, kbeg + p.kchunk);
  const double* __restrict__ A = p.A + r * p.sA;
  const double* __restrict__ x = p.B + r * p.sB;
  const int64_t m = ((int64_t)blockIdx.x * 64 + tx) * 2;
  double2 acc = make_double2(0.0, 0.0);
  if (m < p.M) {
    const bool pair = m + 1 < p.M;
    if (p.vecA && pair) {
      int64_t k = kbeg + ky;
      for (; k + 28 < kend; k += 32) {
        double2 a[8];
        double xv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          a[u] = *reinterpret_cast<const double2*>(A + (k + 4 * u) * p.lda + m);
          xv[u] = x[(k + 4 * u) * xs];
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          acc.x = fma(a[u].x, xv[u], acc.x);
          acc.y = fma(a[u].y, xv[u], acc.y);
        }
      }
      for (; k < kend; k += 4) {
        const double2 a = *reinterpret_cast<const double2*>(A + k * p.lda + m);
        const double xv = x[k * xs];
        acc.x = fma(a.x, xv, acc.x);
        acc.y = fma(a.y, xv, acc.y);
      }
    } else {
      for (int64_t k = kbeg + ky; k < kend; k += 4) {
        const double xv = x[k * xs];
        acc.x = fma(A[k * p.lda + m], xv, acc.x);
        if (pair) acc.y = fma(A[k * p.lda + m + 1], xv, acc.y);
      }
    }
  }
  red[ky][tx] = acc;
  __syncthreads();
  if (ky == 0 && m < p.M) {
    double sx = red[0][tx].x, sy = red[0][tx].y;
#pragma unroll
    for (int q = 1; q < 4; ++q) {
      sx += red[q][tx].x;
      sy += red[q][tx].y;
    }
    double* c = p.C + zb * p.sC + m * p.ldc;
    c[0] = p.alpha * sx + (p.beta != 0.0 ? p.beta * c[0] : 0.0);
    if (m + 1 < p.M) c[p.ldc] = p.alpha * sy + (p.beta != 0.0 ? p.beta * c[p.ldc] : 0.0);
  }
}
// ta == 0: A[m * lda + k].  One warp per row, lanes along k (two adjacent k per lane).
__global__ void __launch_bounds__(256) dgemv_kcontig_kernel(GemmArgs p, int64_t xs) {
  const int lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int64_t zb = blockIdx.y, r = zb / p.splitk, s = zb % p.splitk;
  const int64_t kbeg = s * p.kchunk, kend = min(p.K, kbeg + p.kchunk);
  if (m >= p.M) return;
  const double* __restrict__ a = p.A + r * p.sA + m * p.lda;
  const double* __restrict__ x = p.B + r * p.sB;
  double s0 = 0.0, s1 = 0.0;
  if (p.vecA && xs == 1 && (kbeg & 1) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    // 512 k per pass: eight independent (predicated) 16-byte loads of A and of x per lane
    for (int64_t k0 = kbeg; k0 < kend; k0 += 512) {
      double2 av[8], xv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int64_t k = k0 + 2 * lane + 64 * u;
        av[u] = make_double2(0.0, 0.0);
        xv[u] = make_double2(0.0, 0.0);
        if (k + 1 < kend) {
          av[u] = *reinterpret_cast<const double2*>(a + k);
          xv[u] = *reinterpret_cast<const double2*>(x + k);
        } else if (k < kend) {
          av[u].x = a[k];
          xv[u].x = x[k];
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        s0 = fma(av[u].x, xv[u].x, s0);
        s1 = fma(av[u].y, xv[u].y, s1);
      }
    }
  } else {
    for (int64_t k = kbeg + lane; k < kend; k += 32) s0 = fma(a[k], x[k * xs], s0);
  }
  s0 += s1;
#pragma unroll
  for (int o = 16; o; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
  if (lane == 0) {
    double* c = p.C + zb * p.sC + m * p.ldc;
    c[0] = p.alpha * s0 + (p.beta != 0.0 ? p.beta * c[0] : 0.0);
  }
}

cudaError_t launch_gemv(const GemmArgs& p, cudaStream_t st) {
  const int64_t xs = p.tb ? 1 : p.ldb;             // B[k*ldb + 0] (tb == 0) or B[0*ldb + k] (tb == 1)
  if (p.ta) {
    dim3 grid((unsigned)((p.M + 127) / 128), (unsigned)p.batch, 1);
    dgemv_mcontig_kernel<<<grid, 256, 0, st>>>(p, xs);
  } else {
    dim3 grid((unsigned)((p.M + 7) / 8), (unsigned)p.batch, 1);
    dgemv_kcontig_kernel<<<grid, 256, 0, st>>>(p, xs);
  }
  return cudaGetLastError();
}

template <int BM, int BN, int WM, int WN, int BK, int STAGES, int ILV>
cudaError_t launch_cfg(const GemmArgs& p, cudaStream_t st) {
  constexpr int THREADS = (BM / WM) * (BN / WN) * 32;
  int64_t tiles = ((p.M + BM - 1) / BM) * ((p.N + BN - 1) / BN);
  dim3 grid((unsigned)tiles, (unsigned)p.batch, 1);
#define ECW_LAUNCH(TA_, TB_)                                                                        \
  {                                                                                                 \
    auto kern = dgemm_kernel<BM, BN, WM, WN, BK, TA_, TB_, STAGES, ILV>;                                      \
    size_t smem = sizeof(double) * STAGES * SmemLayout<BM, BN, BK, TA_, TB_>::STAGE;                     \
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e != cudaSuccess) return e;                                                                 \
    kern<<<grid, THREADS, smem, st>>>(p);                                                           \
    return cudaGetLastError();                                                                      \
  }
  if (p.ta == 0 && p.tb == 0) ECW_LAUNCH(0, 0)
  if (p.ta == 0 && p.tb == 1) ECW_LAUNCH(0, 1)
  if (p.ta == 1 && p.tb == 0) ECW_LAUNCH(1, 0)
  ECW_LAUNCH(1, 1)
#undef ECW_LAUNCH
}

}  // namespace

int gemm_pick_config(int64_t M, int64_t N, int64_t K) {
  // 1: 32x128  2: 128x32  3: 128x8  4: 64x64  8: 128x128 (16 warps, interleaved loads)
  // 10: 112x128  11: 96x128 (8 warps) — chosen when they cut the padded-row waste of the M dimension
  // 12: 48x128  13: 128x48 — one tile covers a whole occupied index of up to 48 (no operand re-read)
  // 14: 40x40  15: 48x48 — both extents an occupied index
  // 16: 128x40 — N an occupied index of 33..40 (ovvv.t1 products: no DMMA work on padding columns)
  // 18: 40x128  19: 80x80, both with BK = 8 and six stages — short-K rank updates (see below)
  // (tried and dropped: issuing the old-C loads of a short-K tile before the operand wait — 2-3x slower, gemm per-op
  //  logs profiles/r2_perop_dmma_variants.md)
  // (tried and dropped: 40x200 and 40x80 tiles for ovvv.t2 — five-warp CTAs do not cover the loads, slower than 48x128:
  //  17.6 vs 13.2 ms and 16.2 vs 12.5 ms; the 40x200 run is in profiles/r2_perop_dmma_variants.md)
  if (N <= 8) return 3;
  auto padded = [](int64_t x, int64_t b) { return (x + b - 1) / b * b; };
  if (K > 0 && K <= 40 && K % 8 == 0 && N >= 80) {
    // rank updates over an occupied index (K = nocc, huge M*N): BK = 8 tiles carry no K padding, exact 40 / 80 extents
    // no M/N padding (a 48x128x48 tile spends 1.44x the DMMA work of 40x128x40), and the small stages leave room for
    // three CTAs per SM — these launches are bound by the memory round trips of a tile, not by a pipe
    if (M > 16 && M <= 40) return 18;
    if (M > 40 && padded(N, 80) <= padded(N, 128) && padded(M, 80) <= padded(M, 128)) return 19;
  }
  if (M <= 40 && N <= 40 && M > 16 && N > 16) return 14;     // Gram products over a long index ([mnef,inef->mi], ...):
  if (M <= 48 && N <= 48 && M > 16 && N > 16) return 15;     // one exact tile, no DMMA work on padding columns
  if (M <= 32) return 1;
  if (M <= 48) return 12;
  if (N <= 32) return 2;
  if (N <= 40) return 16;
  if (N <= 48) return 13;
  if (M <= 96 || N <= 96) return 4;
  double w128 = (double)padded(M, 128) * padded(N, 128);
  double w64 = (double)padded(M, 64) * padded(N, 64);
  if (w64 * 1.15 < w128) return 4;
  double p128 = (double)padded(M, 128), p112 = (double)padded(M, 112), p96 = (double)padded(M, 96);
  if (p112 * 1.04 < p128 && p112 <= p96) return 10;
  if (p96 * 1.06 < p128 && p96 < p112) return 11;
  return 8;
}

void gemm_tile_of(int64_t M, int64_t N, int64_t K, int* bm, int* bn) {
  // indexed by the configurations gemm_pick_config returns; {0, 0}: numbers it never returns
  static const int dims[20][2] = {{0, 0}, {32, 128}, {128, 32}, {128, 8}, {64, 64}, {0, 0}, {0, 0}, {0, 0},
                                  {128, 128}, {0, 0}, {112, 128}, {96, 128}, {48, 128}, {128, 48}, {40, 40}, {48, 48},
                                  {128, 40}, {0, 0}, {40, 128}, {80, 80}};
  const int cfg = gemm_pick_config(M, N, K);
  *bm = dims[cfg][0];
  *bn = dims[cfg][1];
}

cudaError_t launch_gemm(const GemmArgs& args, cudaStream_t st, int force_cfg) {
  GemmArgs p = args;
  if (p.M <= 0 || p.N <= 0 || p.batch <= 0) return cudaSuccess;
  if (p.splitk < 1) p.splitk = 1;
  if (p.splitk == 1) p.kchunk = p.K;
  auto aligned = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  p.vecA = aligned(p.A) && (p.lda % 2 == 0) && (p.sA % 2 == 0);
  p.vecB = aligned(p.B) && (p.ldb % 2 == 0) && (p.sB % 2 == 0);
  p.vecC = aligned(p.C) && (p.ldc % 2 == 0) && (p.sC % 2 == 0);
  if (p.batch > 65535) return cudaErrorInvalidValue;
  // matrix-vector products with long rows / many rows; short rows (K = nvir) and M-contiguous A with few rows and many
  // K slices keep the GEMM route, which measured faster there (profiles/r2_perop_dmma_variants.md)
  if (p.N == 1 && force_cfg < 0 && (p.M + 7) / 8 < 0x7fffffff && (p.ta ? p.M >= 1024 : p.kchunk >= 2048))
    return launch_gemv(p, st);
  int cfg = force_cfg >= 0 ? force_cfg : gemm_pick_config(p.M, p.N, p.kchunk);
  // large aligned problems: TMA producer + mbarrier ring + DMMA consumers (gemm_tma.cu)
  const bool tma_cfg = cfg == 20 || cfg == 21;
  if (tma_cfg || (force_cfg < 0 && (cfg == 8 || cfg == 10 || cfg == 11))) {
    if (gemm_tma_eligible(p)) {
      int tcfg = tma_cfg ? cfg : ((cfg != 8 && p.ta == 0) ? 21 : 20);
      cudaError_t e = launch_gemm_tma(p, st, tcfg);
      if (e != cudaErrorNotSupported) return e;
      cudaGetLastError();
    }
    if (tma_cfg) cfg = 8;
  }
  switch (cfg) {
    case 1: return launch_cfg<32, 128, 16, 32, 16, 4, 0>(p, st);
    case 2: return launch_cfg<128, 32, 32, 16, 16, 4, 0>(p, st);
    case 3: return launch_cfg<128, 8, 16, 8, 16, 4, 0>(p, st);
    case 4: return launch_cfg<64, 64, 32, 16, 16, 4, 0>(p, st);
    case 8: return launch_cfg<128, 128, 32, 32, 16, 4, 1>(p, st);
    case 10: return launch_cfg<112, 128, 56, 32, 16, 4, 1>(p, st);
    case 12: return launch_cfg<48, 128, 48, 16, 16, 4, 1>(p, st);
    case 13: return launch_cfg<128, 48, 32, 24, 16, 4, 1>(p, st);
    case 11: return launch_cfg<96, 128, 48, 32, 16, 4, 1>(p, st);
    case 14: return launch_cfg<40, 40, 40, 8, 16, 4, 1>(p, st);
    case 15: return launch_cfg<48, 48, 48, 8, 16, 4, 1>(p, st);
    case 16: return launch_cfg<128, 40, 32, 40, 16, 4, 1>(p, st);
    case 18: return launch_cfg<40, 128, 40, 16, 8, 6, 1>(p, st);
    case 19: return launch_cfg<80, 80, 40, 40, 8, 6, 1>(p, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace ecw
