// ozaki.cu — FP64 GEMM on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM).
//
// Blackwell's tcgen05 path has no FP64 kind; the native FP64 tensor instruction is the legacy DMMA
// (gemm_tma.cu, 37 TFLOP/s pipe peak).  The large contractions of the CC residual (CCSD.py:305 ladder,
// :411 ring, :602 Lambda intermediates) are instead evaluated by splitting the FP64 operands into int8
// digits (Ozaki scheme I) and multiplying the digit planes on the INT8 tensor pipe (4.5 POP/s nominal):
//
//   row r of an operand X[R,K]:  s_r = 2^e_r with |X[r,:]| < s_r;  y = (X[r,k]/s_r + 1)/2 in [0,1) is
//   written in base 256,  y ~ Y 256^-NS,  Y = min(rint(y 256^NS), 256^NS - 1) = sum_{p=1..NS} u_p 256^(NS-p),
//   u_p in [0,255], and stored as the int8 digit  d_p = u_p - 128.  The offsets cancel the "-1" almost exactly:
//       X[r,k] = s_r (2 D + c) + delta,   D = sum_p d_p 256^-p,  c = sum_{p=1..NS-1} 256^-p,
//       |delta| <= s_r 256^-NS (2 s_r 256^-NS in the one clamped case y = 1).
//       (8 bits per int8 digit: NS = 6 digits carry 48 bits.)
//   C[m,n] = sA_m sB_n sum_k (2 Da + c)(2 Db + c) = sA_m sB_n ( 4 P[m,n] + c (tA_m + tB_n) - c^2 K ),
//       P = sum_k Da Db  ~  sum_{p+q <= NS+1} 256^-(p+q) (A_p . B_q^T)      (triangular truncation),
//       t_r = sum_k X[r,k] / s_r  (FP64 row sums, taken while looking for the row maximum).
//   Every int8 product A_p . B_q^T is exact in the int32 accumulator (|d d'| <= 2^14; the accumulators
//   are drained to FP64 every oz_kflush(NS) k, at most NS products each: < 2^31).  Worst-case error: representation
//   4 K 256^-NS + truncation (NS-1) K 256^-NS, relative to sA_m sB_n (< 4 max|A_m| max|B_n|): for NS = 6
//   that is 2^-44.8 K sA sB; observed 1e-14 at 8192^3 on N(0,1) data — the size of the rounding error of a
//   DMMA/FMA dot product of that length.
//   NS(NS+1)/2 int8 products replace one FP64 product: 21 at NS = 6.
//   K-padding holds d = 0 (D = 0 contributes nothing to P; the rank-one terms use the true K).
//
// Data layout (memory laid out for the MMA, not for the host): an operand is stored as *digit planes*
//   planes[kb][p][rg][j][ri][16]   kb = k/32, p = digit, rg = r/8, j = (k%32)/16, ri = r%8
// i.e. for a fixed (k-block, digit) all rows are contiguous in the tcgen05 "no-swizzle K-major" core
// matrix order (8 rows x 16 bytes = 128 contiguous bytes; SBO = 256 B between 8-row groups, LBO =
// 128 B between the two 16-byte k-chunks).  A 128-row A tile of one digit is ONE contiguous 4 KB span,
// a TN-row B tile a TN*32-byte span: the producer streams them with linear bulk TMA (cp.async.bulk), no
// tensor maps, no swizzle, and any operand can serve on either side.  Rows are padded to 128, k to 32.
//
// Kernel (one CTA per SM, persistent over 128 x TN output tiles, 192 threads; TN = 80 at NS = 6):
//   warp 0   lane 0: TMA producer — per k-block one stage = NS A-planes + NS B-planes, mbarrier ring;
//   warp 1   lane 0: MMA issuer — tcgen05.mma kind::i8 (s8 x s8 -> s32, M128 K32); product (p,q)
//                    accumulates into TMEM columns [TN(p+q), TN(p+q)+TN): all products of one weight share
//                    an accumulator and all NS digits of A and B are loaded once per k-block.  Digits
//                    q = 0..NS-1-p of B are contiguous in shared memory, so they are issued as one MMA of
//                    N = TN (NS-p) columns (split at 256);
//   warps 2-5      : epilogue — tcgen05.ld the NS accumulators, Horner in FP64, rank-one terms, scales,
//                    alpha/beta, store (coalesced across lanes when the tile rows are contiguous in C).
// Measured limiter (profiles/r1_oz_limiter.md): a stage is 39.9 KB and 840 clk of MMA
// (47 B/clk); an SM ingests ~32.6 B/clk from L2 whatever the path (bulk TMA, cp.async, both), so the main loop
// runs at 1224 clk per stage = 69 % of the pipe; without loads it reaches 87 %.  TMEM (NS accumulators x TN
// columns <= 512) is what keeps the tile, and with it the bytes per MAC, from growing.
#include <cuda.h>
#include <cstdio>

#include "kernels.h"

namespace ecw {

namespace {

// int32 accumulators are drained to FP64 every oz_kflush(NS) k.  The accumulator of weight NS-1 sums NS digit products
// per k, each at most 128 * 128 = 2^14 in magnitude: NS * K * 2^14 < 2^31 needs K < 2^17 / NS.  8192 keeps a factor of
// two of headroom for every digit count (16384 is admissible up to seven digits and was measured: no gain — the drain
// is ~1 % of a chunk; tests/test_gpu_int8.py::test_int8_accumulator_headroom runs the all-(-128) worst case).
__host__ __device__ constexpr int oz_kflush(int) { return 8192; }
constexpr int OZ_SMEM_MAX = 227 * 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// linear bulk TMA: global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// D[tmem] (+)= A[smem] . B[smem]^T, signed 8-bit operands, int32 accumulate; one thread issues for the CTA
__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
               : "memory");
}
// 8 consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// shared-memory matrix descriptor, K-major, no swizzle (core matrix = 8 rows x 16 bytes, 128 B contiguous):
// bits [0,14) start>>4, [16,30) leading byte offset>>4 (between the two 16-byte k-chunks),
// [32,46) stride byte offset>>4 (between 8-row groups), [46,48) version = 1 (sm_100), [61,64) layout = 0
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | ((uint64_t)1 << 46);
}

struct OzGemmParams {
  const int8_t* pa;      // digit planes of the M-side operand
  const int8_t* pb;      // digit planes of the N-side operand
  const double* sa;      // statistics of the M-side plane set: [scales | row sums | per-k1 row sums ...]
  const double* sb;
  double* C;
  int64_t M, N, K;       // logical extents of ONE product (K = true contraction length of a batch)
  int64_t Mp, Np;        // padded row counts of the two plane sets (multiples of 128)
  int64_t crs, ccs;      // C[b*c_b + m*crs + n*ccs]
  double alpha, beta;
  double cprime;         // c = sum_{p=1..NS-1} 256^-p
  uint32_t lbo, sbo;     // descriptor strides (bytes)
  // batch b = 0..batch-1 of independent products (OzBatch, kernels.h)
  OzBatch bt;
};

template <int NS, int TN>
struct OzCfg {
  static constexpr int A_PLANE = OZ_TM * OZ_BK;           // 4096
  static constexpr int B_PLANE = TN * OZ_BK;
  static constexpr int STAGE = NS * (A_PLANE + B_PLANE);
  static constexpr int STAGES = (OZ_SMEM_MAX - 2048) / STAGE > 8 ? 8 : (OZ_SMEM_MAX - 2048) / STAGE;
  static constexpr int SMEM = STAGES * STAGE + 1024 /*align*/ + 256 /*barriers*/;
  static constexpr int TMEM_COLS = 512;
  static_assert(NS * TN <= 512, "accumulators exceed TMEM");
  static_assert(TN % 16 == 0, "MMA N granularity");
};

// tile index -> (m block, n block); groups of 8 m-blocks are swept along n so that the CTAs running
// together share A and B panels in L2
__device__ __forceinline__ void tile_coord(int64_t tile, int64_t tiles_m, int64_t tiles_n, int64_t& tm, int64_t& tn) {
  const int64_t GROUP = 8;
  const int64_t per_group = GROUP * tiles_n, gid = tile / per_group, first_m = gid * GROUP;
  const int64_t gsz = min(tiles_m - first_m, GROUP);
  tm = first_m + (tile % per_group) % gsz;
  tn = (tile % per_group) / gsz;
}

template <int NS, int TN>
__global__ void __launch_bounds__(192, 1) ozaki_gemm_kernel(OzGemmParams p) {
  using Cfg = OzCfg<NS, TN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t tiles_m = (p.M + OZ_TM - 1) / OZ_TM, tiles_n = (p.N + TN - 1) / TN;
  const int64_t tiles_mn = tiles_m * tiles_n;
  const int64_t ntiles = tiles_mn * p.bt.batch;
  const int nkb = p.bt.nkb > 0 ? (int)p.bt.nkb : (int)((p.K + OZ_BK - 1) / OZ_BK);
  constexpr int KB_FLUSH = oz_kflush(NS) / OZ_BK;
  const int nchunk = (nkb + KB_FLUSH - 1) / KB_FLUSH;

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)Cfg::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =================== TMA producer ===================
    if (lane == 0) {
      const int64_t a_slab = p.Mp * OZ_BK;   // bytes of one (k-block, digit) slab
      const int64_t b_slab = p.Np * OZ_BK;
      uint32_t it = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int64_t tm, tn;
        const int64_t b = tile / tiles_mn;
        tile_coord(tile - b * tiles_mn, tiles_m, tiles_n, tm, tn);
        const int8_t* ga = p.pa + (p.bt.a_row0 + b * p.bt.a_rowb) * OZ_BK + tm * Cfg::A_PLANE +
                           (p.bt.a_kb0 + b * p.bt.a_kbb) * NS * a_slab;
        const int8_t* gb = p.pb + (p.bt.b_row0 + b * p.bt.b_rowb) * OZ_BK + tn * Cfg::B_PLANE +
                           (p.bt.b_kb0 + b * p.bt.b_kbb) * NS * b_slab;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t st = it % STAGES, use = it / STAGES;
          mbar_wait(&empty[st], (use & 1) ^ 1);
          unsigned char* s = smem + st * Cfg::STAGE;
          mbar_expect_tx(&full[st], Cfg::STAGE);
#pragma unroll
          for (int d = 0; d < NS; ++d) {
            bulk_load(s + d * Cfg::A_PLANE, ga + ((int64_t)kb * NS + d) * a_slab, Cfg::A_PLANE, &full[st]);
            bulk_load(s + NS * Cfg::A_PLANE + d * Cfg::B_PLANE, gb + ((int64_t)kb * NS + d) * b_slab, Cfg::B_PLANE,
                      &full[st]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // =================== MMA issuer ===================
    if (lane == 0) {
      // instruction descriptor: D = s32 (2 @bit4), A = B = signed 8-bit (1 @bit7, 1 @bit10), both K-major,
      // N>>3 @bit17, M>>4 @bit24
      const uint32_t idesc0 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_TM >> 4) << 24);
      const uint64_t desc0 = make_desc(0, p.lbo, p.sbo);
      const uint32_t sbase = smem_u32(smem);
      uint32_t it = 0, acc_it = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int c = 0; c < nchunk; ++c, ++acc_it) {
          mbar_wait(tmem_empty, (acc_it & 1) ^ 1);
          tc_fence_after();
          const int kb0 = c * KB_FLUSH, kb1 = min(nkb, kb0 + KB_FLUSH);
          for (int kb = kb0; kb < kb1; ++kb, ++it) {
            const uint32_t st = it % STAGES, use = it / STAGES;
            mbar_wait(&full[st], use & 1);
            tc_fence_after();
            const uint32_t sa = sbase + st * Cfg::STAGE, sb = sa + NS * Cfg::A_PLANE;
            // The B digit planes of a stage are contiguous, so digits q = 0..NS-1-pd form ONE operand of
            // TN (NS-pd) rows: A_pd . [B_0; ..; B_{NS-1-pd}]^T lands in the TMEM columns of the weights
            // pd .. NS-1, which are contiguous too.  One MMA per <= 256 columns.
#pragma unroll
            for (int pd = 0; pd < NS; ++pd) {
              const uint64_t adesc = desc0 | (uint64_t)(((sa + pd * Cfg::A_PLANE) >> 4) & 0x3fff);
              const int ncols = TN * (NS - pd);
#pragma unroll
              for (int n0 = 0; n0 < ncols; n0 += 256) {
                const int nlen = ncols - n0 < 256 ? ncols - n0 : 256;
                const uint64_t bdesc = desc0 | (uint64_t)(((sb + n0 * OZ_BK) >> 4) & 0x3fff);
                mma_i8(tmem_base + (uint32_t)(pd * TN + n0), adesc, bdesc, idesc0 | ((uint32_t)(nlen >> 3) << 17),
                       (kb > kb0 || pd > 0) ? 1u : 0u);
              }
            }
            mma_commit(&empty[st]);
          }
          mma_commit(tmem_full);
        }
      }
    }
  } else {
    // =================== epilogue (4 warps = 128 TMEM lanes = 128 tile rows) ===================
    const int quad = warp & 3;                 // a warp may only touch TMEM lanes [32*(warp%4), +32)
    const int row = quad * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
    const double w = 0.00390625;               // 2^-8
    const double cK = p.cprime * p.cprime * (double)p.K;
    uint32_t acc_it = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int64_t tm, tn;
      const int64_t b = tile / tiles_mn;
      tile_coord(tile - b * tiles_mn, tiles_m, tiles_n, tm, tn);
      const int64_t m = tm * OZ_TM + row, n0 = tn * TN;
      double run[TN];
#pragma unroll
      for (int j = 0; j < TN; ++j) run[j] = 0.0;
      for (int c = 0; c < nchunk; ++c, ++acc_it) {
        mbar_wait(tmem_full, acc_it & 1);
        tc_fence_after();
#pragma unroll
        for (int cb = 0; cb < TN / 8; ++cb) {
          int32_t v[NS][8];
#pragma unroll
          for (int d = 0; d < NS; ++d) tmem_ld8(tlane + (uint32_t)(d * TN + cb * 8), v[d]);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            double s = (double)v[NS - 1][j];
#pragma unroll
            for (int d = NS - 2; d >= 0; --d) s = fma(s, w, (double)v[d][j]);
            run[cb * 8 + j] += s;
          }
        }
        tc_fence_before();
        mbar_arrive(tmem_empty);
      }
      if (m < p.M) {
        // C = alpha sA sB (4 * 2^-16 H + c (tA + tB) - c^2 K) + beta C
        const int64_t ar = p.bt.a_row0 + b * p.bt.a_rowb + m, br = p.bt.b_row0 + b * p.bt.b_rowb;
        const double* __restrict__ ta = p.sa + p.bt.a_t0 + b * p.bt.a_tb;
        const double* __restrict__ tb = p.sb + p.bt.b_t0 + b * p.bt.b_tb;
        const double fa = p.alpha * p.sa[ar];
        const double um = p.cprime * ta[ar] - cK;
        double* crow = p.C + b * p.bt.c_b + m * p.crs + n0 * p.ccs;
        const int nn = (int)min((int64_t)TN, p.N - n0);
        const bool vec = p.ccs == 1 && nn == TN && ((reinterpret_cast<uintptr_t>(crow) & 15) == 0);
#pragma unroll
        for (int jc = 0; jc < TN; jc += 8) {
          double o[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const int64_t n = br + min(n0 + jc + q, p.N - 1);
            o[q] = fa * p.sb[n] * (fma(run[jc + q], 6.103515625e-05 /* 4 * 2^-16 */, um) + p.cprime * tb[n]);
          }
          if (vec) {
            if (p.beta != 0.0) {
              double2 old[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) old[q] = *reinterpret_cast<const double2*>(crow + jc + 2 * q);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                o[2 * q] += p.beta * old[q].x;
                o[2 * q + 1] += p.beta * old[q].y;
              }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) *reinterpret_cast<double2*>(crow + jc + 2 * q) = make_double2(o[2 * q], o[2 * q + 1]);
          } else {
            if (p.beta != 0.0) {
              double old[8];
#pragma unroll
              for (int q = 0; q < 8; ++q) old[q] = (jc + q < nn) ? crow[(jc + q) * p.ccs] : 0.0;
#pragma unroll
              for (int q = 0; q < 8; ++q) o[q] += p.beta * old[q];
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
              if (jc + q < nn) crow[(jc + q) * p.ccs] = o[q];
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// row statistics: s_r = 2^e_r with |X[r,:]| < s_r (1 for an all-zero or padded row), t_r = sum_k X[r,k] / s_r
// (fixed summation order) and, for a two-level contraction index k = (k1, k2), the partial sums per k1.
// X[r*rs + k1*ks1 + k2*ks2]; stats = [scales (Rp) | row sums (Rp) | row sums per k1 (K1 x Rp) when K1 > 1]
// with Rp the padded row count of the WHOLE plane set; the pointers passed here are offset to the chunk's first row.
// A row that holds a NaN or an Inf gets the scale NaN: every product it takes part in is then NaN in the GEMM
// epilogue (alpha * s_m * s_n * ...), as in an FP64 GEMM — the digits of such a row are meaningless.
__device__ __forceinline__ double oz_scale_of(double mx) {
  if (!(mx <= 1.7976931348623157e308)) return __longlong_as_double(0x7ff8000000000000ll);
  int e = 0;
  if (mx > 0.0) frexp(mx, &e);          // mx = f 2^e, f in [0.5, 1)
  // an all-zero (or padded) row: a scale so small that s_m s_n underflows to an exact 0 in the epilogue and the row
  // does not count in the run-time error bound (ozaki_bound_kernel); its digits stand for 2D + c = 0 exactly
  return mx > 0.0 ? ldexp(1.0, e) : 2.4099198651028841e-181 /* 2^-600 */;
}
// max that keeps a NaN once seen (fmax would drop it); a, b >= 0 or NaN
__device__ __forceinline__ double oz_max(double a, double b) { return (b > a || b != b) ? b : a; }
// one warp per row (k2 contiguous)
__global__ void ozaki_rowstat_kcontig(const double* __restrict__ X, int64_t R, int64_t K1, int64_t K2, int64_t rs,
                                      int64_t ks1, int64_t Rp_chunk, int64_t Rp, double* __restrict__ stats) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= Rp_chunk) return;
  double mx = 0.0, tot = 0.0;
  for (int64_t k1 = 0; k1 < K1; ++k1) {
    double sm = 0.0;
    if (r < R) {
      const double* x = X + r * rs + k1 * ks1;
      double s1 = 0.0, s2 = 0.0, s3 = 0.0;
      int64_t k = lane;
      for (; k + 96 < K2; k += 128) {                         // four independent loads in flight per lane
        const double v0 = x[k], v1 = x[k + 32], v2 = x[k + 64], v3 = x[k + 96];
        mx = oz_max(oz_max(mx, fabs(v0)), oz_max(oz_max(fabs(v1), fabs(v2)), fabs(v3)));
        sm += v0; s1 += v1; s2 += v2; s3 += v3;
      }
      for (; k < K2; k += 32) {
        const double v = x[k];
        mx = oz_max(mx, fabs(v));
        sm += v;
      }
      sm += s1 + s2 + s3;
#pragma unroll
      for (int o = 16; o; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
    }
    tot += sm;
    if (K1 > 1 && lane == 0) stats[(2 + k1) * Rp + r] = sm;     // scaled below
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = oz_max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) {
    const double s = oz_scale_of(mx);
    stats[r] = s;
    stats[Rp + r] = tot / s;
    if (K1 > 1)
      for (int64_t k1 = 0; k1 < K1; ++k1) stats[(2 + k1) * Rp + r] /= s;
  }
}
// rows contiguous: 32 rows x 8 k-lanes per block, grid.y = K1 * C2 (k2 cut into C2 chunks so that operands with few
// rows and a long contraction index still fill the machine).  Row maxima are combined with atomicMax on the bit
// pattern (non-negative doubles order like integers; order independent), partial sums go to `part` and are added in
// a fixed order by ozaki_rowstat_finish.
__global__ void ozaki_rowstat_rcontig(const double* __restrict__ X, int64_t R, int64_t K1, int64_t K2, int64_t ks1,
                                      int64_t ks2, int64_t C2, int64_t Rp_chunk, int64_t Rp, double* __restrict__ stats,
                                      double* __restrict__ part) {
  __shared__ double red[8][33], reds[8][33];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * 32 + lane;
  const int64_t k1 = blockIdx.y / C2, c = blockIdx.y - k1 * C2;
  const int64_t len = (K2 + C2 - 1) / C2, kbeg = c * len, kend = min(K2, kbeg + len);
  double mx = 0.0, sm = 0.0;
  if (r < R) {
    const double* x = X + r + k1 * ks1;
    double s1 = 0.0;
    int64_t k = kbeg + wy;
    for (; k + 8 < kend; k += 16) {
      const double v0 = x[k * ks2], v1 = x[(k + 8) * ks2];
      mx = oz_max(oz_max(mx, fabs(v0)), fabs(v1));
      sm += v0; s1 += v1;
    }
    for (; k < kend; k += 8) {
      const double v = x[k * ks2];
      mx = oz_max(mx, fabs(v));
      sm += v;
    }
    sm += s1;
  }
  red[wy][lane] = mx;
  reds[wy][lane] = sm;
  __syncthreads();
  if (wy == 0 && r < Rp_chunk) {
#pragma unroll
    for (int i = 1; i < 8; ++i) {
      mx = oz_max(mx, red[i][lane]);
      sm += reds[i][lane];
    }
    // bit patterns of non-negative doubles order like integers; +Inf and (positive) NaN sort above every finite value
    atomicMax(reinterpret_cast<unsigned long long*>(stats + r), (unsigned long long)__double_as_longlong(fabs(mx)));
    part[(k1 * C2 + c) * Rp + r] = sm;
  }
}
// stats[r] holds the row maximum (bit pattern); part[(k1*C2 + c)*Rp + r] the partial sums
__global__ void ozaki_rowstat_finish(int64_t K1, int64_t C2, int64_t Rp_chunk, int64_t Rp, double* __restrict__ stats,
                                     const double* __restrict__ part) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= Rp_chunk) return;
  const double s = oz_scale_of(stats[r]);
  double tot = 0.0;
  for (int64_t k1 = 0; k1 < K1; ++k1) {
    double sm = 0.0;
    for (int64_t c = 0; c < C2; ++c) sm += part[(k1 * C2 + c) * Rp + r];
    tot += sm;
    if (K1 > 1) stats[(2 + k1) * Rp + r] = sm / s;
  }
  stats[r] = s;
  stats[Rp + r] = tot / s;
}

// cut X into NS digit planes (layout in the header comment).  Block = 128 rows x one k-block (32 k2 of one k1),
// thread t: row t%128, 16-byte k-chunk t/128.  k-block index = k1 * ceil(K2/32) + k2/32: k2 is padded per k1.
// Digits: Y = min(rint(y 2^(8 NS)), 2^(8 NS) - 1) as an integer; digit p is byte NS-1-p of Y, stored with the top
// bit flipped (u - 128 as int8).  One FP64 fma, one multiply and one conversion per element; the rest is byte
// permutes, so the kernel runs at memory speed.  Padding carries 0x80 bytes in Y so that it is stored as d = 0.
template <int NS>
__global__ void __launch_bounds__(256) ozaki_split_kernel(const double* __restrict__ X, int64_t R, int64_t K2, int64_t rs,
                                                          int64_t ks1, int64_t ks2, int64_t Rp, int64_t row0,
                                                          const double* __restrict__ scale,
                                                          int8_t* __restrict__ planes) {
  // X, scale: the chunk (local rows 0..R); planes: the whole set of Rp padded rows, chunk rows start at row0
  const int t = threadIdx.x;
  const int64_t r = (int64_t)blockIdx.x * 128 + (t & 127);
  const int j = t >> 7;
  const int64_t kb = blockIdx.y;
  const int64_t nkb2 = (K2 + OZ_BK - 1) / OZ_BK;
  const int64_t k1 = kb / nkb2;
  const int64_t k0 = (kb - k1 * nkb2) * OZ_BK + j * 16;
  constexpr unsigned long long PAD = 0x8080808080808080ull;
  constexpr unsigned long long YMAX = NS >= 8 ? ~0ull : ((1ull << (8 * (NS & 7))) - 1ull);
  constexpr double two = NS >= 4 ? (double)(1ull << 32) * (double)(1ull << (NS >= 4 ? 8 * NS - 32 : 0))
                                 : (double)(1ull << (NS >= 4 ? 0 : 8 * NS));                // 2^(8 NS)
  uint32_t lo[16], hi[16];
  auto digits_of = [&](double x, double inv, int i) {
    const double y = fma(x, inv, 0.5);                       // (x/s + 1)/2 in [0, 1]
    unsigned long long Y = __double2ull_rn(y * two);         // exact scaling, one rounding; saturates at 2^64-1
    Y = Y < YMAX ? Y : YMAX;
    lo[i] = (uint32_t)Y;
    hi[i] = (uint32_t)(Y >> 32);
  };
  if (r < R) {
    const double inv = 0.5 / scale[r];     // exact: a power of two
    const double* src = X + r * rs + k1 * ks1 + k0 * ks2;
    if (ks2 == 1 && k0 + 16 <= K2 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
      double2 v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const double2*>(src + 2 * i);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        digits_of(v[i].x, inv, 2 * i);
        digits_of(v[i].y, inv, 2 * i + 1);
      }
    } else {
      double v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = (k0 + i < K2) ? src[i * ks2] : 0.0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (k0 + i < K2) digits_of(v[i], inv, i);
        else { lo[i] = (uint32_t)PAD; hi[i] = (uint32_t)(PAD >> 32); }
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) { lo[i] = (uint32_t)PAD; hi[i] = (uint32_t)(PAD >> 32); }
  }
  const int64_t slab = Rp * OZ_BK;
  const int64_t rg = row0 + r;
  int8_t* dst = planes + (kb * NS) * slab + (rg >> 3) * 256 + j * 128 + (rg & 7) * 16;
#pragma unroll
  for (int p = 0; p < NS; ++p) {
    constexpr uint32_t FLIP = 0x80808080u;
    const int b = NS - 1 - p;                                // byte of Y that holds digit p
    const uint32_t sel = (uint32_t)((b & 3) | (((b & 3) + 4) << 4));          // byte b of two words -> low half
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t* s4 = (b < 4 ? lo : hi) + 4 * q;
      const uint32_t t01 = __byte_perm(s4[0], s4[1], sel), t23 = __byte_perm(s4[2], s4[3], sel);
      w[q] = __byte_perm(t01, t23, 0x5410) ^ FLIP;
    }
    *reinterpret_cast<uint4*>(dst + p * slab) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// Run-time error bound of one (batched) product: (NS+3) 256^-NS K |alpha| max_m s_m max_n s_n over the rows the
// product reads (header comment: representation + triangular truncation), combined into *out with an atomic max on
// the bit pattern (non-negative doubles order like integers; a NaN scale — non-finite operand — sorts on top).
__global__ void __launch_bounds__(1024) ozaki_bound_kernel(const double* __restrict__ sa, int64_t a_row0, int64_t a_rowb,
                                                           int64_t M, const double* __restrict__ sb, int64_t b_row0,
                                                           int64_t b_rowb, int64_t N, int64_t batch, double factor,
                                                           double* out) {
  __shared__ double ra[32], rb[32];
  double ma = 0.0, mb = 0.0;
  const int64_t na = (a_rowb ? batch : 1) * M, nb = (b_rowb ? batch : 1) * N;
  for (int64_t i = threadIdx.x; i < na; i += blockDim.x) ma = oz_max(ma, fabs(sa[a_row0 + (i / M) * a_rowb + i % M]));
  for (int64_t i = threadIdx.x; i < nb; i += blockDim.x) mb = oz_max(mb, fabs(sb[b_row0 + (i / N) * b_rowb + i % N]));
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    ma = oz_max(ma, __shfl_xor_sync(0xffffffffu, ma, o));
    mb = oz_max(mb, __shfl_xor_sync(0xffffffffu, mb, o));
  }
  if ((threadIdx.x & 31) == 0) { ra[threadIdx.x >> 5] = ma; rb[threadIdx.x >> 5] = mb; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { ma = oz_max(ma, ra[w]); mb = oz_max(mb, rb[w]); }
    const double bound = fabs(factor * ma * mb);
    atomicMax(reinterpret_cast<unsigned long long*>(out), (unsigned long long)__double_as_longlong(bound));
  }
}

template <int NS, int TN>
cudaError_t launch_gemm_ns_tn(OzGemmParams p, cudaStream_t st, int sm_count) {
  using Cfg = OzCfg<NS, TN>;
  auto kern = ozaki_gemm_kernel<NS, TN>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
  if (e != cudaSuccess) return e;
  double c = 0.0;
  for (int q = 1; q < NS; ++q) c += ldexp(1.0, -8 * q);
  p.cprime = c;
  const int64_t tiles = ((p.M + OZ_TM - 1) / OZ_TM) * ((p.N + TN - 1) / TN) * p.bt.batch;
  const unsigned grid = (unsigned)(tiles < sm_count ? tiles : sm_count);
  kern<<<grid, 192, Cfg::SMEM, st>>>(p);
  return cudaGetLastError();
}
template <int NS>
cudaError_t launch_gemm_ns(OzGemmParams p, cudaStream_t st, int sm_count) {
  return launch_gemm_ns_tn<NS, ozaki_tile_n(NS)>(p, st, sm_count);
}

}  // namespace

cudaError_t launch_ozaki_split2(const double* X, int64_t R, int64_t K1, int64_t K2, int64_t rs, int64_t ks1, int64_t ks2,
                                int ns, int8_t* planes, double* stats, cudaStream_t st, int64_t row0, int64_t total_rows) {
  if (ns < 3 || ns > 8 || (rs != 1 && ks2 != 1) || (row0 & 127) || K1 < 1) return cudaErrorInvalidValue;
  if (total_rows <= 0) total_rows = row0 + R;
  if (row0 + R > total_rows || (row0 + R < total_rows && (R & 127))) return cudaErrorInvalidValue;
  const int64_t Rp = ozaki_padded_rows(R);              // rows this launch writes (incl. zero padding)
  const int64_t Rp_total = ozaki_padded_rows(total_rows);
  double* sc = stats + row0;
  if (ks2 == 1) {
    ozaki_rowstat_kcontig<<<(unsigned)((Rp + 7) / 8), 256, 0, st>>>(X, R, K1, K2, rs, ks1, Rp, Rp_total, sc);
  } else {
    // partial sums: in the statistics array itself when k2 is not chunked (K1 > 1: the per-k1 slots; K1 == 1: the
    // row-sum slot), else in the (not yet written) plane buffer — only for a plane set cut in one piece
    const int64_t rb = (Rp + 31) / 32;
    int64_t C2 = 1;
    if (row0 == 0 && Rp == Rp_total)
      while (rb * K1 * C2 < 1024 && K2 / (C2 * 2) >= 512 && C2 < 256) C2 *= 2;
    if (K1 * C2 > 65535) return cudaErrorInvalidValue;
    double* part = C2 > 1 ? reinterpret_cast<double*>(planes) : (K1 > 1 ? stats + 2 * Rp_total + row0 : stats + Rp_total + row0);
    cudaError_t e = cudaMemsetAsync(sc, 0, (size_t)Rp * sizeof(double), st);
    if (e != cudaSuccess) return e;
    ozaki_rowstat_rcontig<<<dim3((unsigned)rb, (unsigned)(K1 * C2)), 256, 0, st>>>(X, R, K1, K2, ks1, ks2, C2, Rp, Rp_total, sc,
                                                                                  part);
    ozaki_rowstat_finish<<<(unsigned)((Rp + 255) / 256), 256, 0, st>>>(K1, C2, Rp, Rp_total, sc, part);
  }
  const int64_t nkb = ozaki_kblocks(K1, K2);
  if (nkb > 65535) return cudaErrorInvalidValue;
  dim3 grid((unsigned)(Rp / 128), (unsigned)nkb, 1);
  switch (ns) {
#define ECW_OZ_SPLIT(NS_) \
  case NS_: ozaki_split_kernel<NS_><<<grid, 256, 0, st>>>(X, R, K2, rs, ks1, ks2, Rp_total, row0, sc, planes); break;
    ECW_OZ_SPLIT(3) ECW_OZ_SPLIT(4) ECW_OZ_SPLIT(5) ECW_OZ_SPLIT(6) ECW_OZ_SPLIT(7) ECW_OZ_SPLIT(8)
#undef ECW_OZ_SPLIT
  }
  return cudaGetLastError();
}

cudaError_t launch_ozaki_split(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, int8_t* planes,
                               double* scale, cudaStream_t st, int64_t row0, int64_t total_rows) {
  return launch_ozaki_split2(X, R, 1, K, rs, 0, ks, ns, planes, scale, st, row0, total_rows);
}

cudaError_t launch_ozaki_gemm_batched(const int8_t* pa, const double* sa, int64_t a_rows, const int8_t* pb,
                                      const double* sb, int64_t b_rows, int64_t M, int64_t N, int64_t K, double* C,
                                      int64_t crs, int64_t ccs, double alpha, double beta, int ns, const OzBatch& bt,
                                      cudaStream_t st, int sm_count) {
  OzGemmParams p{};
  p.pa = pa; p.pb = pb; p.sa = sa; p.sb = sb; p.C = C;
  p.M = M; p.N = N; p.K = K;
  p.Mp = ozaki_padded_rows(a_rows); p.Np = ozaki_padded_rows(b_rows);
  p.crs = crs; p.ccs = ccs; p.alpha = alpha; p.beta = beta;
  p.lbo = 128; p.sbo = 256;
  p.bt = bt;
  if (bt.batch < 1 || ((bt.a_row0 | bt.a_rowb | bt.b_row0 | bt.b_rowb) & 7)) return cudaErrorInvalidValue;
  if (sm_count <= 0) sm_count = 148;
  switch (ns) {
    case 3: return launch_gemm_ns<3>(p, st, sm_count);
    case 4: return launch_gemm_ns<4>(p, st, sm_count);
    case 5: return launch_gemm_ns<5>(p, st, sm_count);
    case 6: return launch_gemm_ns<6>(p, st, sm_count);
    case 7: return launch_gemm_ns<7>(p, st, sm_count);
    case 8: return launch_gemm_ns<8>(p, st, sm_count);
  }
  return cudaErrorInvalidValue;
}

cudaError_t launch_ozaki_bound(const double* sa, const double* sb, int64_t M, int64_t N, int64_t K, double alpha, int ns,
                               const OzBatch& bt, double* out, cudaStream_t st) {
  if (!out || bt.batch < 1) return cudaErrorInvalidValue;
  const double factor = (double)(ns + 3) * ldexp(1.0, -8 * ns) * (double)K * fabs(alpha);
  ozaki_bound_kernel<<<1, 1024, 0, st>>>(sa, bt.a_row0, bt.a_rowb, M, sb, bt.b_row0, bt.b_rowb, N, bt.batch, factor, out);
  return cudaGetLastError();
}

cudaError_t launch_ozaki_gemm(const int8_t* pa, const double* sa, const int8_t* pb, const double* sb, int64_t M, int64_t N,
                              int64_t K, double* C, int64_t crs, int64_t ccs, double alpha, double beta, int ns,
                              cudaStream_t st, int sm_count) {
  OzBatch bt{};
  bt.batch = 1;
  bt.a_t0 = ozaki_padded_rows(M);        // whole-K row sums
  bt.b_t0 = ozaki_padded_rows(N);
  return launch_ozaki_gemm_batched(pa, sa, M, pb, sb, N, M, N, K, C, crs, ccs, alpha, beta, ns, bt, st, sm_count);
}

}  // namespace ecw
