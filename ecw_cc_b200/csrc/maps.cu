// maps.cu — electron-density maps of a fitted state (sm_100a, FP64 throughout):
// the density rho(r) = sum_mu,nu D_mu,nu phi_mu(r) phi_nu(r) on a box grid (ecw_density_grid) and the Fourier synthesis
// rho(x) = (1/V) sum_h F(h) exp(-2 pi i h.x) on the fractional grid of a unit cell (ecw_fourier_map).
// The references of these kernels are ecw_cc_b200.molint.density_points and molint.fourier_map.
#include "kernels.h"

#include <cmath>

namespace ecw {

namespace {

constexpr int AO_THREADS = 256;
constexpr int RD_THREADS = 256;     // row-dot: one warp per point
constexpr int FM_THREADS = 256;
constexpr int FM_CHUNK = 256;       // reflections staged in shared memory per pass
constexpr int AO_LMAX = 2;          // per-direction angular momentum of one primitive (s, p, d)

// x^l for 0 <= l <= AO_LMAX, the product order of molint.ao_values
__device__ __forceinline__ double ipow(double x, int l) { return l == 0 ? 1.0 : (l == 1 ? x : x * x); }

// Phi[p][mu] for the points p0 .. p0 + np - 1 of the box grid r_ijk = origin + i a1 + j a2 + k a3 (flat index
// (i n2 + j) n3 + k).  One thread per (point, AO), AO fastest, so the stores are coalesced.  Each value is the sum of the
// AO's primitives in table order, coef (x-Ax)^lx (y-Ay)^ly (z-Az)^lz exp(-alpha |r-A|^2), with no screening.  A
// malformed table (primitive range outside [0, nprim) or l outside [0, AO_LMAX]) gives NaN.
__global__ void __launch_bounds__(AO_THREADS)
ao_values_kernel(const double* __restrict__ prim, int64_t nprim, const int64_t* __restrict__ ao_first, int nao,
                 double ox, double oy, double oz, double a1x, double a1y, double a1z, double a2x, double a2y, double a2z,
                 double a3x, double a3y, double a3z, int n2, int n3, int64_t p0, int64_t np, double* __restrict__ phi) {
  const int64_t g = (int64_t)blockIdx.x * AO_THREADS + threadIdx.x;
  if (g >= np * nao) return;
  const int64_t lp = g / nao;
  const int mu = (int)(g - lp * nao);
  const int64_t p = p0 + lp;
  const int64_t i = p / ((int64_t)n2 * n3);
  const int64_t j = (p / n3) % n2;
  const int64_t k = p % n3;
  const double di = (double)i, dj = (double)j, dk = (double)k;
  // ((origin + i a1) + j a2) + k a3 without contraction to FMA: the same rounding as the host expression
  const double x = __dadd_rn(__dadd_rn(__dadd_rn(ox, __dmul_rn(di, a1x)), __dmul_rn(dj, a2x)), __dmul_rn(dk, a3x));
  const double y = __dadd_rn(__dadd_rn(__dadd_rn(oy, __dmul_rn(di, a1y)), __dmul_rn(dj, a2y)), __dmul_rn(dk, a3y));
  const double z = __dadd_rn(__dadd_rn(__dadd_rn(oz, __dmul_rn(di, a1z)), __dmul_rn(dj, a2z)), __dmul_rn(dk, a3z));
  const int64_t q0 = ao_first[mu], q1 = ao_first[mu + 1];
  double v = 0.0;
  if (q0 < 0 || q1 < q0 || q1 > nprim) {
    v = nan("");
  } else {
    for (int64_t q = q0; q < q1; ++q) {
      const double* P = prim + 8 * q;
      const int lx = (int)P[5], ly = (int)P[6], lz = (int)P[7];
      if (lx < 0 || ly < 0 || lz < 0 || lx > AO_LMAX || ly > AO_LMAX || lz > AO_LMAX) { v = nan(""); break; }
      const double dx = x - P[0], dy = y - P[1], dz = z - P[2];
      const double r2 = dx * dx + dy * dy + dz * dz;
      v += P[4] * ipow(dx, lx) * ipow(dy, ly) * ipow(dz, lz) * exp(-P[3] * r2);
    }
  }
  phi[lp * nao + mu] = v;
}

// out[p] = sum_mu X[p][mu] Phi[p][mu]: one warp per point, lane-strided partial sums and a fixed butterfly, so the
// order of the sum is the same on every call.
__global__ void __launch_bounds__(RD_THREADS)
rowdot_kernel(const double* __restrict__ X, const double* __restrict__ phi, int nao, int64_t np,
              double* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * (RD_THREADS / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (p >= np) return;
  const double* x = X + p * nao;
  const double* f = phi + p * nao;
  double s = 0.0;
  for (int mu = lane; mu < nao; mu += 32) s += x[mu] * f[mu];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[p] = s;
}

// m mod n for 0 <= m < n * n <= 2^24: a float quotient estimate (off by at most one) and an integer fix-up
__device__ __forceinline__ int mod_small(int m, int n, float inv_n) {
  int r = m - n * (int)((float)m * inv_n);
  if (r < 0) r += n;
  if (r >= n) r -= n;
  return r;
}

// rho at the fractional grid points x_ijk = (i/n1, j/n2, k/n3): one thread per point (flat index (i n2 + j) n3 + k).
// The block stages FM_CHUNK reflections (h reduced mod n_d, Re F, Im F) and the per-axis tables (cos, sin)(2 pi m / n_d)
// in shared memory.  The phase of term h is exact: m_d = (h_d i_d) mod n_d in integers, exp(-2 pi i h.x) = prod_d
// conj(tab_d[m_d]).  Every thread sums its terms in reflection order, with no atomics: identical bits on every call.
__global__ void __launch_bounds__(FM_THREADS)
fourier_map_kernel(const int64_t* __restrict__ hkl, const double* __restrict__ coef, int64_t N, double F000,
                   double inv_volume, int n1, int n2, int n3, double* __restrict__ out) {
  extern __shared__ double sm[];
  double2* tab = reinterpret_cast<double2*>(sm);                    // [n1 + n2 + n3] (cos, sin)
  double2* sF = tab + (n1 + n2 + n3);                                // [FM_CHUNK] (Re F, Im F)
  int* sh = reinterpret_cast<int*>(sF + FM_CHUNK);                   // [FM_CHUNK][3] h_d mod n_d
  for (int t = threadIdx.x; t < n1 + n2 + n3; t += FM_THREADS) {
    const int n = t < n1 ? n1 : (t < n1 + n2 ? n2 : n3);
    const int m = t - (t < n1 ? 0 : (t < n1 + n2 ? n1 : n1 + n2));
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tab[t] = make_double2(c, s);
  }
  const int64_t npts = (int64_t)n1 * n2 * n3;
  const int64_t p = (int64_t)blockIdx.x * FM_THREADS + threadIdx.x;
  const int64_t pp = p < npts ? p : 0;
  const int i = (int)(pp / ((int64_t)n2 * n3)), j = (int)((pp / n3) % n2), k = (int)(pp % n3);
  const float inv1 = 1.0f / (float)n1, inv2 = 1.0f / (float)n2, inv3 = 1.0f / (float)n3;
  const double2* t1 = tab;
  const double2* t2 = tab + n1;
  const double2* t3 = tab + n1 + n2;
  double acc = 0.0;
  for (int64_t c0 = 0; c0 < N; c0 += FM_CHUNK) {
    const int nc = (int)(N - c0 < FM_CHUNK ? N - c0 : FM_CHUNK);
    __syncthreads();                                                 // the previous chunk has been read
    if (threadIdx.x < nc) {
      const int64_t r = c0 + threadIdx.x;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const int n = d == 0 ? n1 : (d == 1 ? n2 : n3);
        const int64_t h = hkl[3 * r + d] % n;
        sh[3 * threadIdx.x + d] = (int)(h < 0 ? h + n : h);
      }
      sF[threadIdx.x] = make_double2(coef[r], coef[N + r]);
    }
    __syncthreads();
    for (int c = 0; c < nc; ++c) {
      const double2 e1 = t1[mod_small(sh[3 * c] * i, n1, inv1)];
      const double2 e2 = t2[mod_small(sh[3 * c + 1] * j, n2, inv2)];
      const double2 e3 = t3[mod_small(sh[3 * c + 2] * k, n3, inv3)];
      // (cos, sin) of 2 pi h.x = e1 e2 e3; the term is Re F cos + Im F sin
      const double c12 = e1.x * e2.x - e1.y * e2.y, s12 = e1.x * e2.y + e1.y * e2.x;
      const double co = c12 * e3.x - s12 * e3.y, si = c12 * e3.y + s12 * e3.x;
      const double2 F = sF[c];
      acc += F.x * co + F.y * si;
    }
  }
  if (p < npts) out[p] = (F000 + 2.0 * acc) * inv_volume;
}

}  // namespace

int64_t density_grid_chunk(int64_t npts) { return npts < DG_CHUNK ? npts : DG_CHUNK; }

int64_t density_grid_workspace_elems(int nao, int64_t npts) {
  const int64_t c = density_grid_chunk(npts);
  return 2 * ((c * nao + 31) / 32 * 32);
}

cudaError_t launch_density_grid(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* dm,
                                const double* box, int n1, int n2, int n3, double* out, double* workspace,
                                cudaStream_t st) {
  const int64_t npts = (int64_t)n1 * n2 * n3;
  if (nao <= 0 || npts <= 0) return cudaSuccess;
  const int64_t chunk = density_grid_chunk(npts);
  double* phi = workspace;
  double* X = workspace + (chunk * nao + 31) / 32 * 32;
  for (int64_t p0 = 0; p0 < npts; p0 += chunk) {
    const int64_t np = npts - p0 < chunk ? npts - p0 : chunk;
    const int64_t nb = (np * nao + AO_THREADS - 1) / AO_THREADS;
    if (nb > 0x7fffffffLL) return cudaErrorInvalidValue;
    ao_values_kernel<<<(unsigned)nb, AO_THREADS, 0, st>>>(prim, nprim, ao_first, nao, box[0], box[1], box[2], box[3],
                                                          box[4], box[5], box[6], box[7], box[8], box[9], box[10],
                                                          box[11], n2, n3, p0, np, phi);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // X [np, nao] = Phi [np, nao] . D [nao, nao]
    GemmArgs g{};
    g.A = phi; g.B = dm; g.C = X; g.M = np; g.N = nao; g.K = nao; g.lda = nao; g.ldb = nao; g.ldc = nao;
    g.batch = 1; g.splitk = 1; g.kchunk = nao; g.ta = 0; g.tb = 0; g.alpha = 1.0; g.beta = 0.0;
    e = launch_gemm(g, st);
    if (e != cudaSuccess) return e;
    const int64_t rb = (np + RD_THREADS / 32 - 1) / (RD_THREADS / 32);
    rowdot_kernel<<<(unsigned)rb, RD_THREADS, 0, st>>>(X, phi, nao, np, out + p0);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

cudaError_t launch_fourier_map(const int64_t* hkl, const double* coef, int64_t N, double F000, double volume, int n1,
                               int n2, int n3, double* out, cudaStream_t st) {
  const int64_t npts = (int64_t)n1 * n2 * n3;
  if (npts <= 0) return cudaSuccess;
  if (n1 > FM_MAX_N || n2 > FM_MAX_N || n3 > FM_MAX_N || N < 0) return cudaErrorInvalidValue;
  const size_t smem = sizeof(double2) * (n1 + n2 + n3 + FM_CHUNK) + sizeof(int) * 3 * FM_CHUNK;
  const int64_t nb = (npts + FM_THREADS - 1) / FM_THREADS;
  if (nb > 0x7fffffffLL) return cudaErrorInvalidValue;
  fourier_map_kernel<<<(unsigned)nb, FM_THREADS, smem, st>>>(hkl, coef, N, F000, 1.0 / volume, n1, n2, n3, out);
  return cudaGetLastError();
}

}  // namespace ecw
