// ftao.cu — structure-factor target of the ECW fit (sm_100a, FP64 throughout):
// Fourier-transformed AO pairs A_mu,nu(G) = int phi_mu phi_nu exp(+i G.r) d^3r over primitive Cartesian Gaussians, and
// the two small kernels of the per-iteration potential (ecw_vexp_sf; its GEMM/GEMV steps run on gemm.cu's kernels).
//
// One primitive pair (exponents a, b, p = a + b, centre P, Hermite coefficients E_t^(d) of McMurchie-Davidson) gives
//   K exp(-|G|^2 / 4p) exp(i G.P) prod_d sum_t E_t^(d) (i G_d)^t,   K = c_a c_b exp(-a b |A-B|^2 / p) (pi/p)^(3/2).
// The reference of this kernel is ecw_cc_b200.molint.ft_aopair (same recurrence, same formula).
#include "kernels.h"

#include <algorithm>
#include <cmath>

namespace ecw {

namespace {

constexpr int FT_THREADS = 128;
constexpr int FT_GPT = 4;          // G vectors per thread: independent accumulators for every staged pair
constexpr int FT_CHUNK = 64;       // primitive pairs staged in shared memory per pass (cc-pVDZ s AOs: 8 primitives)
constexpr int FT_LMAX = 2;         // per-direction angular momentum of one primitive (s, p, d)
constexpr int FT_T = 2 * FT_LMAX + 1;
constexpr int SF_THREADS = 256;

// G-independent data of one primitive pair
struct FtPair {
  double K, q, P[3];               // q = 1 / 4p
  double E[3][FT_T];               // E_t^(d), zero beyond la_d + lb_d
};

// E^{i,j}_t -> E^{i+1,j}_t or E^{i,j+1}_t (X = X_PA or X_PB), the recurrence of molint._hermite_E
__device__ __forceinline__ void hermite_step(double (&c)[FT_T], double X, double two_p) {
  double n[FT_T];
#pragma unroll
  for (int t = 0; t < FT_T; ++t)
    n[t] = (t > 0 ? c[t - 1] / two_p : 0.0) + X * c[t] + (t + 1 < FT_T ? (t + 1) * c[t + 1] : 0.0);
#pragma unroll
  for (int t = 0; t < FT_T; ++t) c[t] = n[t];
}

// One block: the AO pair (mu >= nu) of blockIdx.x and FT_THREADS * FT_GPT scattering vectors from blockIdx.y.  The
// block stages the pair data of up to FT_CHUNK primitive pairs at a time and every thread adds them, in the fixed
// (i, j) order, to its own G vectors: no atomics, so the result is the same bit for bit on every call.  The (mu, nu)
// and (nu, mu) elements of both planes are written from the same sums.
__global__ void __launch_bounds__(FT_THREADS)
ft_aopair_kernel(const double* __restrict__ prim, int64_t nprim, const int64_t* __restrict__ ao_first, int nao,
                 const double* __restrict__ G, int64_t nG, double* __restrict__ out) {
  __shared__ FtPair sp[FT_CHUNK];
  const int64_t k = blockIdx.x;
  int64_t mu = (int64_t)((sqrt(8.0 * (double)k + 1.0) - 1.0) * 0.5);
  while (mu * (mu + 1) / 2 > k) --mu;
  while ((mu + 1) * (mu + 2) / 2 <= k) ++mu;
  const int64_t nu = k - mu * (mu + 1) / 2;
  const int64_t i0 = ao_first[mu], ni = ao_first[mu + 1] - i0;
  const int64_t j0 = ao_first[nu], nj = ao_first[nu + 1] - j0;
  // a malformed table (range outside [0, nprim) or l > FT_LMAX) poisons the element instead of reading out of bounds
  bool bad = ni < 0 || nj < 0 || i0 < 0 || j0 < 0 || i0 + ni > nprim || j0 + nj > nprim;

  double gx[FT_GPT], gy[FT_GPT], gz[FT_GPT], g2[FT_GPT], ar[FT_GPT], ai[FT_GPT];
  const int64_t gbase = (int64_t)blockIdx.y * FT_THREADS * FT_GPT + threadIdx.x;
#pragma unroll
  for (int u = 0; u < FT_GPT; ++u) {
    const int64_t g = gbase + (int64_t)u * FT_THREADS;
    gx[u] = gy[u] = gz[u] = 0.0;
    if (g < nG) { gx[u] = G[3 * g]; gy[u] = G[3 * g + 1]; gz[u] = G[3 * g + 2]; }
    g2[u] = gx[u] * gx[u] + gy[u] * gy[u] + gz[u] * gz[u];
    ar[u] = ai[u] = 0.0;
  }

  const int64_t npp = bad ? 0 : ni * nj;
  for (int64_t c0 = 0; c0 < npp; c0 += FT_CHUNK) {
    const int nc = (int)(npp - c0 < FT_CHUNK ? npp - c0 : FT_CHUNK);
    if (threadIdx.x < nc) {
      const int64_t pp = c0 + threadIdx.x;
      const double* A = prim + 8 * (i0 + pp / nj);
      const double* B = prim + 8 * (j0 + pp % nj);
      const double a = A[3], b = B[3], p = a + b, two_p = 2.0 * p;
      FtPair r;
      double r2 = 0.0;
      bool lbad = false;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const double P = (a * A[d] + b * B[d]) / p;
        const double ab = A[d] - B[d];
        r2 += ab * ab;
        r.P[d] = P;
        const int la = (int)A[5 + d], lb = (int)B[5 + d];
        lbad |= la < 0 || lb < 0 || la > FT_LMAX || lb > FT_LMAX;
        double e[FT_T];
#pragma unroll
        for (int t = 0; t < FT_T; ++t) e[t] = t == 0 ? 1.0 : 0.0;
        for (int j = 0; j < lb && j < FT_LMAX; ++j) hermite_step(e, P - B[d], two_p);
        for (int i = 0; i < la && i < FT_LMAX; ++i) hermite_step(e, P - A[d], two_p);
#pragma unroll
        for (int t = 0; t < FT_T; ++t) r.E[d][t] = e[t];
      }
      r.K = lbad ? nan("") : A[4] * B[4] * exp(-a * b / p * r2) * pow(3.141592653589793 / p, 1.5);
      r.q = 0.25 / p;
      sp[threadIdx.x] = r;
    }
    __syncthreads();
    for (int c = 0; c < nc; ++c) {
      const FtPair& r = sp[c];
#pragma unroll
      for (int u = 0; u < FT_GPT; ++u) {
        const double damp = r.K * exp(-g2[u] * r.q);
        double s, co;
        sincos(gx[u] * r.P[0] + gy[u] * r.P[1] + gz[u] * r.P[2], &s, &co);
        // prod_d sum_t E_t (i g_d)^t, with (i g)^t = 1, i g, -g^2, -i g^3, g^4
        double pr = 1.0, pi = 0.0;
        const double gd[3] = {gx[u], gy[u], gz[u]};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const double q2 = gd[d] * gd[d];
          const double xr = r.E[d][0] + q2 * (-r.E[d][2] + q2 * r.E[d][4]);
          const double xi = gd[d] * (r.E[d][1] - q2 * r.E[d][3]);
          const double nr = pr * xr - pi * xi;
          pi = pr * xi + pi * xr;
          pr = nr;
        }
        ar[u] += damp * (pr * co - pi * s);
        ai[u] += damp * (pr * s + pi * co);
      }
    }
    __syncthreads();
  }
  if (bad) {
#pragma unroll
    for (int u = 0; u < FT_GPT; ++u) ar[u] = ai[u] = nan("");
  }
  const int64_t n2 = (int64_t)nao * nao;
#pragma unroll
  for (int u = 0; u < FT_GPT; ++u) {
    const int64_t g = gbase + (int64_t)u * FT_THREADS;
    if (g >= nG) continue;
    double* re = out + g * n2;
    double* im = out + (nG + g) * n2;
    re[mu * nao + nu] = ar[u];
    im[mu * nao + nu] = ai[u];
    re[nu * nao + mu] = ar[u];
    im[nu * nao + mu] = ai[u];
  }
}

// coef = L [Re dF | Im dF], dF = F_exp - F_calc: Re[conj(dF) A] = Re dF Re A + Im dF Im A, so the AO potential is the
// transposed GEMV of the two planes with this vector.  stats[0] = sum_h |dF_h|.  nG is 10^3-10^4: one block, fixed
// reduction order.
__global__ void __launch_bounds__(SF_THREADS)
sf_coef_kernel(const double* __restrict__ F_exp, const double* __restrict__ F_calc, double L, double* __restrict__ coef,
               double* __restrict__ stats, int64_t nG) {
  __shared__ double sh[SF_THREADS];
  double s = 0.0;
  for (int64_t h = threadIdx.x; h < nG; h += SF_THREADS) {
    const double dr = F_exp[h] - F_calc[h], di = F_exp[nG + h] - F_calc[nG + h];
    coef[h] = L * dr;
    coef[nG + h] = L * di;
    s += hypot(dr, di);
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = SF_THREADS / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) stats[0] = sh[0];
}

// fsp = fock - vexp, stats[1] = max |vexp|  (n x n: one block)
__global__ void __launch_bounds__(SF_THREADS)
sf_finish_kernel(const double* __restrict__ vexp, const double* __restrict__ fock, double* __restrict__ fsp,
                 double* __restrict__ stats, int64_t n2) {
  __shared__ double sh[SF_THREADS];
  double m = 0.0;
  for (int64_t i = threadIdx.x; i < n2; i += SF_THREADS) {
    fsp[i] = fock[i] - vexp[i];
    m = fmax(m, fabs(vexp[i]));
  }
  sh[threadIdx.x] = m;
  __syncthreads();
  for (int w = SF_THREADS / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + w]);
    __syncthreads();
  }
  if (threadIdx.x == 0) stats[1] = sh[0];
}

}  // namespace

cudaError_t launch_ft_aopair(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* G,
                             int64_t nG, double* out, cudaStream_t st) {
  if (nao <= 0 || nG <= 0) return cudaSuccess;
  const int64_t npairs = (int64_t)nao * (nao + 1) / 2;
  const int64_t gblocks = (nG + FT_THREADS * FT_GPT - 1) / (FT_THREADS * FT_GPT);
  if (npairs > 0x7fffffffLL || gblocks > 65535) return cudaErrorInvalidValue;
  dim3 grid((unsigned)npairs, (unsigned)gblocks, 1);
  ft_aopair_kernel<<<grid, FT_THREADS, 0, st>>>(prim, nprim, ao_first, nao, G, nG, out);
  return cudaGetLastError();
}

cudaError_t launch_sf_coef(const double* F_exp, const double* F_calc, double L, double* coef, double* stats, int64_t nG,
                           cudaStream_t st) {
  if (nG <= 0) return cudaSuccess;
  sf_coef_kernel<<<1, SF_THREADS, 0, st>>>(F_exp, F_calc, L, coef, stats, nG);
  return cudaGetLastError();
}

cudaError_t launch_sf_finish(const double* vexp, const double* fock, double* fsp, double* stats, int64_t n2,
                             cudaStream_t st) {
  if (n2 <= 0) return cudaSuccess;
  sf_finish_kernel<<<1, SF_THREADS, 0, st>>>(vexp, fock, fsp, stats, n2);
  return cudaGetLastError();
}

}  // namespace ecw
