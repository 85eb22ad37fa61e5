// ftao.cu — structure-factor target of the ECW fit (sm_100a, FP64 throughout):
// Fourier-transformed AO pairs A_mu,nu(G) = int phi_mu phi_nu exp(+i G.r) d^3r over primitive Cartesian Gaussians, and
// the two small kernels of the per-iteration potential (ecw_vexp_sf; its GEMM/GEMV steps run on gemm.cu's kernels);
// for the amplitude target 'Fobs', the symmetrised, thermally smeared planes of a unit cell (ecw_ft_aopair_cryst) and the
// scale / coefficient kernel of its potential (ecw_vexp_sfobs).
//
// One primitive pair (exponents a, b, p = a + b, centre P, Hermite coefficients E_t^(d) of McMurchie-Davidson) gives
//   K exp(-|G|^2 / 4p) exp(i G.P) prod_d sum_t E_t^(d) (i G_d)^t,   K = c_a c_b exp(-a b |A-B|^2 / p) (pi/p)^(3/2).
// The references of these kernels are ecw_cc_b200.molint.ft_aopair and ft_aopair_cryst (same recurrence, same formula).
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
constexpr int FT_MAX_SYM = 192;    // general positions of the largest space groups (Fm-3m: 48 x 4 centrings)
constexpr double FOBS_ZERO = 1e-12;  // |F_calc| <= FOBS_ZERO max |F_calc| counts as zero (molint.FOBS_ZERO)

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

// G-independent data of one primitive pair from two rows {Ax, Ay, Az, alpha, coef, lx, ly, lz} of the primitive table;
// l outside [0, FT_LMAX] gives K = NaN
__device__ __forceinline__ FtPair stage_pair(const double* A, const double* B) {
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
  return r;
}

// (ar, ai) += the transform of one staged primitive pair at G = (gx, gy, gz), g2 = |G|^2
__device__ __forceinline__ void add_pair(const FtPair& r, double gx, double gy, double gz, double g2, double& ar,
                                         double& ai) {
  const double damp = r.K * exp(-g2 * r.q);
  double s, co;
  sincos(gx * r.P[0] + gy * r.P[1] + gz * r.P[2], &s, &co);
  // prod_d sum_t E_t (i g_d)^t, with (i g)^t = 1, i g, -g^2, -i g^3, g^4
  double pr = 1.0, pi = 0.0;
  const double gd[3] = {gx, gy, gz};
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double q2 = gd[d] * gd[d];
    const double xr = r.E[d][0] + q2 * (-r.E[d][2] + q2 * r.E[d][4]);
    const double xi = gd[d] * (r.E[d][1] - q2 * r.E[d][3]);
    const double nr = pr * xr - pi * xi;
    pi = pr * xi + pi * xr;
    pr = nr;
  }
  ar += damp * (pr * co - pi * s);
  ai += damp * (pr * s + pi * co);
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
      sp[threadIdx.x] = stage_pair(prim + 8 * (i0 + pp / nj), prim + 8 * (j0 + pp % nj));
    }
    __syncthreads();
    for (int c = 0; c < nc; ++c) {
#pragma unroll
      for (int u = 0; u < FT_GPT; ++u) add_pair(sp[c], gx[u], gy[u], gz[u], g2[u], ar[u], ai[u]);
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

// Symmetrised, smeared planes B(h) = sum_s exp(2 pi i h.t_s) T(G_hs) A(G_hs) of the 'Fobs' target.  The grid is that
// of ft_aopair_kernel (AO pair mu >= nu per blockIdx.x, FT_THREADS * FT_GPT reflections per blockIdx.y); the operations
// are the OUTER loop, so a thread holds the A accumulators of one operation at a time (no per-(h, s) registers for any
// nsym) and adds T * phase * A to its B sums in the fixed order s = 0, 1, ...  An AO pair whose primitive pairs fit one
// shared-memory chunk (every pair of the embedded bases) stages them once for all operations; a longer one restages
// its chunks per operation.  Gs [nG][nsym][3] holds G_hs (bohr^-1), phase [nG][nsym][2] (cos, sin) of 2 pi h.t_s, U
// [natom][6] the Cartesian ADP (xx, yy, zz, xy, xz, yz, bohr^2) and ao_atom [nao] the atom of each AO.
__global__ void __launch_bounds__(FT_THREADS)
ft_aopair_cryst_kernel(const double* __restrict__ prim, int64_t nprim, const int64_t* __restrict__ ao_first,
                       const int64_t* __restrict__ ao_atom, int nao, const double* __restrict__ U, int natom,
                       const double* __restrict__ Gs, const double* __restrict__ phase, int nsym, int64_t nG,
                       double* __restrict__ out) {
  __shared__ FtPair sp[FT_CHUNK];
  const int64_t k = blockIdx.x;
  int64_t mu = (int64_t)((sqrt(8.0 * (double)k + 1.0) - 1.0) * 0.5);
  while (mu * (mu + 1) / 2 > k) --mu;
  while ((mu + 1) * (mu + 2) / 2 <= k) ++mu;
  const int64_t nu = k - mu * (mu + 1) / 2;
  const int64_t i0 = ao_first[mu], ni = ao_first[mu + 1] - i0;
  const int64_t j0 = ao_first[nu], nj = ao_first[nu + 1] - j0;
  const int64_t am = ao_atom[mu], an = ao_atom[nu];
  // a malformed table (primitive range, atom index, l > FT_LMAX) poisons the element instead of reading out of bounds
  const bool bad = ni < 0 || nj < 0 || i0 < 0 || j0 < 0 || i0 + ni > nprim || j0 + nj > nprim || am < 0 || an < 0 ||
                   am >= natom || an >= natom;
  double ua[6], ub[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    ua[c] = bad ? 0.0 : U[6 * am + c];
    ub[c] = bad ? 0.0 : U[6 * an + c];
  }
  double br[FT_GPT], bi[FT_GPT];
#pragma unroll
  for (int u = 0; u < FT_GPT; ++u) br[u] = bi[u] = 0.0;
  const int64_t gbase = (int64_t)blockIdx.y * FT_THREADS * FT_GPT + threadIdx.x;
  const int64_t npp = bad ? 0 : ni * nj;
  const bool resident = npp <= FT_CHUNK;

  for (int s = 0; s < nsym; ++s) {
    double gx[FT_GPT], gy[FT_GPT], gz[FT_GPT], g2[FT_GPT], ar[FT_GPT], ai[FT_GPT];
#pragma unroll
    for (int u = 0; u < FT_GPT; ++u) {
      const int64_t g = gbase + (int64_t)u * FT_THREADS;
      gx[u] = gy[u] = gz[u] = 0.0;
      if (g < nG) {
        const double* q = Gs + 3 * (g * nsym + s);
        gx[u] = q[0]; gy[u] = q[1]; gz[u] = q[2];
      }
      g2[u] = gx[u] * gx[u] + gy[u] * gy[u] + gz[u] * gz[u];
      ar[u] = ai[u] = 0.0;
    }
    for (int64_t c0 = 0; c0 < npp; c0 += FT_CHUNK) {
      const int nc = (int)(npp - c0 < FT_CHUNK ? npp - c0 : FT_CHUNK);
      if (s == 0 || !resident) {
        __syncthreads();                                  // the previous chunk has been read by every thread
        if (threadIdx.x < nc) {
          const int64_t pp = c0 + threadIdx.x;
          sp[threadIdx.x] = stage_pair(prim + 8 * (i0 + pp / nj), prim + 8 * (j0 + pp % nj));
        }
        __syncthreads();
      }
      for (int c = 0; c < nc; ++c) {
#pragma unroll
        for (int u = 0; u < FT_GPT; ++u) add_pair(sp[c], gx[u], gy[u], gz[u], g2[u], ar[u], ai[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < FT_GPT; ++u) {
      const int64_t g = gbase + (int64_t)u * FT_THREADS;
      if (g >= nG) continue;
      const double xx = gx[u] * gx[u], yy = gy[u] * gy[u], zz = gz[u] * gz[u];
      const double xy = gx[u] * gy[u], xz = gx[u] * gz[u], yz = gy[u] * gz[u];
      const double qa = ua[0] * xx + ua[1] * yy + ua[2] * zz + 2.0 * (ua[3] * xy + ua[4] * xz + ua[5] * yz);
      const double qb = ub[0] * xx + ub[1] * yy + ub[2] * zz + 2.0 * (ub[3] * xy + ub[4] * xz + ub[5] * yz);
      const double T = 0.5 * (exp(-0.5 * qa) + exp(-0.5 * qb));
      const double co = phase[2 * (g * nsym + s)], sn = phase[2 * (g * nsym + s) + 1];
      br[u] += T * (ar[u] * co - ai[u] * sn);
      bi[u] += T * (ar[u] * sn + ai[u] * co);
    }
  }
  if (bad) {
#pragma unroll
    for (int u = 0; u < FT_GPT; ++u) br[u] = bi[u] = nan("");
  }
  const int64_t n2 = (int64_t)nao * nao;
#pragma unroll
  for (int u = 0; u < FT_GPT; ++u) {
    const int64_t g = gbase + (int64_t)u * FT_THREADS;
    if (g >= nG) continue;
    double* re = out + g * n2;
    double* im = out + (nG + g) * n2;
    re[mu * nao + nu] = br[u];
    im[mu * nao + nu] = bi[u];
    re[nu * nao + mu] = br[u];
    im[nu * nao + mu] = bi[u];
  }
}

// Amplitude target: a_h = |F_calc(h)|, w_h = 1/sigma_h^2.  Pass 1: a_max = max a and, for a refined scale, k = sum w
// |Fo| a / sum w a^2.  Pass 2: coef [2][nG] = [Re c | Im c], c_h = 2 L k / (nG - Np) w_h (|Fo| - k a_h) F_calc / a_h,
// the coefficients of the same transposed GEMV as sf_coef_kernel's.  An amplitude a_h <= FOBS_ZERO a_max counts as zero
// (c_h = 0): |F| has a cusp there, and F_calc / a_h would be the direction of rounding noise (a reflection that a point
// symmetry of the density extinguishes).  stats[0] = sum |k a - |Fo||, stats[2] = k, stats[3] = chi^2 = sum w (k a -
// |Fo|)^2 / (nG - Np).  k_fixed > 0 fixes the scale (Np = 0), else it is refined (Np = 1).  One block, fixed reduction
// order.
__global__ void __launch_bounds__(SF_THREADS)
sfobs_coef_kernel(const double* __restrict__ F_obs, const double* __restrict__ w, const double* __restrict__ F_calc,
                  double L, double k_fixed, double* __restrict__ coef, double* __restrict__ stats, int64_t nG) {
  __shared__ double s1[SF_THREADS], s2[SF_THREADS], s3[SF_THREADS];
  const bool refine = !(k_fixed > 0.0);
  double a = 0.0, b = 0.0, m = 0.0;
  for (int64_t h = threadIdx.x; h < nG; h += SF_THREADS) {
    const double fc = hypot(F_calc[h], F_calc[nG + h]);
    m = fmax(m, fc);
    if (refine) {
      a += w[h] * F_obs[h] * fc;
      b += w[h] * fc * fc;
    }
  }
  s1[threadIdx.x] = a;
  s2[threadIdx.x] = b;
  s3[threadIdx.x] = m;
  __syncthreads();
  for (int r = SF_THREADS / 2; r > 0; r >>= 1) {
    if (threadIdx.x < r) {
      s1[threadIdx.x] += s1[threadIdx.x + r];
      s2[threadIdx.x] += s2[threadIdx.x + r];
      s3[threadIdx.x] = fmax(s3[threadIdx.x], s3[threadIdx.x + r]);
    }
    __syncthreads();
  }
  const double k = refine ? s1[0] / s2[0] : k_fixed;
  const double zero = FOBS_ZERO * s3[0];
  const double dof = (double)nG - (refine ? 1.0 : 0.0);
  const double f = 2.0 * L * k / dof;
  __syncthreads();                                        // s1 / s2 are reused below
  double r1 = 0.0, chi = 0.0;
  for (int64_t h = threadIdx.x; h < nG; h += SF_THREADS) {
    const double re = F_calc[h], im = F_calc[nG + h];
    const double fc = hypot(re, im);
    const double r = F_obs[h] - k * fc;
    chi += w[h] * r * r;
    r1 += fabs(k * fc - F_obs[h]);
    const double c = fc > zero ? f * w[h] * r / fc : 0.0;
    coef[h] = c * re;
    coef[nG + h] = c * im;
  }
  s1[threadIdx.x] = r1;
  s2[threadIdx.x] = chi;
  __syncthreads();
  for (int r = SF_THREADS / 2; r > 0; r >>= 1) {
    if (threadIdx.x < r) {
      s1[threadIdx.x] += s1[threadIdx.x + r];
      s2[threadIdx.x] += s2[threadIdx.x + r];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    stats[0] = s1[0];
    stats[2] = k;
    stats[3] = s2[0] / dof;
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

cudaError_t launch_ft_aopair_cryst(const double* prim, int64_t nprim, const int64_t* ao_first, const int64_t* ao_atom,
                                   int nao, const double* U, int natom, const double* Gs, const double* phase, int nsym,
                                   int64_t nG, double* out, cudaStream_t st) {
  if (nao <= 0 || nG <= 0) return cudaSuccess;
  const int64_t npairs = (int64_t)nao * (nao + 1) / 2;
  const int64_t gblocks = (nG + FT_THREADS * FT_GPT - 1) / (FT_THREADS * FT_GPT);
  if (npairs > 0x7fffffffLL || gblocks > 65535 || nsym < 1 || nsym > FT_MAX_SYM || natom < 1)
    return cudaErrorInvalidValue;
  dim3 grid((unsigned)npairs, (unsigned)gblocks, 1);
  ft_aopair_cryst_kernel<<<grid, FT_THREADS, 0, st>>>(prim, nprim, ao_first, ao_atom, nao, U, natom, Gs, phase, nsym,
                                                       nG, out);
  return cudaGetLastError();
}

cudaError_t launch_sfobs_coef(const double* F_obs, const double* w, const double* F_calc, double L, double k_fixed,
                              double* coef, double* stats, int64_t nG, cudaStream_t st) {
  if (nG <= 0) return cudaSuccess;
  sfobs_coef_kernel<<<1, SF_THREADS, 0, st>>>(F_obs, w, F_calc, L, k_fixed, coef, stats, nG);
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
