// kernels.h — launchers of the hand-written sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "ozaki_layout.h"

namespace ecw {

struct GemmArgs {
  const double* A;
  const double* B;
  double* C;
  int64_t M, N, K, lda, ldb, ldc, sA, sB, sC, batch, splitk, kchunk;
  int ta, tb;
  double alpha, beta;
  int vecA, vecB, vecC;   // filled by launch_gemm (16-byte cp.async / double2 stores allowed)
};

int gemm_pick_config(int64_t M, int64_t N, int64_t K = 0);
// CTA tile the automatic choice uses for this problem (the plan sizes its split-K by the real tile count)
void gemm_tile_of(int64_t M, int64_t N, int64_t K, int* bm, int* bn);
cudaError_t launch_gemm(const GemmArgs& a, cudaStream_t st, int force_cfg = -1);
// warp-specialised TMA + mbarrier variant (gemm_tma.cu); cfg 20: 128x128, 21: 112x128
bool gemm_tma_eligible(const GemmArgs& a);
cudaError_t launch_gemm_tma(const GemmArgs& a, cudaStream_t st, int cfg);

// FP64 GEMM by error-free splitting on the INT8 tcgen05 tensor pipe (ozaki.cu).
// An operand X[R,K] (element (r,k) at X[r*rs + k*ks], one of rs/ks == 1) is cut into `ns` int8 digit
// planes (ozaki_plane_bytes) plus row statistics `scale` = [2^e scales | row sums / scale], each
// ozaki_padded_rows doubles long (sizes: ozaki_layout.h).
// row0/total_rows: X holds rows [row0, row0+R) of an operand of total_rows rows whose plane set is cut chunk
// by chunk (row0 a multiple of 128; every chunk but the last a multiple of 128 rows)
cudaError_t launch_ozaki_split(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, int8_t* planes,
                               double* scale, cudaStream_t st, int64_t row0 = 0, int64_t total_rows = 0);
// two-level contraction index k = (k1, k2), element at X[r*rs + k1*ks1 + k2*ks2] (rs == 1 or ks2 == 1); k2 is padded
// to a multiple of 32 per k1 (k-block index k1*ceil(K2/32) + k2/32), and the statistics also hold the row sums per k1:
// stats = [scales | row sums | row sums of k1 = 0 | ... ] (ozaki_stat_elems doubles).  A contiguous range of k1
// values of such a plane set is itself a valid operand (OzBatch::*_kb0/_kbb/_t0/_tb).
cudaError_t launch_ozaki_split2(const double* X, int64_t R, int64_t K1, int64_t K2, int64_t rs, int64_t ks1, int64_t ks2,
                                int ns, int8_t* planes, double* stats, cudaStream_t st, int64_t row0 = 0,
                                int64_t total_rows = 0);
// C[m*crs + n*ccs] = alpha * sum_k A[m,k] B[n,k] + beta * C  from the digit planes of A (M rows) and B (N rows)
cudaError_t launch_ozaki_gemm(const int8_t* pa, const double* sa, const int8_t* pb, const double* sb, int64_t M, int64_t N,
                              int64_t K, double* C, int64_t crs, int64_t ccs, double alpha, double beta, int ns,
                              cudaStream_t st, int sm_count);
// batch of independent products b = 0..batch-1 over sub-blocks of two plane sets:
//   rows   [x_row0 + b*x_rowb, +M or +N)   (multiples of 8) of the set,
//   k-blocks [x_kb0 + b*x_kbb, + nkb)  (nkb = 0: ceil(K/32); a two-level index has nk1*ceil(K2/32)),
//   row sums at stats[x_t0 + b*x_tb + row]  (x_t0 = padded rows of the set: whole-K sums; (2+k1)*padded: per-k1 sums),
//   C_b = C + b*c_b.
struct OzBatch {
  int64_t batch;
  int64_t a_row0, a_rowb, b_row0, b_rowb;
  int64_t a_kb0, a_kbb, b_kb0, b_kbb;
  int64_t a_t0, a_tb, b_t0, b_tb;
  int64_t c_b;
  int64_t nkb;
};
// a_rows / b_rows: total rows of the two plane sets (their slab size)
cudaError_t launch_ozaki_gemm_batched(const int8_t* pa, const double* sa, int64_t a_rows, const int8_t* pb,
                                      const double* sb, int64_t b_rows, int64_t M, int64_t N, int64_t K, double* C,
                                      int64_t crs, int64_t ccs, double alpha, double beta, int ns, const OzBatch& bt,
                                      cudaStream_t st, int sm_count);

// *out = max(*out, (ns+3) 256^-ns K |alpha| max s_m max s_n): worst-case absolute error of the product(s) above,
// from the row scales actually present (a NaN scale, i.e. a non-finite operand row, yields NaN)
cudaError_t launch_ozaki_bound(const double* sa, const double* sb, int64_t M, int64_t N, int64_t K, double alpha, int ns,
                               const OzBatch& bt, double* out, cudaStream_t st);

constexpr int KMAXD = 6;
struct PermArgs {
  const double* in;
  double* out;
  int nd;
  int64_t dim[KMAXD], sin[KMAXD], sout[KMAXD];
  double alpha, beta;
};
cudaError_t launch_permute(const PermArgs& a, cudaStream_t st);

cudaError_t launch_fill(double* c, int64_t n, double value, cudaStream_t st);
// strided element-wise: out = alpha * a * b + beta * out  (b == nullptr: alpha*a; a == nullptr: fill alpha)
struct Ew2Args {
  const double* a;
  const double* b;
  double* out;
  int nd;
  int64_t dim[KMAXD], sa[KMAXD], sb[KMAXD], so[KMAXD];
  double alpha, beta;
};
cudaError_t launch_ew2(const Ew2Args& a, cudaStream_t st);
// partial[z][M*N] -> C[m*sr + n*sc] = alpha*sum + beta*C
cudaError_t launch_reduce(const double* part, int64_t nz, int64_t M, int64_t N, double* C, int64_t sr,
                          int64_t sc, double alpha, double beta, cudaStream_t st);
// out[ijab] = t2[ijab] + c1*t1[ia]t1[jb] - c2*t1[ib]t1[ja]
// i0 / ni: t2 and out hold only the rows i0 .. i0+ni-1 of the leading occupied index (ni < 0: all from i0)
cudaError_t launch_tau(const double* t2, const double* t1, double* out, int o, int v, double c1, double c2,
                       cudaStream_t st, int i0 = 0, int ni = -1);
// out[ijab] = c0 base[ijab] + z[ijab] - z[jiab] - z[ijba] + z[jiba] + beta out[ijab]  (base may be null)
cudaError_t launch_asym4(const double* base, double c0, const double* z, double* out, double beta, int o, int v,
                         cudaStream_t st);
// out[0] = max(|x[ijab]+x[jiab]|, |x[ijab]+x[ijba]|)  (0 for exactly antisymmetric doubles amplitudes), out[1] = max|x|
cudaError_t launch_antisym_defect(const double* x, int o, int v, double* out, cudaStream_t st);

struct PackArgs {
  const double* src;   // 4-index view (pack) / matrix (unpack)
  double* dst;
  int64_t d0, d1, d2, d3;          // dims of the 4-index side
  int64_t s0, s1, s2, s3;          // strides of the 4-index side
  int64_t ld;                      // leading dim of the matrix side
  int flags;
  double alpha, beta;
};
cudaError_t launch_pack(const PackArgs& a, cudaStream_t st);
cudaError_t launch_unpack(const PackArgs& a, cudaStream_t st);

// residual -> update (CCSD.py:316-338); fock is the bare n x n Fock matrix
// shift is added to every denominator (EOM-like updates divide by Em + e_i - e_a, CCS.py:938);
// sub_singles applies the soft threshold to rank-2 amplitudes too (CCS.py:377, 610)
cudaError_t launch_finish(const double* r, const double* amp, const double* fock, int64_t ldf, double* out,
                          int o, int v, int rank, int has_alpha, int equation, double alpha, double shift,
                          int sub_singles, cudaStream_t st);
cudaError_t launch_subdiff(const double* e, const double* v, double alpha, double* out, int64_t n, cudaStream_t st);
// conv = |a| + |b| (b null: a); scal = beta*scal + sum (conv - prev)^2 (prev null: + 0); partial: nblocks doubles
cudaError_t launch_vexp_mat(const double* rdm1, const double* target, const double* fock, double L, double* vexp,
                            double* fsp, double* stats, int64_t n, cudaStream_t st);
// structure-factor target (ftao.cu).  prim [nprim, 8] = {Ax, Ay, Az, alpha, coef, lx, ly, lz} per primitive Cartesian
// Gaussian (l <= 2 per direction), the primitives of AO mu at rows ao_first[mu] .. ao_first[mu+1]-1; G [nG, 3] in
// bohr^-1; out [2][nG][nao][nao] = Re and Im planes of int phi_mu phi_nu exp(+i G.r)
cudaError_t launch_ft_aopair(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* G,
                             int64_t nG, double* out, cudaStream_t st);
// coef [2][nG] = L (F_exp - F_calc) (Re, Im planes), stats[0] = sum_h |F_exp(h) - F_calc(h)|
cudaError_t launch_sf_coef(const double* F_exp, const double* F_calc, double L, double* coef, double* stats, int64_t nG,
                           cudaStream_t st);
// amplitude ('Fobs') target.  Symmetrised, smeared planes B(h) = sum_s exp(2 pi i h.t_s) T(G_hs) A(G_hs), out as for
// launch_ft_aopair; ao_atom [nao] (int64), U [natom][6] = Cartesian ADP (xx, yy, zz, xy, xz, yz) in bohr^2, Gs
// [nG][nsym][3] = G_{R_s^T h} in bohr^-1, phase [nG][nsym][2] = (cos, sin) of 2 pi h.t_s; 1 <= nsym <= 192
cudaError_t launch_ft_aopair_cryst(const double* prim, int64_t nprim, const int64_t* ao_first, const int64_t* ao_atom,
                                   int nao, const double* U, int natom, const double* Gs, const double* phase, int nsym,
                                   int64_t nG, double* out, cudaStream_t st);
// scale k (k_fixed > 0: fixed, else refined), coef [2][nG] of the amplitude potential, stats[0] = sum |k|Fc| - Fo|,
// stats[2] = k, stats[3] = chi^2 (w = 1/sigma^2 per reflection)
cudaError_t launch_sfobs_coef(const double* F_obs, const double* w, const double* F_calc, double L, double k_fixed,
                              double* coef, double* stats, int64_t nG, cudaStream_t st);
// fsp = fock - vexp, stats[1] = max |vexp|
cudaError_t launch_sf_finish(const double* vexp, const double* fock, double* fsp, double* stats, int64_t n2,
                             cudaStream_t st);
// density maps (maps.cu).  rho on the box grid r_ijk = origin + i a1 + j a2 + k a3, box[12] (host) = origin, a1, a2, a3
// in bohr, out [n1][n2][n3] (k fastest); dm [nao][nao] is the AO density (need not be symmetric), prim / ao_first as for
// launch_ft_aopair.  Points go in chunks of DG_CHUNK: Phi [chunk][nao] by ao_values_kernel, X = Phi D by launch_gemm,
// rho_p = sum_mu X_p,mu Phi_p,mu; workspace: density_grid_workspace_elems(nao, npts) doubles (Phi and X)
constexpr int64_t DG_CHUNK = 32768;
int64_t density_grid_chunk(int64_t npts);
int64_t density_grid_workspace_elems(int nao, int64_t npts);
cudaError_t launch_density_grid(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* dm,
                                const double* box, int n1, int n2, int n3, double* out, double* workspace,
                                cudaStream_t st);
// rho(x_ijk) = (F000 + 2 sum_h (Re F_h cos 2 pi h.x + Im F_h sin 2 pi h.x)) / volume at x_ijk = (i/n1, j/n2, k/n3) for
// the half set hkl [N][3] (int64), coef [2][N] (Re, Im); out [n1][n2][n3]; 1 <= n_d <= FM_MAX_N
constexpr int FM_MAX_N = 512;
cudaError_t launch_fourier_map(const int64_t* hkl, const double* coef, int64_t N, double F000, double volume, int n1,
                               int n2, int n3, double* out, cudaStream_t st);
cudaError_t launch_conv(const double* a, const double* b, const double* prev, double* conv, int64_t n, double* partial,
                        int nblocks, double* scal, double beta, cudaStream_t st);
cudaError_t launch_dot(const double* a, const double* b, int64_t n, double* partial, int nblocks, double* scal,
                       double alpha, double beta, cudaStream_t st);
cudaError_t launch_scale_dev(double* c, int64_t n, const double* scal, double d0, double d1, cudaStream_t st);
cudaError_t launch_diag_add(double* c, int64_t ldc, int64_t m, const double* fock, int64_t ldf, int64_t foff,
                            double alpha, cudaStream_t st);
cudaError_t launch_rdm1(const double* doo, const double* dvoT, const double* l1, const double* dvv, double* out,
                        int o, int v, cudaStream_t st);

// synthetic, function-defined inputs (DESIGN.md "Synthetic inputs"); kind selects the tensor
enum SynthKind : int {
  SY_OOOO = 0, SY_OOOV, SY_OOVV, SY_OOVV_PH, SY_OVOV_PH, SY_OVVV, SY_OOOO_P, SY_OOVV_P, SY_OVVV_P, SY_VVVV_P,
  SY_FOCK, SY_FSP, SY_T1, SY_L1, SY_T2, SY_L2
};
// row0/nrows restrict generation to a leading-index range (shards of vvvv_p / ovvv)
cudaError_t launch_synth(int kind, double* out, int o, int v, int64_t row0, int64_t nrows, double scale,
                         cudaStream_t st);
// constant layouts derived from dense canonical blocks
cudaError_t launch_eris_layouts_from_dense(const double* oovv, const double* ovov, double* oovv_ph, double* ovov_ph,
                                           int o, int v, cudaStream_t st);

}  // namespace ecw
