/* ecw_b200.h — C ABI of the B200-native coupled-cluster residual path.
 *
 * Drop-in boundary for the hot path of MilaimKas/ECW_CC.  The reference has no
 * FFI of its own (it is pure Python/numpy); the boundary is the method surface
 * of `CCSD.GCC` / `CCS.Gccs` that the unchanged solver loops call
 * (Solver_GS.py:683-705, Solver_GS.py:172-204, Solver_ES.py:258-368).  Each
 * entry point below replaces one of those methods and cites it; the Python
 * classes in ecw_cc_b200/CCSD.py and ecw_cc_b200/CCS.py bind them with ctypes
 * (see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to FP64 data in C (row-major) order
 *     unless a parameter says "host";
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered,
 *     nothing synchronises the device;
 *   - return value 0 = ok, negative = error (message: ecw_last_error), 1 = collective pending
 *     (multi-GPU contexts only, see ecw_ctx_set_shard);
 *   - the library never allocates device memory: the caller binds the constant
 *     integral layouts and one workspace (sizes: ecw_slot_elems,
 *     ecw_workspace_bytes);
 *   - there is no CPU path: without a CUDA device every compute call fails.
 */
#ifndef ECW_B200_H
#define ECW_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ecw_ctx ecw_ctx;

/* mode flags of tupdate/lupdate: mirror `alpha is not None` / `equation=True`
 * of GCC.tupdate (CCSD.py:248) and GCC.lupdate (CCSD.py:419). */
#define ECW_HAS_ALPHA 1
#define ECW_EQUATION 2
/* ECW_ANTISYM: the caller guarantees t2 (and l2) are antisymmetric in (i,j) and (a,b)
 * (check with ecw_antisym_defect).  Then the ladders also pack the (i,j) rows.  Without
 * it only the antisymmetry of the integrals is used — required after an L1-regularised
 * update, which breaks amplitude antisymmetry in the reference (utilities.py:59-67). */
#define ECW_ANTISYM 4

/* ---- context ------------------------------------------------------------ */
/* One context per (device, nocc, nvir); replaces `GCC.__init__` (CCSD.py:186-198)
 * and `Gccs.__init__`. Touches no CUDA API. */
int ecw_ctx_create(ecw_ctx** out, int nocc, int nvir);
void ecw_ctx_destroy(ecw_ctx* ctx);
const char* ecw_last_error(ecw_ctx* ctx);
const char* ecw_version(void);
/* Multi-GPU (one process per GPU): rank r of `world` keeps rows [r*ceil(P_v/world), ...) of "vvvv_p"
 * (the packed virtual pair index) and computes its share of the heavy contractions.  Calls then
 * return 1 whenever a collective is due: the host reads it with ecw_pending_collective
 * (desc = {kind 1=all-gather | 2=all-to-all, send offset, elements per rank / per block, recv offset, world, rank}; offsets
 * are FP64-element offsets into the workspace), performs it (torch.distributed / NCCL) and calls
 * ecw_resume until it returns 0. */
int ecw_ctx_set_shard(ecw_ctx* ctx, int rank, int world);
int ecw_resume(ecw_ctx* ctx, void* stream);
/* The context's own NCCL communicator (SURVEY 8(b)).  The library resolves NCCL at run time (dlopen of `libpath`, or of
 * the libnccl.so.2 the process already has); rank 0 makes the 128-byte unique id with ecw_nccl_unique_id, the host
 * hands it to every rank (any channel: the Python side broadcasts it with torch.distributed), and each rank calls
 * ecw_ctx_init_nccl after ecw_ctx_set_shard.  From then on the collectives of a call (all-gathers of slab results,
 * the all-to-all of Wovvo, the rank sums) are enqueued by the executor itself on the caller's stream — calls never
 * return 1, nothing round-trips through the host.  Without it the yield protocol above stays in force (used by the
 * single-GPU "virtual ranks" tests). */
int ecw_nccl_unique_id(const char* libpath, void* id128);
int ecw_ctx_init_nccl(ecw_ctx* ctx, const char* libpath, const void* id128, int rank, int world);
int64_t ecw_ctx_nccl_ops(ecw_ctx* ctx);   /* collectives enqueued by the executor so far */
/* GEMM engine.  int8_digits = 0: every contraction runs on the FP64 DMMA kernels.  int8_digits = 3..8:
 * unbatched GEMMs with 2MNK >= min_flops for which the time model of the engine prefers it (min_flops = -1: all of
 * them; min_flops = -t < -1.5: those with 2MNK >= t, no time model — tests) run on the INT8 tcgen05 tensor pipe by
 * splitting the operands into that many base-256 int8 digits (csrc/ozaki.cu; 6 digits = 48 bits,
 * |err| <= 2^-42.8 K max|A_row| max|B_row| worst case, the size of an FP64 dot product's own rounding error).  Replaces the BLAS dgemm behind numpy/pyscf einsum
 * (CCSD.py:25).  A context starts with int8_digits = 0. */
int ecw_ctx_set_gemm(ecw_ctx* ctx, int int8_digits, double min_flops);
int ecw_ctx_get_gemm(ecw_ctx* ctx);
/* Run-time accuracy guard of the INT8 route.  Every INT8 product of a call adds (max) its worst-case absolute error
 *   (int8_digits + 3) 256^-int8_digits K |alpha| max_m s_m max_n s_n
 * — computed on the device from the power-of-two row scales s_r > max|row| of the operands actually multiplied — to a
 * device scalar that is reset when a call starts; ecw_int8_error_bound reads it back (synchronises the stream).  NaN:
 * an operand held a non-finite value (its rows get the scale NaN, so the affected outputs are NaN as in FP64).
 * ecw_ctx_set_engine_override(ctx, 1) makes the following calls run their plans without the INT8 route (FP64 DMMA
 * kernels; needs the FP64 layouts "vvvv_p" / "ovvv_p" bound) — the host re-runs a call this way when the bound
 * exceeds its tolerance (ecw_cc_b200/eris.py: INT8_TOL); 0 restores the configured engine. */
int ecw_int8_error_bound(ecw_ctx* ctx, double* bound_out, void* stream);
int ecw_ctx_set_engine_override(ecw_ctx* ctx, int force_dmma);
/* INT8 products with fewer output tiles than SMs and a contraction length >= min_k (a multiple of 32) are cut into
 * equal K chunks, one product each, summed in a fixed order (default 65536; <= 0: never). */
int ecw_ctx_set_int8_splitk(ecw_ctx* ctx, int64_t min_k);
/* CUDA-graph replay (default on): on one GPU a call of ecw_ccsd_tupdate / lupdate / gamma / energy whose plan and
 * pointer arguments were seen before is one cudaGraphLaunch on the caller's stream (captured on a private stream at the
 * first such call; up to 24 graphs are kept, least recently used first out).  The small shapes of the molecular
 * configurations are bound by the launch rate of the several hundred kernels of a residual evaluation.  Off while
 * ecw_profile_enable is on and for sharded contexts.  ecw_ctx_graph_stats: replays / captures so far. */
int ecw_ctx_set_graphs(ecw_ctx* ctx, int on);
int ecw_ctx_graph_stats(ecw_ctx* ctx, int64_t* hits, int64_t* captures);
int ecw_pending_collective(ecw_ctx* ctx, int64_t* desc6);

/* ---- integral container (consumed type `Eris.geris`, Eris.py:132-154) ---- */
/* Constant device layouts, by slot name:
 *   "oooo" [o,o,o,o]  "ooov" [o,o,o,v]  "oovv" [o,o,v,v]  "ovvv" [o,v,v,v]
 *   "oovv_ph" [(m,e),(n,f)] = oovv[m,n,e,f]     "ovov_ph" [(i,a),(n,f)] = ovov[n,a,i,f]
 *   "oooo_p" [ij_p,kl_p]  "oovv_p" [ij_p,ab_p]  "ovvv_p" [m,a,ef_p]  "vvvv_p" [ab_p,cd_p]
 *   "vvvv_oz" / "vvvv_ozs": int8 digit planes / row statistics of vvvv_p (ecw_eris_vvvv_planes)
 *   "ovvv_oz1" / "ovvv_oz1s", "ovvv_oz2" / "ovvv_oz2s": the same for ovvv_p, both orientations (ecw_eris_ovvv_planes)
 * with the antisymmetric pair index p(x<y) = y(y-1)/2 + x.  Also bindable:
 * "scal" (16 doubles of device scratch for scalars). */
int64_t ecw_slot_elems(ecw_ctx* ctx, const char* slot);
int ecw_bind(ecw_ctx* ctx, const char* slot, void* device_ptr);
/* Fill the derived layouts (oovv_ph, ovov_ph, *_p) from dense canonical blocks
 * already on the device; "oooo","ooov","oovv","ovvv" must be bound to the dense
 * blocks themselves.  Replaces the block copies of Eris.py:132-150. */
int ecw_eris_pack_from_dense(ecw_ctx* ctx, const double* ovov_dense, const double* vvvv_dense, void* stream);
/* INT8 engine: the packed vvvv shard lives on the device as digit planes only.  Bind "vvvv_oz"
 * (ecw_slot_elems x 8 bytes) and "vvvv_ozs", then pass the FP64 rows [row0, row0+nrows) of this rank's
 * shard ([nrows, P_v], row0 a multiple of 128, every chunk but the last a multiple of 128 rows) chunk by
 * chunk; after the last chunk the plans read the planes and "vvvv_p" need not be bound. */
int ecw_eris_vvvv_planes(ecw_ctx* ctx, const double* rows, int64_t row0, int64_t nrows, void* stream);
/* INT8 engine, optional (needs nocc % 8 == 0 and nvir % 8 == 0): cut the bound "ovvv_p" into digit planes in both
 * orientations — bind "ovvv_oz1"/"ovvv_oz1s" (rows (m,a), k = ef_p) and "ovvv_oz2"/"ovvv_oz2s" (rows ef_p,
 * k = (m,a)) first.  Afterwards "ovvv_p" need not stay bound; R4/R6/R9 (CCSD.py:602-605, 461-470, 396-402) skip
 * their per-call cuts and the ovvv terms of CCSD.py:294, 311-312, 499, 585-600 run as batched INT8 products. */
int ecw_eris_ovvv_planes(ecw_ctx* ctx, void* stream);
/* Fill every bound integral layout with the function-defined synthetic
 * integrals (DESIGN.md "Synthetic inputs"); dense vvvv never exists. */
int ecw_eris_synthetic(ecw_ctx* ctx, double scale, void* stream);
/* One synthetic tensor (kinds: ecw SynthKind in kernels.h: 10 fock, 11 fsp,
 * 12 t1, 13 l1, 14 t2, 15 l2, 0..9 integral layouts), rows [row0,row0+nrows). */
int ecw_synth_tensor(int kind, double* out, int nocc, int nvir, int64_t row0, int64_t nrows, double scale,
                     void* stream);

/* ---- workspace ------------------------------------------------------------ */
/* func: "tupdate","lupdate","gamma","energy", or a CCS entry name. */
int64_t ecw_workspace_bytes(ecw_ctx* ctx, const char* func, int mode_flags);
int ecw_set_workspace(ecw_ctx* ctx, void* device_ptr, int64_t bytes);

/* ---- CCSD (CCSD.py) --------------------------------------------------------- */
/* GCC.tupdate(t1,t2,fsp,alpha,equation) — CCSD.py:248-338.  fock = bare Fock (n x n). */
int ecw_ccsd_tupdate(ecw_ctx* ctx, const double* t1, const double* t2, const double* fsp, const double* fock,
                     int mode_flags, double alpha, double* t1new, double* t2new, void* stream);
/* GCC.lupdate(t1,t2,l1,l2,fsp,alpha,equation) — CCSD.py:419-535 (incl. Linter :543-623). */
int ecw_ccsd_lupdate(ecw_ctx* ctx, const double* t1, const double* t2, const double* l1, const double* l2,
                     const double* fsp, const double* fock, int mode_flags, double alpha, double* l1new,
                     double* l2new, void* stream);
/* GCC.gamma(t1,t2,l1,l2) — CCSD.py:136-182, 204-208.  rdm1: n x n. */
int ecw_ccsd_gamma(ecw_ctx* ctx, const double* t1, const double* t2, const double* l1, const double* l2,
                   double* rdm1, void* stream);
/* GCC.energy(t1,t2,fsp) — CCSD.py:224-242.  e_out: one device double. */
int ecw_ccsd_energy(ecw_ctx* ctx, const double* t1, const double* t2, const double* fsp, double* e_out,
                    void* stream);
/* ---- ECW-CCS intermediates (replace Gccs.T1inter / L1inter / R1inter / es_L1inter, CCS.py:271-312, :490-537,
 * :774-872, :1164-1234) ------------------------------------------------------------
 * One cached plan — one call, and on one GPU one CUDA-graph launch — per function: everything of a CCS ground- or
 * excited-state iteration that reads an integral block.  ts [o,v], fsp [n,n], vm [n,n] (the state potential, or null:
 * Pia / P = 0).  Results: F [n,n], whose blocks carry the one-body intermediates
 *     t1inter:   vv = Fab, oo = Fji, vo = Fai            l1inter:   ov = Fia, vv = Fba, oo = Fij
 *     r1inter:   vv = Fab, oo = Fji, ov = Tia            esl1inter: vv = Fba, oo = Fij, ov = Zia
 * (other blocks zero); W [v,o,o,v] = Wbija / Wakic; X [o,v] = Pia / P; e_out[0] = E / Er / El on the device
 * (l1inter: written only when e_term != 0, CCS.py:490 `E_term`).  The singles-sized updates that consume them
 * (tsupdate, lsupdate, rsupdate, es_lsupdate, r0 / l0) are sequences of the primitive ops below with host-side
 * scalars between them (ecw_cc_b200/CCS.py). */
int ecw_ccs_t1inter(ecw_ctx* ctx, const double* ts, const double* fsp, double* F, void* stream);
int ecw_ccs_l1inter(ecw_ctx* ctx, const double* ts, const double* fsp, int e_term, double* F, double* W, double* e_out,
                    void* stream);
int ecw_ccs_r1inter(ecw_ctx* ctx, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                    double* e_out, void* stream);
int ecw_ccs_esl1inter(ecw_ctx* ctx, const double* ts, const double* fsp, const double* vm, double* F, double* W, double* X,
                      double* e_out, void* stream);

/* out[0] = max |x[ijab]+x[jiab]|, |x[ijab]+x[ijba]| over a doubles amplitude, out[1] = max |x| (two device doubles). */
int ecw_antisym_defect(const double* x, int nocc, int nvir, double* out, void* stream);
/* utilities.subdiff(eq,var,alpha) — utilities.py:26-73 (element-wise, any shape). */
int ecw_subdiff(const double* eq, const double* var, double alpha, double* out, int64_t n, void* stream);

/* ---- solver loop (Solver_GS.Solver_CCSD.SCF, Solver_GS.py:621-742) ------------------------------------------
 * Convergence vector of one amplitude pair and its squared distance to the previous iteration's
 * (tl_check / l_check, Solver_GS.py:598-612): conv[i] = |a[i]| + |b[i]| (b == NULL: conv[i] = a[i]);
 * sumsq[0] = (accumulate ? sumsq[0] : 0) + sum_i (conv[i] - prev[i])^2 (prev == NULL: + 0).  conv may not alias prev;
 * scratch1024: 1024 device doubles.  Deterministic (fixed two-stage reduction). */
int ecw_conv_check(const double* a, const double* b, const double* prev, double* conv, int64_t n, double* scratch1024,
                   double* sumsq, int accumulate, void* stream);

/* Experimental potential of the density-matrix ('mat') ground-state target and the dressed Fock matrix, on the device
 * (exp_pot.Exp.Vexp_update 'mat' branch, exp_pot.py:185-195, and Solver_GS.py:690-692): for the n = dim*dim elements
 * diff = target - rdm1, vexp = L*diff, fsp = fock - vexp; stats2[0] = sum |diff|, stats2[1] = max |diff| (the numerator
 * of Delta and vmax).  All pointers are device pointers; deterministic. */
int ecw_vexp_mat(const double* rdm1, const double* target, const double* fock, double L, double* vexp, double* fsp,
                 double* stats2, int64_t n, void* stream);

/* Structure-factor ('F') target.  ecw_ft_aopair fills out[2][nG][nao][nao] (Re plane, then Im plane) with the
 * Fourier-transformed AO pairs A_mu,nu(G) = int phi_mu phi_nu exp(+i G.r) d^3r for the scattering vectors G[nG,3]
 * (bohr^-1).  prim[nprim,8] = {Ax, Ay, Az, alpha, coef, lx, ly, lz} lists primitive Cartesian Gaussians (bohr; coef
 * includes normalisation and contraction; l <= 2 per direction), those of AO mu at rows ao_first[mu] ..
 * ao_first[mu+1]-1 (ao_first[nao+1], int64).  FP64, fixed summation order: two calls give identical bits.  A malformed
 * table yields NaN elements.  All pointers are device pointers. */
int ecw_ft_aopair(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* G, int64_t nG,
                  double* out, void* stream);
/* One iteration of the 'F' potential, ground state: D = C_a gamma C_a^T + C_b gamma C_b^T (rdm1 gamma [n,n] in
 * spin-orbital MOs, mo_coeff_g [2nao,n] with alpha rows first), F_calc[2][nG] = sum_mu,nu D_mu,nu A_mu,nu(G_h) (Re, Im),
 * dF = F_exp - F_calc (F_exp[2][nG]), vexp = L sum_h Re[conj(dF_h) C_g^T blockdiag(A_h, A_h) C_g] (= -dP/dgamma of
 * P = L/2 sum_h |dF_h|^2), fsp = fock - vexp; stats2[0] = sum_h |dF_h|, stats2[1] = max |vexp|.  ft: the planes of
 * ecw_ft_aopair.  workspace: ecw_vexp_sf_workspace_bytes(n, nao, nG) bytes of device memory.  Device pointers;
 * stream-ordered, no synchronisation; fixed reduction order. */
int ecw_vexp_sf(const double* rdm1, int n, const double* mo_coeff_g, int nao, const double* ft, int64_t nG,
                const double* F_exp, double L, const double* fock, double* vexp, double* fsp, double* F_calc,
                double* stats2, double* workspace, void* stream);
int64_t ecw_vexp_sf_workspace_bytes(int n, int nao, int64_t nG);

/* Amplitude ('Fobs') target: measured |F_obs| with weights 1/sigma^2, a unit cell of nsym copies of the molecule and
 * thermal smearing.  ecw_ft_aopair_cryst fills out[2][nG][nao][nao] with the symmetrised, smeared planes
 *   B_mu,nu(h) = sum_s exp(+2 pi i h.t_s) T_mu,nu(G_hs) A_mu,nu(G_hs),   T_mu,nu = (T_A + T_B)/2, T_A(G) = exp(-G^T U_A G/2)
 * (A as for ecw_ft_aopair; mu on atom A, nu on atom B).  prim / ao_first as for ecw_ft_aopair; ao_atom[nao] (int64) is
 * the atom of each AO; U[natom][6] = Cartesian ADP (xx, yy, zz, xy, xz, yz) in bohr^2; Gs[nG][nsym][3] = G_{R_s^T h} in
 * bohr^-1 and phase[nG][nsym][2] = (cos, sin) of 2 pi h.t_s, tabulated by the caller; 1 <= nsym <= 192.  FP64, fixed
 * summation order (operations in list order), identical bits call to call; a malformed table yields NaN elements. */
int ecw_ft_aopair_cryst(const double* prim, int64_t nprim, const int64_t* ao_first, const int64_t* ao_atom, int nao,
                        const double* U, int natom, const double* Gs, const double* phase, int nsym, int64_t nG,
                        double* out, void* stream);
/* One iteration of the 'Fobs' potential, ground state: D and F_calc[2][nG] as for ecw_vexp_sf (ft: the planes of
 * ecw_ft_aopair_cryst), a_h = |F_calc(h)|, w = weight[nG] (1/sigma^2).  Scale k = k_fixed if k_fixed > 0 (N_p = 0), else
 * refined, k = sum w F_obs a / sum w a^2 (N_p = 1, needs nG >= 2).  chi^2 = sum w (k a - F_obs)^2 / (nG - N_p), the
 * penalty P = L chi^2, vexp = sum_h Re[conj(c_h) C_g^T blockdiag(B_h, B_h) C_g] with c_h = 2 L k / (nG - N_p) w_h (F_obs
 * - k a_h) F_calc(h) / a_h, c_h = 0 where a_h <= 1e-12 max a (a cusp of |F|, the direction there is rounding noise)
 * (= -dP/dgamma at fixed k; also at the refined k, where dP/dk = 0), fsp = fock - vexp.  stats4 = [sum_h |k a_h - F_obs(h)|, max |vexp|, k, chi^2].  workspace:
 * ecw_vexp_sfobs_workspace_bytes(n, nao, nG) bytes.  Device pointers; stream-ordered, no synchronisation; fixed
 * reduction order. */
int ecw_vexp_sfobs(const double* rdm1, int n, const double* mo_coeff_g, int nao, const double* ft, int64_t nG,
                   const double* F_obs, const double* weight, double k_fixed, double L, const double* fock, double* vexp,
                   double* fsp, double* F_calc, double* stats4, double* workspace, void* stream);
int64_t ecw_vexp_sfobs_workspace_bytes(int n, int nao, int64_t nG);

/* Density maps.  ecw_density_grid fills out[n1][n2][n3] (k fastest, the cube-file order) with
 *   rho(r_ijk) = sum_mu,nu dm[mu][nu] phi_mu(r_ijk) phi_nu(r_ijk),   r_ijk = origin + i a1 + j a2 + k a3,
 * box[12] = {origin, a1, a2, a3} in bohr (a HOST array), dm[nao][nao] the AO density (need not be symmetric), prim /
 * ao_first as for ecw_ft_aopair.  Points are processed in chunks of 32768: the AO values Phi[chunk][nao] (a fixed-order
 * sum over each AO's primitives, no screening), X = Phi dm (FP64 GEMM), rho_p = sum_mu X_p,mu Phi_p,mu (fixed order).
 * workspace: ecw_density_grid_workspace_bytes(nao, n1 n2 n3) bytes of device memory.  Identical bits call to call; a
 * malformed table yields NaN.  Device pointers except box; stream-ordered, no synchronisation. */
int ecw_density_grid(const double* prim, int64_t nprim, const int64_t* ao_first, int nao, const double* dm,
                     const double* box, int n1, int n2, int n3, double* out, double* workspace, void* stream);
int64_t ecw_density_grid_workspace_bytes(int nao, int64_t npts);
/* Fourier synthesis on the fractional grid x_ijk = (i/n1, j/n2, k/n3) of a unit cell, out[n1][n2][n3]:
 *   rho(x) = (F000 + 2 sum_h (Re F_h cos 2 pi h.x + Im F_h sin 2 pi h.x)) / volume_bohr3
 * over the half set hkl_half[N][3] (int64; the Friedel mate -h of each is implied) with coef[2][N] = (Re F, Im F): the
 * inverse of the exp(+i G.r) convention of ecw_ft_aopair.  The phase is exact, (h_d i_d) mod n_d in integers and a
 * table of 2 pi m / n_d per axis; 1 <= n_d <= 512, N >= 0.  Fixed summation order, identical bits call to call.  Device
 * pointers; stream-ordered, no synchronisation. */
int ecw_fourier_map(const int64_t* hkl_half, const double* coef, int64_t N, double F000, double volume_bohr3, int n1,
                    int n2, int n3, double* out, void* stream);

/* ---- primitive device ops ---------------------------------------------------------
 * The CCS class (CCS.py:197-1518: T1inter/tsupdate/L1inter/lsupdate/R1inter/rsupdate/es_L1inter/
 * es_lsupdate/R0inter/L0inter/*_fromE/gamma_*) and the GCC intermediate getters (cc_Fvv, cc_Woooo,
 * cc_Wovvo, Linter, ...) are short sequences of o x v / o^2 v^2 contractions; the host states them
 * with the same index strings as the reference and each one runs through the contraction engine
 * (permutes + FP64 tensor-core GEMM).  Tensors are described by pointer, rank, extents and
 * element strides.  A return value of -2 means the bound workspace is too small:
 * ecw_op_workspace_needed() gives the bytes, rebind with ecw_set_workspace and retry. */
typedef struct ecw_tensor {
  void* ptr;
  int32_t nd;
  int64_t dim[6];
  int64_t str[6];
} ecw_tensor;
#define ECW_SUBDIFF_SINGLES 8
/* C[sc] = alpha * sum_contracted A[sa] B[sb] + beta * C[sc]   (numpy.einsum / pyscf.lib.einsum) */
int ecw_op_contract(ecw_ctx* ctx, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B,
                    const char* sb, double beta, const ecw_tensor* C, const char* sc, void* stream);
/* C[sc] = alpha * A[sa] + beta * C[sc]   (sa a permutation of sc: transposes, block copies, axpy) */
int ecw_op_axpby(ecw_ctx* ctx, double alpha, const ecw_tensor* A, const char* sa, double beta, const ecw_tensor* C,
                 const char* sc, void* stream);
/* C = alpha * A * B + beta * C element-wise (A and/or B may be NULL: scaling / fill) */
int ecw_op_mul(ecw_ctx* ctx, double alpha, const ecw_tensor* A, const ecw_tensor* B, double beta, const ecw_tensor* C,
               void* stream);
/* C4[p,q,r,s] = alpha * sign * A2[pair(p,q), pair(r,s)] + beta * C4 — expand antisymmetry-packed pairs
 * (flags bit0: first pair packed, bit1: second pair packed); used by GCC.cc_Wvvvv at small sizes. */
int ecw_op_unpack(ecw_ctx* ctx, double alpha, const ecw_tensor* A2, int flags, double beta, const ecw_tensor* C4,
                  void* stream);
/* C[i,i] += alpha * fock[offset+i, offset+i]   (CCS.py:307-308, 529-530, 927-928, 1384-1385) */
int ecw_op_diag_shift(ecw_ctx* ctx, const ecw_tensor* C, double alpha, const ecw_tensor* fock, int64_t offset,
                      void* stream);
/* residual -> update: out = resid / (shift + e_i - e_a), or with ECW_HAS_ALPHA the L1 form
 * (subdiff(resid, amp, alpha) + amp * d) / d   (CCS.py:349, 377-382, 938; CCSD.py:316-336) */
int ecw_op_denom(ecw_ctx* ctx, const ecw_tensor* resid, const ecw_tensor* amp, const ecw_tensor* fock, int nocc,
                 int mode_flags, double alpha, double shift, const ecw_tensor* out, void* stream);
/* out_dev[0] = beta * out_dev[0] + alpha * <A, B> */
int ecw_op_dot(ecw_ctx* ctx, double alpha, const ecw_tensor* A, const ecw_tensor* B, double beta, double* out_dev,
               void* stream);
int64_t ecw_op_workspace_needed(ecw_ctx* ctx);

/* ---- introspection / test hooks ---------------------------------------------- */
/* Host-only test hook: plan as if ecw_eris_vvvv_planes had completed (so the lowering of the
 * digit-plane ladders can be dumped and replayed on a box without a GPU). */
int ecw_ctx_test_assume_vvvv_planes(ecw_ctx* ctx);
int ecw_ctx_test_assume_ovvv_planes(ecw_ctx* ctx);
/* Host-only test hook: operands of at least min_elems elements keep their digit planes for a second use within a
 * plan (default 2^20); small values let CPU-sized plans exercise that cache. */
int ecw_ctx_test_cut_cache_min(ecw_ctx* ctx, int64_t min_elems);
/* JSON dump of the op list a call would launch (host only, no CUDA). */
int64_t ecw_plan_dump(ecw_ctx* ctx, const char* func, int mode_flags, char* buf, int64_t buflen);
/* the same for one ecw_op_contract call (operands appear as slots "a0", "a1", "b0"; host only, pointers unused) */
int64_t ecw_plan_dump_contract(ecw_ctx* ctx, double alpha, const ecw_tensor* A, const char* sa, const ecw_tensor* B,
                               const char* sb, double beta, const ecw_tensor* C, const char* sc, char* buf,
                               int64_t buflen);
/* executed GEMM flops (sum of 2MNK) and launches of a plan */
double ecw_plan_flops(ecw_ctx* ctx, const char* func, int mode_flags);
int64_t ecw_plan_launches(ecw_ctx* ctx, const char* func, int mode_flags);
/* Raw FP64 tensor-core GEMM: C = alpha op(A) op(B) + beta C (row-major C);
 * ta/tb: 0 = A is [M,K] / B is [K,N] row-major, 1 = transposed storage.
 * cfg < 0 picks the tile configuration automatically; cfg = 1-4, 8, 10-16, 18 or 19 forces one of the DMMA tiles
 * the picker chooses from (csrc/gemm.cu, gemm_pick_config), 20 / 21 the TMA-fed 128x128 / 112x128 tiles (the 128x128
 * DMMA tile where TMA does not apply).  Any other cfg returns non-zero without launching. */
int ecw_dgemm(int ta, int tb, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
              const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int cfg, void* stream);
/* FP64 GEMM on the INT8 tcgen05 tensor pipe (csrc/ozaki.cu: operands cut into base-256 int8 digits).
 * ecw_ozaki_split cuts X[R,K] (element (r,k) at X[r*rs + k*ks], one of rs/ks == 1) into `ns` int8
 * digit planes (ecw_ozaki_plane_bytes bytes) and row statistics (ecw_ozaki_stat_elems doubles: power-of-two
 * row scales, then row sums); ecw_ozaki_gemm forms C[m*crs + n*ccs] = alpha * sum_k A[m,k] B[n,k]
 * + beta * C from two plane sets.  Replaces the numpy einsum of the large contractions
 * (CCSD.py:305, 411, 484, 602) together with ecw_dgemm. */
int64_t ecw_ozaki_plane_bytes(int64_t R, int64_t K, int ns);
int64_t ecw_ozaki_padded_rows(int64_t R);
int64_t ecw_ozaki_stat_elems(int64_t R);
int ecw_ozaki_tile_n(int ns);
int ecw_ozaki_split(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, void* planes, double* scale,
                    void* stream);
/* two-level contraction index k = (k1, k2) (element at X[r*rs + k1*ks1 + k2*ks2], k2 padded to 32 per k1; the
 * statistics then also hold the row sums per k1) and batches of products over sub-blocks of two plane sets:
 * bt15 = {batch, a_row0, a_rowb, b_row0, b_rowb, a_kb0, a_kbb, b_kb0, b_kbb, a_t0, a_tb, b_t0, b_tb, c_b, nkb}
 * (csrc/kernels.h, struct OzBatch). */
int64_t ecw_ozaki_plane_bytes2(int64_t R, int64_t K1, int64_t K2, int ns);
int64_t ecw_ozaki_stat_elems2(int64_t R, int64_t K1);
int ecw_ozaki_split2(const double* X, int64_t R, int64_t K1, int64_t K2, int64_t rs, int64_t ks1, int64_t ks2, int ns,
                     void* planes, double* stats, void* stream);
int ecw_ozaki_gemm_batched(const void* planes_a, const double* stats_a, int64_t a_rows, const void* planes_b,
                           const double* stats_b, int64_t b_rows, int64_t M, int64_t N, int64_t K, double* C,
                           int64_t crs, int64_t ccs, double alpha, double beta, int ns, const int64_t* bt15,
                           void* stream);
/* chunked cut: X holds rows [row0, row0+R) of an operand of total_rows rows (row0 and every chunk but the
 * last multiples of 128); planes/scale address the whole plane set */
int ecw_ozaki_split_rows(const double* X, int64_t R, int64_t K, int64_t rs, int64_t ks, int ns, void* planes,
                         double* scale, int64_t row0, int64_t total_rows, void* stream);
int ecw_ozaki_gemm(const void* planes_a, const double* scale_a, const void* planes_b, const double* scale_b, int64_t M,
                   int64_t N, int64_t K, double* C, int64_t crs, int64_t ccs, double alpha, double beta, int ns,
                   void* stream);
/* per-op device timing of the last executed plan (ms), written as JSON */
int ecw_profile_enable(ecw_ctx* ctx, int on);
int64_t ecw_profile_dump(ecw_ctx* ctx, char* buf, int64_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* ECW_B200_H */
