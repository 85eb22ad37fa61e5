// plan.h — execution plans for the coupled-cluster residual path.
//
// A Plan is a flat list of device operations (GEMMs, index permutes, a few
// fused element-wise kernels) over buffer *slots*: caller-owned amplitude /
// Fock / output arrays, the constant integral layouts of the eris container,
// and one workspace arena whose offsets are fixed at plan-build time.  The
// builders in ccsd_plan.cpp / ccs_plan.cpp state the reference equations
// (CCSD.py:136-623, CCS.py:23-1518) as binary tensor contractions; the
// contraction engine here lowers each one to (optional permutes) + one FP64
// tensor-core GEMM.  Plans are pure host data: building one touches no CUDA
// API, so the lowering can be inspected (ecw_plan_dump) and is replayed on the
// stream by exec.cu, optionally captured into a CUDA graph.
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include <stdexcept>
#include <algorithm>

#include "ozaki_layout.h"

namespace ecw {

constexpr int MAXD = 6;

// Buffer slots.  Everything the kernels touch is (slot, element offset).
enum Slot : int {
  S_WS = 0,       // workspace arena (caller allocated, ecw_workspace_bytes)
  S_T1, S_T2, S_L1, S_L2, S_FSP, S_FOCK,        // inputs (device, FP64, C order)
  S_OUT1, S_OUT2, S_RDM1, S_SCAL,               // outputs; S_SCAL = 16 device scalars
  // constant integral layouts (eris container)
  S_OOOO, S_OOOV, S_OOVV, S_OOVV_PH, S_OVOV_PH, S_OVVV,
  S_OOOO_P, S_OOVV_P, S_OVVV_P, S_VVVV_P,
  // int8 digit planes + row scales of vvvv_p for the INT8-tensor-core GEMM (ozaki.cu); element
  // offsets into these two slots are in units of 8 bytes like everywhere else
  S_VVVV_OZ, S_VVVV_OZS,
  // digit planes of ovvv_p in both orientations: OZ1 = rows (m,a), k = ef_p;  OZ2 = rows ef_p, k = (m, a)
  S_OVVV_OZ1, S_OVVV_OZ1S, S_OVVV_OZ2, S_OVVV_OZ2S,
  // generic argument slots for the CCS entry points
  S_A0, S_A1, S_A2, S_A3, S_A4, S_A5, S_A6, S_A7, S_A8, S_A9,
  S_B0, S_B1, S_B2, S_B3, S_B4, S_B5, S_B6, S_B7,
  S_COUNT
};
const char* slot_name(int s);

// the device scalars of slot S_SCAL
enum Scalar : int {
  SC_RESULT = 0,        // the scalar result of a plan (energy-like), copied out by the entry points
  SC_DOT = 1,           // ecw_op_dot
  SC_INT8_BOUND = 15,   // run-time error bound of the INT8-route products of the last call (ecw_int8_error_bound)
  SC_COUNT = 16
};

// this rank's part [*i0, *i0 + *ni) of an index of extent L that is distributed in chunks of ceil(L / world)
inline void shard_range(int64_t L, int rank, int world, int64_t* i0, int64_t* ni) {
  const int64_t ch = (L + world - 1) / world;
  *i0 = std::min<int64_t>(L, (int64_t)rank * ch);
  *ni = std::min<int64_t>(L, *i0 + ch) - *i0;
}

struct Tensor {
  int slot = -1;
  int64_t off = 0;
  int nd = 0;
  int64_t dim[MAXD] = {0};
  int64_t str[MAXD] = {0};
  int64_t size() const { int64_t n = 1; for (int i = 0; i < nd; ++i) n *= dim[i]; return n; }
  bool valid() const { return slot >= 0; }
};

Tensor make_tensor(int slot, int64_t off, std::initializer_list<int64_t> dims);
Tensor reshape(const Tensor& t, std::initializer_list<int64_t> dims);   // contiguous only
Tensor block2(const Tensor& m, int64_t r0, int64_t nr, int64_t c0, int64_t nc);  // 2-D sub-block
Tensor transpose2(const Tensor& m);
Tensor slice0(const Tensor& t, int64_t i0, int64_t n);                   // leading-dim range
Tensor slice_dim(const Tensor& t, int d, int64_t i0, int64_t n);         // range of dimension d

enum OpKind : int {
  OP_GEMM = 0,    // C = alpha op(A) op(B) + beta C   (batched / split-K)
  OP_REDUCE,      // C = alpha sum_z P[z] + beta C
  OP_PERMUTE,     // C[..] = alpha A[perm ..] + beta C   (strided N-d copy)
  OP_FILL,        // C = alpha
  OP_TAU,         // C = t2 + alpha t1[ia]t1[jb] - beta t1[ib]t1[ja]
  OP_PACK,        // antisymmetric pair packing of a 4-index view
  OP_UNPACK,      // inverse (scatter with signs)
  OP_FINISH,      // residual -> update / subdiff (CCSD.py:316-338)
  OP_DOT,         // scal[k] = beta scal[k] + alpha <A,B>
  OP_SCALE_DEV,   // C *= d0 + d1 * scal[k]
  OP_DIAG_ADD,    // C[i,i] += alpha * fock[off+i, off+i]
  OP_RDM1,        // assemble the symmetrised rdm1 (CCSD.py:154-160)
  OP_EWISE,       // small CCS element-wise helpers (sub-kind in i0)
  OP_ALLGATHER,   // collective: every rank contributes `a` (i0 elements); `c` receives world*i0 (host runs it)
  OP_OZ_SPLIT,    // a = X[R=M, (K1=i1, K2=K)] (element strides lda, ldc, ldb) -> c = i0 int8 digit planes, d = statistics
  OP_OZ_GEMM,     // C_b[m*i1 + n*i2] = alpha sum_k A_b[m,k] B_b[n,k] + beta C_b from plane sets a (stats d, lda rows)
                  // and b (stats e, ldb rows); sub-blocks per batch in oz[] (OzBatch order), sC = C offset per batch
  OP_ASYM4,       // c[ijab] = alpha b[ijab] + a[ijab] - a[jiab] - a[ijba] + a[jiba] + beta c[ijab]  (b may be unset)
  OP_ALLTOALL,    // collective: block q (i0 elements) of `a` goes to rank q; block q of `c` comes from rank q
};
const char* op_kind_name(int kind);

struct Op {
  int kind = 0;
  Tensor a, b, c, d, e;       // operands (meaning per kind)
  double alpha = 1.0, beta = 0.0;
  // GEMM
  int64_t M = 0, N = 0, K = 0, lda = 0, ldb = 0, ldc = 0;
  int64_t sA = 0, sB = 0, sC = 0, batch = 1;
  int ta = 0, tb = 0;         // 0: K-contiguous A / N-contiguous B (row-major), 1: transposed
  int64_t splitk = 1, kchunk = 0;
  // generic ints / doubles
  int64_t i0 = 0, i1 = 0, i2 = 0, i3 = 0;
  double d0 = 0.0, d1 = 0.0;
  int64_t oz[13] = {0};       // OP_OZ_GEMM: a_row0,a_rowb,b_row0,b_rowb,a_kb0,a_kbb,b_kb0,b_kbb,a_t0,a_tb,b_t0,b_tb,nkb
  std::string note;
};

// A plane set: the int8 digits of an operand X[R, (K1, K2)] (ozaki.cu) plus its row statistics.
struct OzSet {
  Tensor planes, stats;
  int64_t R = 0, K1 = 1, K2 = 0;
  bool owned = false;          // lives in the workspace arena and is released by oz_release
  bool cached = false;         // lives in the workspace arena, owned by the cut cache of the plan
  int64_t rp() const { return ozaki_padded_rows(R); }
  int64_t nkb2() const { return ozaki_kblocks(1, K2); }
};
// The part of a plane set one product of a batch reads: rows [row0 + b*rowb, +M|N), k1 values [k10 + b*k1b, +nk1)
// (nk1 = K1: the whole contraction index; otherwise nk1 must be 1).
struct OzSel {
  int64_t row0 = 0, rowb = 0, k10 = 0, k1b = 0, nk1 = 0;   // nk1 = 0: all K1
};

struct Arena {
  struct Blk { int64_t off, size; bool used; };
  std::vector<Blk> blks;
  int64_t peak = 0;
  int64_t alloc(int64_t n);
  void release(int64_t off);
};

struct PlanError : std::runtime_error { using std::runtime_error::runtime_error; };

class Plan {
 public:
  std::vector<Op> ops;
  Arena arena;
  int sm_count = 148;
  int rank = 0, world = 1;     // owner-computes distribution of the heavy contractions
  // Large unbatched GEMMs run on the INT8 tcgen05 pipe by error-free splitting (ozaki.cu) when
  // oz_ns > 0 and 2MNK >= oz_min_flops; oz_ns = number of 7-bit digits (7: FP64-level accuracy).
  int oz_ns = 0;
  double oz_min_flops = 0.0;
  int64_t oz_splitk_min_k = 65536;   // INT8 products with few output tiles and K >= this are cut into K chunks
  bool vvvv_planes = false;    // vvvv_p is bound as digit planes (S_VVVV_OZ/S_VVVV_OZS), not as FP64
  bool ovvv_planes = false;    // ovvv_p is bound as digit planes in both orientations (S_OVVV_OZ1/2)
  int64_t nocc = 0, nvir = 0;  // needed to recognise the constant plane sets
  double oz_flops = 0.0;       // part of gemm_flops that runs on the INT8 pipe
  double gemm_flops = 0.0;     // sum of 2MNK over GEMM ops (executed flops)
  double perm_bytes = 0.0;     // bytes moved by engine-inserted permutes

  Tensor tmp(std::initializer_list<int64_t> dims);
  Tensor tmpv(const std::vector<int64_t>& dims);
  // dense temp whose leading extent is padded to a multiple of `world` chunks (for in-place allgather)
  Tensor tmp_lead_padded(std::initializer_list<int64_t> dims);
  int64_t lead_chunk(int64_t extent) const { return (extent + world - 1) / world; }
  // C (leading index distributed) = alpha * A (same leading label) . B ; then allgather of C
  void contract_lead_dist(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                          const Tensor& C, const char* sc, const char* note = "");
  void allgather(const Tensor& chunk, int64_t count, const Tensor& full, const char* note = "");
  // send / recv: world blocks of `count` elements each (workspace); no-op copy when world == 1
  void alltoall(const Tensor& send, int64_t count, const Tensor& recv, const char* note = "");
  // C += sum over ranks of `part` (same shape, contiguous; all-gathered and added in rank order on every rank:
  // bit-identical replicas).  world == 1: C += part.
  void sum_ranks_add(const Tensor& part, const Tensor& C, const char* note = "");
  // this rank's range of an index of extent L that is distributed in chunks of lead_chunk(L)
  void my_range(int64_t L, int64_t* i0, int64_t* ni) const { shard_range(L, rank, world, i0, ni); }
  // C (contiguous) += alpha * sum_K A.B with the range of the contracted label `lab` split across ranks
  // (partial sums are all-gathered and added in rank order on every rank: bit-identical replicas)
  void contract_split(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                      const Tensor& C, const char* sc, char lab, const char* note = "");
  void release(const Tensor& t);

  // C[sc] = alpha * sum_K A[sa] B[sb] + beta * C[sc]
  void contract(double alpha, const Tensor& A, const char* sa, const Tensor& B, const char* sb,
                double beta, const Tensor& C, const char* sc, const char* note = "");
  // C[sc] = alpha * A[sa] + beta * C[sc]   (sa is a permutation of sc)
  void permute(double alpha, const Tensor& A, const char* sa, double beta, const Tensor& C,
               const char* sc, const char* note = "");
  void axpby(double alpha, const Tensor& A, double beta, const Tensor& C, const char* note = "");
  void fill(const Tensor& C, double value);
  // out = t2 + c1 t1[ia]t1[jb] - c2 t1[ib]t1[ja]
  void tau(const Tensor& t2, const Tensor& t1, double c1, double c2, const Tensor& out);
  // the same for the rows i0 .. i0+ni-1 of the leading occupied index: t2 and out are [ni, o, v, v] views
  void tau_rows(const Tensor& t2_rows, const Tensor& t1, int64_t i0, double c1, double c2, const Tensor& out_rows);
  // out[ijab] = c0 base[ijab] + z[ijab] - z[jiab] - z[ijba] + z[jiba] + beta out[ijab]; all contiguous [o,o,v,v]
  void asym4(double c0, const Tensor* base, const Tensor& z, double beta, const Tensor& out, const char* note = "");
  // pack/unpack: flags bit0 = first pair packed, bit1 = second pair packed,
  //              bit2 = antisymmetrise second pair while packing (x[..rs]-x[..sr])
  //              bit3 = antisymmetrise first pair while packing  (x[pq..]-x[qp..])
  void pack(double alpha, const Tensor& a4, int flags, double beta, const Tensor& c2);
  void unpack(double alpha, const Tensor& a2, int flags, double beta, const Tensor& c4);
  void finish(const Tensor& resid, const Tensor& amp, const Tensor& fock, int nocc, int rank,
              int has_alpha, int equation, double alpha, const Tensor& out, double shift = 0.0,
              int sub_singles = 0);
  void dot(double alpha, const Tensor& A, const Tensor& B, double beta, int k);
  void scale_dev(const Tensor& C, double d0, double d1, int k);
  void diag_add(const Tensor& Cmat, double alpha, const Tensor& fock, int64_t foff);
  void rdm1(const Tensor& doo, const Tensor& dvoT, const Tensor& l1, const Tensor& dvv, const Tensor& out);
  void ewise(int sub, const Tensor& a, const Tensor& b, const Tensor& c, double alpha, double beta,
             int64_t i1 = 0, int64_t i2 = 0);

  // ---- INT8-pipe primitives (ozaki.cu)
  // cut X[R, (K1,K2)] (element strides rs, ks1, ks2) into oz_ns digit planes in the workspace
  OzSet oz_cut(const Tensor& X, int64_t R, int64_t rs, int64_t K1, int64_t ks1, int64_t K2, int64_t ks2,
               const std::string& note);
  void oz_release(const OzSet& s);
 private:
  bool written_since(size_t op_index, int slot, int64_t lo, int64_t hi) const;
  void drop_cuts_of(int slot, int64_t lo, int64_t hi);
 public:
  OzSet oz_const_vvvv(int64_t rows) const;     // this rank's shard of vvvv_p: rows x P_v
  OzSet oz_const_ovvv1() const;                // rows (m,a), k = ef_p
  OzSet oz_const_ovvv2() const;                // rows ef_p, k = (m, a)
  // batch of products C_b[m*crs + n*ccs] = alpha sum_k A_b[m,k] B_b[n,k] + beta C_b  (C_b = C + b*c_b);
  // the role assignment (which operand feeds the 128-row side of the tile) is chosen here
  void oz_mm(double alpha, const OzSet& A, const OzSel& a, const OzSet& B, const OzSel& b, int64_t M, int64_t N,
             int64_t batch, double beta, const Tensor& C, int64_t crs, int64_t ccs, int64_t c_b, const std::string& note);

  // ---- cut cache: a large operand view that is cut twice while nothing has written into it in between (t2 / l2 in
  // particle-hole layout feed several ring products) keeps its planes; they are dropped when the source is released.
  struct CutEntry {
    int slot; int64_t off, R, rs, K1, ks1, K2, ks2; int ns;
    int64_t lo, hi;          // element range of the source view
    size_t op_index;         // the OP_OZ_SPLIT that made the planes
    OzSet set;
    int users = 0;           // oz_cut calls not yet matched by oz_release: the planes must stay allocated
  };
  std::vector<CutEntry> cut_cache;
  std::vector<CutEntry> cut_orphans;   // dropped from the cache (source released / overwritten) while still in use
  void retire_cut(size_t i);
  int64_t cut_cache_min_elems = 1 << 20;
  int64_t cut_cache_hits = 0;

  int64_t workspace_elems() const { return arena.peak; }
  std::string dump_json() const;

 private:
  // INT8-pipe route of one unbatched GEMM: X[M,K] (strides ars, aks) . Y[N,K]^T (strides brs, bks)
  void emit_oz(double alpha, const Tensor& A, int64_t ars, int64_t aks, const Tensor& B, int64_t brs, int64_t bks,
               int64_t M, int64_t N, int64_t K, double beta, const Tensor& C, int64_t crs, int64_t ccs,
               const std::string& note);
};

int64_t npair(int64_t n);

}  // namespace ecw
