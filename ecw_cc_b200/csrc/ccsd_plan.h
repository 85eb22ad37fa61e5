// ccsd_plan.h — plan builders (host-only) for the CCSD / CCS residual path.
#pragma once
#include "plan.h"

namespace ecw {

struct Sizes {
  int64_t nocc = 0, nvir = 0;
  int rank = 0, world = 1;   // vvvv_p is row-sharded over the packed virtual pair index; heavy GEMMs owner-computes
  // GEMM engine: oz_ns > 0 routes large unbatched GEMMs to the INT8 tcgen05 pipe (ozaki.cu) with oz_ns
  // 7-bit digits when 2MNK >= oz_min_flops (negative: every unbatched GEMM); vvvv_planes: the packed
  // vvvv shard is bound as digit planes ("vvvv_oz"/"vvvv_ozs") instead of FP64 ("vvvv_p")
  int oz_ns = 0;
  double oz_min_flops = 2e10;
  int64_t oz_splitk_min_k = 65536;
  bool vvvv_planes = false;
  // ovvv_p is bound as digit planes in both orientations ("ovvv_oz1/2" + statistics) instead of FP64: R4/R6/R9 skip
  // their per-call cuts and the ovvv-streaming terms with a contracted or free antisymmetric pair run on the INT8
  // pipe as batched products (needs nocc % 8 == 0 and nvir % 8 == 0: sub-blocks start on 8-row groups)
  bool ovvv_planes = false;
  int64_t cut_cache_min_elems = 1 << 20;   // operands at least this large keep their digit planes for a second use
  void apply(Plan& P) const {
    P.rank = rank; P.world = world;
    P.nocc = nocc; P.nvir = nvir;
    P.oz_ns = oz_ns; P.oz_min_flops = oz_min_flops; P.oz_splitk_min_k = oz_splitk_min_k;
    P.vvvv_planes = vvvv_planes && oz_ns > 0;
    P.ovvv_planes = ovvv_planes && oz_ns > 0;
    P.cut_cache_min_elems = cut_cache_min_elems;
  }
};

// mode flags mirror the reference keyword arguments of GCC.tupdate/lupdate
// (CCSD.py:248, :419): has_alpha <=> `alpha is not None`, equation <=> `equation=True`.
void build_ccsd_tupdate(Plan& P, const Sizes& z, int has_alpha, int equation);
void build_ccsd_lupdate(Plan& P, const Sizes& z, int has_alpha, int equation);
// general variants: amplitudes not assumed antisymmetric (only the integrals are)
void build_ccsd_tupdate_general(Plan& P, const Sizes& z, int has_alpha, int equation);
void build_ccsd_lupdate_general(Plan& P, const Sizes& z, int has_alpha, int equation);
void build_ccsd_gamma(Plan& P, const Sizes& z);
void build_ccsd_energy(Plan& P, const Sizes& z);
// ECW-CCS intermediates (csrc/ccs_plan.cpp; CCS.py:271-312, :490-537, :774-872, :1164-1234)
void build_ccs_t1inter(Plan& P, const Sizes& z);
void build_ccs_l1inter(Plan& P, const Sizes& z, int e_term);
void build_ccs_r1inter(Plan& P, const Sizes& z, int has_vm);
void build_ccs_esl1inter(Plan& P, const Sizes& z, int has_vm);

}  // namespace ecw
