// ccsd_plan_detail.h — helpers shared by the CCSD plan builders (ccsd_plan.cpp: general variants, rdm1, energy;
// ccsd_plan_slab.cpp: the packed variants with the doubles intermediates distributed over the leading occupied index).
#pragma once
#include <algorithm>

#include "ccsd_plan.h"

namespace ecw {
namespace detail {

struct Slots {
  int64_t o, v, n, po, pv;
  Tensor t1, t2, l1, l2, fsp, fock, out1, out2, rdm1;
  Tensor foo, fov, fvo, fvv;
  Tensor oooo, ooov, oovv, oovv_ph, ovov_ph, ovvv, oooo_p, oovv_p, ovvv_p, ovvv_p2, vvvv_p;
  int rank, world;
  int64_t nshmax, n0, nsh;   // this rank's rows [n0, n0+nsh) of vvvv_p (packed virtual pair index)
  explicit Slots(const Sizes& z) {
    rank = z.rank; world = z.world;
    o = z.nocc; v = z.nvir; n = o + v; po = npair(o); pv = npair(v);
    t1 = make_tensor(S_T1, 0, {o, v});
    t2 = make_tensor(S_T2, 0, {o, o, v, v});
    l1 = make_tensor(S_L1, 0, {o, v});
    l2 = make_tensor(S_L2, 0, {o, o, v, v});
    fsp = make_tensor(S_FSP, 0, {n, n});
    fock = make_tensor(S_FOCK, 0, {n, n});
    out1 = make_tensor(S_OUT1, 0, {o, v});
    out2 = make_tensor(S_OUT2, 0, {o, o, v, v});
    rdm1 = make_tensor(S_RDM1, 0, {n, n});
    foo = block2(fsp, 0, o, 0, o);
    fov = block2(fsp, 0, o, o, v);
    fvo = block2(fsp, o, v, 0, o);
    fvv = block2(fsp, o, v, o, v);
    oooo = make_tensor(S_OOOO, 0, {o, o, o, o});
    ooov = make_tensor(S_OOOV, 0, {o, o, o, v});
    oovv = make_tensor(S_OOVV, 0, {o, o, v, v});
    oovv_ph = make_tensor(S_OOVV_PH, 0, {o, v, o, v});
    ovov_ph = make_tensor(S_OVOV_PH, 0, {o, v, o, v});
    ovvv = make_tensor(S_OVVV, 0, {o, v, v, v});
    oooo_p = make_tensor(S_OOOO_P, 0, {po, po});
    oovv_p = make_tensor(S_OOVV_P, 0, {po, pv});
    ovvv_p = make_tensor(S_OVVV_P, 0, {o, v, pv});
    ovvv_p2 = make_tensor(S_OVVV_P, 0, {o * v, pv});
    nshmax = (pv + world - 1) / world;
    shard_range(pv, rank, world, &n0, &nsh);
    vvvv_p = make_tensor(S_VVVV_P, 0, {nsh, pv});   // local shard (all of it when world == 1)
  }
};

// r2[ijab] += P(ij)P(ab) ring[iajb]; x is an o2v2 scratch.
inline void add_antisym_ph(Plan& P, const Tensor& ring, const Tensor& x, const Tensor& r2) {
  P.permute(1.0, ring, "iajb", 0.0, x, "ijab", "ph->ijab");
  P.permute(-1.0, ring, "jaib", 1.0, x, "ijab", "P(ij)");
  P.axpby(1.0, x, 1.0, r2);
  P.permute(-1.0, x, "ijba", 1.0, r2, "ijab", "P(ab)");
}

// scal[k] = CCSD correlation-energy functional (CCSD.py:236-240 / :608-610)
inline void emit_energy(Plan& P, const Slots& s, const Tensor& fov_dense, int k) {
  P.dot(1.0, fov_dense, s.t1, 0.0, k);
  P.dot(0.25, s.t2, s.oovv, 1.0, k);
  Tensor G = P.tmp({s.o, s.v});
  P.contract(1.0, s.oovv_ph, "menf", s.t1, "nf", 0.0, G, "me");
  P.dot(0.5, s.t1, G, 1.0, k);
  P.release(G);
}

// Wph[(me),(jb)] = Wovvo[m,b,e,j] (CCSD.py:404-413) for the rows m in [m0, m0+nm); `t2x`/`c2` are the
// t2 operand of the o^3v^3 term and its coefficient (the general path passes t2ph2, -1/2).
inline void emit_wovvo_rows(Plan& P, const Slots& s, const Tensor& t1, const Tensor& t2x, double c2, const Tensor& Wph,
                     int64_t m0, int64_t nm) {
  const int64_t o = s.o, v = s.v;
  Tensor Wl = slice0(Wph, m0, nm);
  P.contract(c2, slice0(s.oovv_ph, m0, nm), "menf", t2x, "nfjb", 0.0, Wl, "mejb", "R1 Wovvo");
  P.contract(1.0, slice0(s.ovvv, m0, nm), "mbef", t1, "jf", 1.0, Wl, "mejb");
  // -t1[nb] (oovv[mnef] t1[jf] - ooov[mnje]) (CCSD.py:409-410 and the t1.ooov term): the two o^3v operands are
  // combined first, so that the o^2v^2 result is updated by ONE K = nocc product instead of two
  Tensor U = P.tmp({nm, o, o, v});
  P.axpby(-1.0, slice0(s.ooov, m0, nm), 0.0, U);
  P.contract(1.0, slice0(s.oovv, m0, nm), "mnef", t1, "jf", 1.0, U, "mnje");
  P.contract(-1.0, t1, "nb", U, "mnje", 1.0, Wl, "mejb");
  P.release(U);
  P.axpby(-1.0, slice0(s.ovov_ph, m0, nm), 1.0, Wl);
}

// whole Wph, rows distributed over the ranks and all-gathered once
inline void emit_wovvo(Plan& P, const Slots& s, const Tensor& t1, const Tensor& t2x, double c2, const Tensor& Wph) {
  const int64_t L = s.o, chunk = P.lead_chunk(L);
  int64_t m0, nm;
  P.my_range(L, &m0, &nm);
  if (P.world == 1) {
    emit_wovvo_rows(P, s, t1, t2x, c2, Wph, 0, L);
    return;
  }
  if (nm > 0) emit_wovvo_rows(P, s, t1, t2x, c2, Wph, m0, nm);
  Tensor mine = Wph;
  mine.off = Wph.off + (int64_t)P.rank * chunk * Wph.str[0];
  mine.dim[0] = chunk;
  Tensor full = Wph;
  full.dim[0] = chunk * P.world;
  P.allgather(mine, chunk * Wph.str[0], full, "Wovvo rows");
}


// ---- ovvv-streaming terms on the INT8 pipe from the constant digit planes of ovvv_p (one GPU, nocc, nvir % 8 == 0)
inline bool ovvv_fast(const Plan& P) { return P.ovvv_planes && P.world == 1; }

// out[i,a] += alpha * sum_{m,e,f} amp[i,m,e,f] ovvv[m,a,e,f]      (CCSD.py:294 T1, :585-586 v5, :499-500 L1)
// = alpha * sum_m sum_{e<f} (amp[imef] - amp[imfe]) ovvv_p[(m,a), ef_p]: one product per m over rows of the plane
// set OZ1, partial results summed in a fixed order.
inline void emit_pair_ovvv(Plan& P, const Slots& s, double alpha, const Tensor& amp, const Tensor& out, const char* note) {
  const int64_t o = s.o, v = s.v, pv = s.pv;
  Tensor av = amp;                                   // view [m,i,e,f]
  std::swap(av.dim[0], av.dim[1]);
  std::swap(av.str[0], av.str[1]);
  Tensor Tp = P.tmp({o * o, pv});
  P.pack(1.0, av, 2 | 4, 0.0, Tp);
  OzSet T = P.oz_cut(Tp, o * o, pv, 1, 0, pv, 1, note);
  P.release(Tp);
  Tensor part = P.tmp({o, o, v});                    // [m, i, a]
  OzSel sa, sb;
  sa.rowb = v;                                       // rows (m, a) of OZ1
  sb.rowb = o;                                       // rows (m, i) of the amplitude planes
  P.oz_mm(1.0, P.oz_const_ovvv1(), sa, T, sb, v, o, o, 0.0, part, 1, v, o * v, note);
  P.oz_release(T);
  Op r;
  r.kind = OP_REDUCE;
  r.a = part;
  r.i0 = o;
  r.M = o; r.N = v;
  r.c = out;
  r.i1 = out.str[0]; r.i2 = out.str[1];
  r.alpha = alpha; r.beta = 1.0;
  r.note = std::string(note) + " [sum over m]";
  P.ops.push_back(r);
  P.release(part);
}

// xp[i,j,ab_p] = alpha * sum_e amp1[i,e] ovvv[j,e,a,b]  for a<b   (CCSD.py:311-312, :484-486): one product per j
// over one k1 = j of the plane set OZ2 (rows ab_p, k = (j, e)).
inline void emit_t1_ovvv_packed(Plan& P, const Slots& s, double alpha, const Tensor& amp1, const Tensor& xp, const char* note) {
  const int64_t o = s.o, v = s.v, pv = s.pv;
  OzSet T = P.oz_cut(amp1, o, amp1.str[0], 1, 0, v, amp1.str[1], note);
  OzSel sa, sb;
  sa.k1b = 1; sa.nk1 = 1;                            // k1 = j
  P.oz_mm(alpha, P.oz_const_ovvv2(), sa, T, sb, pv, o, o, 0.0, xp, 1, o * pv, pv, note);
  P.oz_release(T);
}

// r2[ijab] += x[ijab] - x[jiab] with x[ijab] = -sum_e t1[ie] ovvv[jeab] (CCSD.py:311-312), distributed over j
inline void emit_t1_ovvv_term(Plan& P, const Slots& s, const Tensor& t1, const Tensor& x, const Tensor& r2) {
  if (ovvv_fast(P)) {
    Tensor xp = P.tmp({s.o * s.o, s.pv});            // [(i,j), ab_p]
    emit_t1_ovvv_packed(P, s, -1.0, t1, xp, "t1.ovvv (packed pair, INT8)");
    Tensor r2T = r2;
    std::swap(r2T.str[0], r2T.str[1]);
    P.unpack(1.0, xp, 2, 1.0, r2);
    P.unpack(-1.0, xp, 2, 1.0, r2T);
    P.release(xp);
    return;
  }
  if (P.world == 1) {
    P.contract(-1.0, t1, "ie", s.ovvv, "jeab", 0.0, x, "ijab");
    P.axpby(1.0, x, 1.0, r2);
    P.permute(-1.0, x, "jiab", 1.0, r2, "ijab");
    return;
  }
  Tensor xj = P.tmp_lead_padded({s.o, s.o, s.v, s.v});   // xj[j,i,a,b] = x[i,j,a,b]
  P.contract_lead_dist(-1.0, s.ovvv, "jeab", t1, "ie", xj, "jiab", "t1.ovvv (distributed over j)");
  P.permute(1.0, xj, "jiab", 1.0, r2, "ijab");
  P.axpby(-1.0, xj, 1.0, r2);
  P.release(xj);
}

// acc[rows, ab_p] = X[rows, cd_p] . vvvv_p[ab_p, cd_p]^T + beta * acc   (particle-particle ladder).
// With world > 1 every rank multiplies by its row shard of vvvv_p (columns [n0, n0+nsh) of the result);
// the column blocks are all-gathered and assembled.  CCSD.py:305 (K1) and :470 (K2).
inline void ladder_dist(Plan& P, const Slots& s, const Tensor& X, const Tensor& acc, double beta, const char* note) {
  if (s.world == 1) {
    P.contract(1.0, X, "if", s.vvvv_p, "af", beta, acc, "ia", note);
    return;
  }
  const int64_t rows = X.dim[0];
  Tensor accL = P.tmp({rows, s.nshmax});
  Tensor G = P.tmp({(int64_t)s.world, rows, s.nshmax});
  if (s.nsh > 0) {
    Tensor accv = accL;
    accv.dim[1] = s.nsh;
    P.contract(1.0, X, "if", s.vvvv_p, "af", 0.0, accv, "ia", note);
  }
  P.allgather(accL, rows * s.nshmax, G, note);
  for (int r = 0; r < s.world; ++r) {
    int64_t c0, nc;
    shard_range(s.pv, r, s.world, &c0, &nc);
    if (nc <= 0) continue;
    Tensor src = make_tensor(G.slot, G.off + (int64_t)r * rows * s.nshmax, {rows, nc});
    src.str[0] = s.nshmax;
    Tensor dst = acc;
    dst.off = acc.off + c0;
    dst.dim[1] = nc;
    P.permute(1.0, src, "ia", beta, dst, "ia", "ladder shard -> accumulator");
  }
  P.release(G);
  P.release(accL);
}

}  // namespace detail
}  // namespace ecw
