// ccsd_plan.cpp — plan builders for the spin-orbital CCSD residual path: the
// general T / Lambda variants (amplitudes not assumed antisymmetric), the rdm1
// (gamma) and the energy.  The T / Lambda plans for antisymmetric amplitudes
// are built in ccsd_plan_slab.cpp.
//
// Each builder states the reference equations as binary contractions over the
// constant integral layouts of the eris container; the contraction list is
// the one proven equal to the reference in oracle/refactored_np.py (same index
// strings, same order).  Reference: CCSD.py:248-338 (tupdate), :346-413
// (T intermediates), :419-535 (lupdate), :543-623 (Linter), :136-182 (rdm1),
// :224-242 (energy).  Differences from the reference factorisation, all exact
// identities (DESIGN.md "Algorithm"):
//   * Wvvvv (CCSD.py:396-402) is never formed: its tau.oovv part is folded into
//     Woooo (coefficient 1/4 -> 1/2), its t1.ovvv part becomes Y[ijma].t1;
//   * wvvvo (CCSD.py:602-605) is never formed: each of its four pieces is
//     contracted with l2 first;
//   * the two particle-particle ladders and the hole-hole ladder contract
//     antisymmetry-packed integral pairs  p(a<b) = b(b-1)/2 + a;
//   * ring terms run in the particle-hole layout X[(ia),(jb)].
#include "ccsd_plan_detail.h"

#include <algorithm>

namespace ecw {

using namespace detail;

void build_ccsd_energy(Plan& P, const Sizes& z) {
  z.apply(P);
  Slots s(z);
  Tensor f = P.tmp({s.o, s.v});
  P.axpby(1.0, s.fov, 0.0, f);
  emit_energy(P, s, f, 0);
  P.release(f);
}

// ======================================================================
// GENERAL variants: only the antisymmetry of the INTEGRALS (Eris.py:128) is
// used, never that of t2/l2.  Needed because the reference's L1 update
// (utilities.py:59-67, Q1: v<=0 is soft-thresholded, v>0 gets e+alpha) breaks
// the antisymmetry of the doubles amplitudes, and its dense einsums are then
// evaluated on the non-antisymmetric tensors.  Contracted integral pairs are
// still packed (the amplitude is antisymmetrised while packing), the (i,j)
// rows of the ladders stay dense.  Spec: oracle/refactored_np.py *_general.
// ======================================================================
void build_ccsd_tupdate_general(Plan& P, const Sizes& z, int has_alpha, int equation) {
  z.apply(P);
  Slots s(z);
  const int64_t o = s.o, v = s.v, po = s.po, pv = s.pv, oo = o * o, vv = v * v;
  const bool shift = !equation && !has_alpha;
  const Tensor &t1 = s.t1, &t2 = s.t2, &r1 = s.out1, &r2 = s.out2;

  Tensor tau = P.tmp({o, o, v, v});
  P.tau(t2, t1, 1.0, 1.0, tau);
  Tensor tau_q = P.tmp({oo, pv});          // [(ij), ef_p] = 1/2 (tau[ijef]-tau[ijfe])
  P.pack(0.5, tau, 2 | 4, 0.0, tau_q);
  Tensor tau_r = P.tmp({po, vv});          // [mn_p, (ab)] = 1/2 (tau[mnab]-tau[nmab])
  P.pack(0.5, tau, 1 | 8, 0.0, tau_r);
  P.release(tau);
  Tensor ttl = P.tmp({o, o, v, v});
  P.tau(t2, t1, 0.5, 0.5, ttl);
  Tensor t2ph = P.tmp({o, v, o, v});
  P.permute(1.0, t2, "ijab", 0.0, t2ph, "iajb", "t2 ph layout");

  Tensor Fov = P.tmp({o, v});
  P.axpby(1.0, s.fov, 0.0, Fov);
  P.contract(1.0, s.oovv_ph, "menf", t1, "nf", 1.0, Fov, "me", "cc_Fov");
  Tensor Fvv = P.tmp({v, v});
  P.axpby(1.0, s.fvv, 0.0, Fvv);
  P.contract(-0.5, s.fov, "me", t1, "ma", 1.0, Fvv, "ae", "cc_Fvv");
  P.contract_split(-1.0, s.ovvv, "maef", t1, "mf", Fvv, "ae", 'm', "cc_Fvv vovv");
  P.contract(0.5, ttl, "mnaf", s.oovv, "mnfe", 1.0, Fvv, "ae", "cc_Fvv tau~");
  Tensor Foo = P.tmp({o, o});
  P.axpby(1.0, s.foo, 0.0, Foo);
  P.contract(0.5, s.fov, "me", t1, "ie", 1.0, Foo, "mi", "cc_Foo");
  P.contract(1.0, s.ooov, "mnie", t1, "ne", 1.0, Foo, "mi", "cc_Foo ooov");
  P.contract(0.5, s.oovv, "mnef", ttl, "inef", 1.0, Foo, "mi", "cc_Foo tau~");
  P.release(ttl);
  if (shift) {
    P.diag_add(Fvv, -1.0, s.fock, o);
    P.diag_add(Foo, -1.0, s.fock, 0);
  }

  P.axpby(1.0, s.fov, 0.0, r1);
  P.contract(1.0, t1, "ie", Fvv, "ae", 1.0, r1, "ia");
  P.contract(-1.0, Foo, "mi", t1, "ma", 1.0, r1, "ia");
  P.contract(1.0, t2ph, "iame", Fov, "me", 1.0, r1, "ia");
  P.contract(-1.0, s.ovov_ph, "ianf", t1, "nf", 1.0, r1, "ia");
  if (ovvv_fast(P)) emit_pair_ovvv(P, s, -0.5, t2, r1, "T1 ovvv");
  else P.contract_split(-0.5, t2, "imef", s.ovvv, "maef", r1, "ia", 'm', "T1 ovvv");
  P.contract(-0.5, t2, "mnae", s.ooov, "mnie", 1.0, r1, "ia");

  Tensor x = P.tmp({o, o, v, v});
  Tensor F1 = P.tmp({v, v});
  P.axpby(1.0, Fvv, 0.0, F1);
  P.contract(-0.5, t1, "mb", Fov, "me", 1.0, F1, "be");
  P.contract(1.0, t2, "ijae", F1, "be", 0.0, x, "ijab");
  P.axpby(1.0, s.oovv, 0.0, r2);
  P.axpby(1.0, x, 1.0, r2);
  P.permute(-1.0, x, "ijba", 1.0, r2, "ijab");
  P.release(F1);
  Tensor F2 = P.tmp({o, o});
  P.axpby(1.0, Foo, 0.0, F2);
  P.contract(0.5, t1, "je", Fov, "me", 1.0, F2, "mj");
  P.contract(1.0, F2, "mj", t2, "imab", 0.0, x, "ijab");
  P.axpby(-1.0, x, 1.0, r2);
  P.permute(1.0, x, "jiab", 1.0, r2, "ijab");
  P.release(F2);

  // hole-hole ladder: W[mn_p,(ij)] (first pair antisymmetric through the integrals), dense output
  Tensor w4 = P.tmp({o, o, o, o});
  P.contract(1.0, s.ooov, "mnie", t1, "je", 0.0, w4, "mnij");
  Tensor w4a = P.tmp({o, o, o, o});
  P.axpby(1.0, s.oooo, 0.0, w4a);
  P.axpby(1.0, w4, 1.0, w4a);
  P.permute(-1.0, w4, "mnji", 1.0, w4a, "mnij");
  P.release(w4);
  Tensor Woo_p = P.tmp({po, oo});
  P.pack(1.0, w4a, 1, 0.0, Woo_p);
  P.release(w4a);
  P.contract(1.0, s.oovv_p, "mf", tau_q, "if", 1.0, Woo_p, "mi", "Woooo tau.oovv (K3 folded)");
  P.contract(1.0, Woo_p, "mi", tau_r, "ma", 1.0, reshape(r2, {oo, vv}), "ia", "hh ladder");
  P.release(Woo_p);
  P.release(tau_r);
  // particle-particle ladder + t1.ovvv part of Wvvvv: [(ij), ab_p]
  Tensor acc_q = P.tmp({oo, pv});
  ladder_dist(P, s, tau_q, acc_q, 0.0, "K1 pp ladder (general)");
  Tensor Z = P.tmp({oo, v, v});
  if (P.world == 1) {
    Tensor Y_q = P.tmp({oo, o * v});
    P.contract(-2.0, tau_q, "if", s.ovvv_p2, "qf", 0.0, Y_q, "iq", "R9 Y[ijma]");
    P.contract(1.0, reshape(Y_q, {oo, o, v}), "pma", t1, "mb", 0.0, Z, "pab");
    P.release(Y_q);
  } else {
    Tensor YT = P.tmp_lead_padded({o, v, oo});
    P.contract_lead_dist(-2.0, s.ovvv_p, "maf", tau_q, "if", YT, "mai", "R9 Y[ijma]");
    P.contract(1.0, YT, "map", t1, "mb", 0.0, Z, "pab");
    P.release(YT);
  }
  P.release(tau_q);
  P.pack(-0.5, reshape(Z, {oo, 1, v, v}), 2 | 4, 1.0, acc_q);
  P.release(Z);
  P.unpack(1.0, acc_q, 2, 1.0, r2);
  P.release(acc_q);

  // ring; t2ph2[(nf),(jb)] = t2[j,n,f,b]
  Tensor t2ph2 = P.tmp({o, v, o, v});
  P.permute(1.0, t2, "jnfb", 0.0, t2ph2, "nfjb", "t2 ph2 layout");
  Tensor Wph = P.tmp_lead_padded({o, v, o, v});
  emit_wovvo(P, s, t1, t2ph2, -0.5, Wph);
  P.release(t2ph2);
  Tensor ring = P.tmp_lead_padded({o, v, o, v});
  P.contract_lead_dist(1.0, t2ph, "iame", Wph, "mejb", ring, "iajb", "R2 ring");
  P.release(Wph);
  Tensor Q = P.tmp({o, v, o, o});
  P.contract(1.0, s.ovov_ph, "jbme", t1, "ie", 0.0, Q, "jbmi");
  P.contract(1.0, t1, "ma", Q, "jbmi", 1.0, ring, "iajb");
  P.release(Q);
  add_antisym_ph(P, ring, x, r2);
  P.release(ring);
  P.release(t2ph);

  emit_t1_ovvv_term(P, s, t1, x, r2);
  P.contract(1.0, t1, "ma", s.ooov, "ijmb", 0.0, x, "ijab");
  P.axpby(-1.0, x, 1.0, r2);
  P.permute(1.0, x, "ijba", 1.0, r2, "ijab");
  P.release(x);
  P.release(Fov);
  P.release(Fvv);
  P.release(Foo);

  P.finish(r1, t1, s.fock, (int)o, 2, has_alpha, equation, 0.0, r1);
  P.finish(r2, t2, s.fock, (int)o, 4, has_alpha, equation, 0.0, r2);
}

void build_ccsd_lupdate_general(Plan& P, const Sizes& z, int has_alpha, int equation) {
  z.apply(P);
  Slots s(z);
  const int64_t o = s.o, v = s.v, po = s.po, pv = s.pv, oo = o * o, vv = v * v;
  const bool shift = !equation && !has_alpha;
  const Tensor &t1 = s.t1, &t2 = s.t2, &l1 = s.l1, &l2 = s.l2, &r1 = s.out1, &r2 = s.out2;

  Tensor tau = P.tmp({o, o, v, v});
  P.tau(t2, t1, 2.0, 0.0, tau);                          // CCSD.py:565 exactly
  Tensor tau_q = P.tmp({oo, pv});
  P.pack(0.5, tau, 2 | 4, 0.0, tau_q);
  Tensor l2_q = P.tmp({oo, pv});
  P.pack(0.5, l2, 2 | 4, 0.0, l2_q);
  Tensor t2ph = P.tmp({o, v, o, v});
  P.permute(1.0, t2, "ijab", 0.0, t2ph, "iajb", "t2 ph layout");

  Tensor Fov = P.tmp({o, v});
  P.axpby(1.0, s.fov, 0.0, Fov);
  P.contract(1.0, s.oovv_ph, "menf", t1, "nf", 1.0, Fov, "me");
  Tensor v1 = P.tmp({v, v});
  P.axpby(1.0, s.fvv, 0.0, v1);
  P.contract(-1.0, s.fov, "ja", t1, "jb", 1.0, v1, "ba");
  P.contract_split(-1.0, s.ovvv, "jbac", t1, "jc", v1, "ba", 'j', "v1 ovvv");
  P.contract(0.5, s.oovv, "jkca", tau, "jkbc", 1.0, v1, "ba");
  Tensor v2 = P.tmp({o, o});
  P.axpby(1.0, s.foo, 0.0, v2);
  P.contract(1.0, s.fov, "ib", t1, "jb", 1.0, v2, "ij");
  P.contract(-1.0, s.ooov, "kijb", t1, "kb", 1.0, v2, "ij");
  P.contract(0.5, s.oovv, "ikbc", tau, "jkbc", 1.0, v2, "ij");
  // dense l2.tau (no symmetry left): lt[ij,kl]
  Tensor lt = P.tmp({o, o, o, o});
  P.contract(1.0, l2, "ijcd", tau, "klcd", 0.0, lt, "ijkl", "l2.tau (dense)");
  P.release(tau);

  Tensor v4ph = P.tmp_lead_padded({o, v, o, v});
  P.contract_lead_dist(1.0, t2ph, "kcld", s.oovv_ph, "ldjb", v4ph, "kcjb", "R3 v4");
  P.axpby(-1.0, s.ovov_ph, 1.0, v4ph);

  Tensor v5T = P.tmp({o, v});
  P.permute(1.0, s.fvo, "bj", 0.0, v5T, "jb");
  P.contract(1.0, t2ph, "jbkc", s.fov, "kc", 1.0, v5T, "jb");
  Tensor q = P.tmp({o, o});
  P.contract(1.0, Fov, "kc", t1, "jc", 0.0, q, "kj");
  P.contract(1.0, q, "kj", t1, "kb", 1.0, v5T, "jb");
  P.release(q);
  P.contract(-0.5, s.ooov, "kljc", t2, "klbc", 1.0, v5T, "jb");
  if (ovvv_fast(P)) emit_pair_ovvv(P, s, -0.5, t2, v5T, "v5 ovvv");
  else P.contract_split(-0.5, t2, "jkdc", s.ovvv, "kbdc", v5T, "jb", 'k', "v5 ovvv");

  Tensor w3T = P.tmp({o, v});
  P.axpby(1.0, v5T, 0.0, w3T);
  P.release(v5T);
  P.contract(1.0, v4ph, "kcjb", t1, "jb", 1.0, w3T, "kc");
  P.contract(1.0, t1, "kb", v1, "cb", 1.0, w3T, "kc");
  P.contract(-1.0, v2, "jk", t1, "jc", 1.0, w3T, "kc");

  // woooo packed on its (integral-)antisymmetric first pair: [ij_p, (kl)]
  Tensor y4 = P.tmp({o, o, o, o});
  P.axpby(0.5, s.oooo, 0.0, y4);
  P.contract(1.0, s.ooov, "jilc", t1, "kc", 1.0, y4, "jilk");
  Tensor woo_p = P.tmp({po, oo});
  P.pack(1.0, y4, 1, 0.0, woo_p);
  P.release(y4);
  P.contract(0.5, s.oovv_p, "if", tau_q, "kf", 1.0, woo_p, "ik", "v3");

  Tensor S = P.tmp({o, o, o, v});
  P.axpby(-1.0, s.ooov, 0.0, S);
  P.contract(1.0, s.oovv, "ljbd", t1, "kd", 1.0, S, "ljkb");
  Tensor wph = P.tmp({o, v, o, v});
  P.axpby(1.0, v4ph, 0.0, wph);
  P.contract(1.0, t1, "lc", S, "ljkb", 1.0, wph, "kcjb");
  P.release(S);
  if (P.world == 1) {
    P.contract(1.0, s.ovvv, "jcbd", t1, "kd", 1.0, wph, "kcjb");
  } else {
    Tensor wj = P.tmp_lead_padded({o, v, v, o});
    P.contract_lead_dist(1.0, s.ovvv, "jcbd", t1, "kd", wj, "jcbk", "wovvo ovvv.t1 (distributed over j)");
    P.permute(1.0, wj, "jcbk", 1.0, wph, "kcjb");
    P.release(wj);
  }

  Tensor wovoo = P.tmp_lead_padded({o, v, o, o});
  {
    Tensor w3d = wovoo;           // [i, c, (jk)]
    w3d.nd = 3;
    w3d.dim[2] = oo;
    w3d.str[2] = 1;
    P.contract_lead_dist(0.5, s.ovvv_p, "icf", tau_q, "kf", w3d, "ick", "R4 wovoo");
  }
  P.release(tau_q);
  P.permute(0.5, s.ooov, "jkic", 1.0, wovoo, "icjk");
  P.contract(1.0, v4ph, "kcib", t1, "jb", 1.0, wovoo, "icjk");
  P.contract(-1.0, t2ph, "kclb", s.ooov, "lijb", 1.0, wovoo, "icjk", "wovoo ooov.t2");

  // ---- m3 dense [ij,ab]
  Tensor m3 = P.tmp({o, o, v, v});
  Tensor m3a = P.tmp({po, vv});
  P.contract(1.0, woo_p, "ik", reshape(l2, {oo, vv}), "ka", 0.0, m3a, "ia", "l2.woooo");
  P.release(woo_p);
  P.unpack(1.0, m3a, 1, 0.0, m3);
  P.release(m3a);
  Tensor ltp = P.tmp({oo, po});
  P.pack(1.0, lt, 2 | 4, 0.0, ltp);
  Tensor acc_q = P.tmp({oo, pv});
  P.contract(0.25, ltp, "ik", s.oovv_p, "ka", 0.0, acc_q, "ia");
  P.release(ltp);
  Tensor l2t1 = P.tmp({o, o, v, o});
  P.contract(1.0, l2, "ijcd", t1, "kd", 0.0, l2t1, "ijck");
  Tensor a_q = P.tmp({o, o, o, v});
  P.permute(1.0, l2t1, "ijck", 0.0, a_q, "ijkc");
  P.release(l2t1);
  if (P.world == 1) {
    P.contract(1.0, reshape(a_q, {oo, o * v}), "pq", s.ovvv_p2, "qa", 1.0, acc_q, "pa", "R6 ovvv.(l2 t1)");
  } else {
    Tensor r6 = P.tmp_lead_padded({oo, pv});
    P.contract_lead_dist(1.0, reshape(a_q, {oo, o * v}), "pq", s.ovvv_p2, "qa", r6, "pa", "R6 ovvv.(l2 t1)");
    P.axpby(1.0, r6, 1.0, acc_q);
    P.release(r6);
  }
  P.release(a_q);
  ladder_dist(P, s, l2_q, acc_q, 1.0, "K2 pp ladder (general)");
  P.release(l2_q);
  P.unpack(1.0, acc_q, 2, 1.0, m3);
  P.release(acc_q);

  Tensor m_vv = P.tmp({v, v});
  P.contract(0.5, t2, "klcb", l2, "klca", 0.0, m_vv, "ba");
  Tensor m_oo = P.tmp({o, o});
  P.contract(0.5, l2, "kicd", t2, "kjcd", 0.0, m_oo, "ij");
  Tensor x_vv = P.tmp({v, v});
  P.axpby(1.0, m_vv, 0.0, x_vv);
  P.contract(1.0, l1, "ka", t1, "kb", 1.0, x_vv, "ba");
  Tensor x_oo = P.tmp({o, o});
  P.axpby(1.0, m_oo, 0.0, x_oo);
  P.contract(1.0, l1, "ic", t1, "kc", 1.0, x_oo, "ik");
  if (shift) {
    P.diag_add(v1, -1.0, s.fock, o);
    P.diag_add(v2, -1.0, s.fock, 0);
  }

  // ---- L2
  P.axpby(1.0, s.oovv, 0.0, r2);
  P.axpby(1.0, m3, 1.0, r2);
  Tensor l2ph2 = P.tmp({o, v, o, v});      // [(ia),(kc)] = l2[k,i,c,a]
  P.permute(1.0, l2, "kica", 0.0, l2ph2, "iakc", "l2 ph2 layout");
  Tensor ring = P.tmp_lead_padded({o, v, o, v});
  P.contract_lead_dist(1.0, l2ph2, "iakc", wph, "kcjb", ring, "iajb", "R7 ring");
  P.release(wph);
  P.contract(1.0, l1, "ia", Fov, "jb", 1.0, ring, "iajb");
  Tensor y = P.tmp({o, o, v, v});
  add_antisym_ph(P, ring, y, r2);
  P.release(ring);
  P.contract(1.0, l1, "ka", s.ooov, "ijkb", 0.0, y, "ijab");
  P.contract(1.0, l2, "ijca", v1, "cb", 1.0, y, "ijab");
  P.contract(-1.0, s.oovv, "ijbc", x_vv, "ca", 1.0, y, "ijab");     // oovv[ijcb] = -oovv[ijbc] (Eris.py:128)
  P.axpby(-1.0, y, 1.0, r2);
  P.permute(1.0, y, "ijba", 1.0, r2, "ijab");
  if (ovvv_fast(P)) {
    // y[pqrs] = sum_c l1[qc] ovvv[pcrs]: yp[q,p,rs_p] from the planes, expanded with the (p,q) view of y
    Tensor yp = P.tmp({o * o, s.pv});
    emit_t1_ovvv_packed(P, s, 1.0, l1, yp, "l1.ovvv (packed pair, INT8)");
    Tensor yT = y;
    std::swap(yT.str[0], yT.str[1]);
    P.unpack(1.0, yp, 2, 0.0, yT);
    P.release(yp);
  } else if (P.world == 1) {
    P.contract(1.0, l1, "qc", s.ovvv, "pcrs", 0.0, y, "pqrs");
  } else {
    Tensor yp = P.tmp_lead_padded({o, o, v, v});
    P.contract_lead_dist(1.0, s.ovvv, "pcrs", l1, "qc", yp, "pqrs", "l1.ovvv (distributed over p)");
    P.axpby(1.0, yp, 0.0, y);
    P.release(yp);
  }
  P.contract(1.0, v2, "qk", l2, "kprs", 1.0, y, "pqrs");
  P.contract(-1.0, x_oo, "pk", s.oovv, "kqrs", 1.0, y, "pqrs");
  P.axpby(1.0, y, 1.0, r2);
  P.permute(-1.0, y, "qprs", 1.0, r2, "pqrs");
  P.release(y);

  // ---- L1
  P.axpby(1.0, s.fov, 0.0, r1);
  P.contract(-1.0, s.ovov_ph, "jbia", l1, "jb", 1.0, r1, "ia");
  P.contract(1.0, l1, "ib", v1, "ba", 1.0, r1, "ia");
  P.contract(-1.0, v2, "ij", l1, "ja", 1.0, r1, "ia");
  P.contract(-1.0, wovoo, "icjk", l2, "kjca", 1.0, r1, "ia");
  P.release(wovoo);
  Tensor l2t1b = P.tmp({o, o, v, o});
  P.contract(1.0, l2, "ikbc", t1, "jb", 0.0, l2t1b, "ikcj");
  P.contract(-1.0, l2t1b, "ikcj", v4ph, "kcja", 1.0, r1, "ia", "wvvvo: v4.t1");
  P.release(l2t1b);
  P.release(v4ph);
  P.contract(-0.25, lt, "ikjl", s.ooov, "jlka", 1.0, r1, "ia", "wvvvo: ooov.tau");
  P.release(lt);
  if (ovvv_fast(P)) emit_pair_ovvv(P, s, -0.5, l2, r1, "wvvvo: ovvv");
  else P.contract_split(-0.5, l2, "ikbc", s.ovvv, "kabc", r1, "ia", 'k', "wvvvo: ovvv");
  Tensor l2ph = P.tmp({o, v, o, v});
  P.permute(1.0, l2, "ijab", 0.0, l2ph, "iajb", "l2 ph layout");
  Tensor Xph = P.tmp_lead_padded({o, v, o, v});
  P.contract_lead_dist(1.0, l2ph, "ibjc", t2ph, "jckd", Xph, "ibkd", "R8 l2.t2");
  P.release(l2ph);
  P.contract_split(1.0, Xph, "ibkd", s.ovvv, "kbda", r1, "ia", 'k', "wvvvo: ovvv.t2 (K4 refactored)");
  P.release(Xph);
  P.contract(1.0, m3, "ijab", t1, "jb", 1.0, r1, "ia");
  P.release(m3);
  P.contract(1.0, l2ph2, "iajb", w3T, "jb", 1.0, r1, "ia");
  P.release(l2ph2);
  Tensor zz = P.tmp({o, v});
  P.axpby(1.0, t1, 0.0, zz);
  P.contract(1.0, t2ph, "kcjb", l1, "kc", 1.0, zz, "jb");
  P.release(t2ph);
  P.contract(-1.0, x_vv, "bd", t1, "jd", 1.0, zz, "jb");
  P.contract(-1.0, m_oo, "lj", t1, "lb", 1.0, zz, "jb");
  P.contract(1.0, s.oovv_ph, "iajb", zz, "jb", 1.0, r1, "ia");
  P.release(zz);
  P.contract_split(-1.0, s.ovvv, "icba", x_vv, "bc", r1, "ia", 'c', "L1 ovvv.x_vv");
  P.contract(-1.0, s.ooov, "jika", x_oo, "kj", 1.0, r1, "ia");
  P.contract(-1.0, m_oo, "ik", Fov, "ka", 1.0, r1, "ia");
  P.contract(-1.0, m_vv, "ca", Fov, "ic", 1.0, r1, "ia");

  if (shift) {
    Tensor f = P.tmp({o, v});
    P.axpby(1.0, s.fov, 0.0, f);
    emit_energy(P, s, f, 0);
    P.release(f);
    P.scale_dev(r1, 1.0, -1.0, 0);
    P.scale_dev(r2, 1.0, -1.0, 0);
  }
  P.release(Fov); P.release(v1); P.release(v2); P.release(w3T);
  P.release(m_vv); P.release(m_oo); P.release(x_vv); P.release(x_oo);

  P.finish(r1, l1, s.fock, (int)o, 2, has_alpha, equation, 0.0, r1);
  P.finish(r2, l2, s.fock, (int)o, 4, has_alpha, equation, 0.0, r2);
}

void build_ccsd_gamma(Plan& P, const Sizes& z) {
  z.apply(P);
  Slots s(z);
  const int64_t o = s.o, v = s.v;
  const Tensor &t1 = s.t1, &t2 = s.t2, &l1 = s.l1, &l2 = s.l2;
  // gamma_inter, CCSD.py:165-182.  The three products over the doubles run on this rank's part of an occupied index
  // (no symmetry of the amplitudes is used: the rdm1 is also taken of L1-regularised, non-antisymmetric amplitudes)
  // and are summed over ranks in a fixed order.
  int64_t i0, ni;
  P.my_range(o, &i0, &ni);
  Tensor D = P.tmp({o, o});
  P.fill(D, 0.0);
  Tensor dvv = P.tmp({v, v});
  P.fill(dvv, 0.0);
  Tensor dvoT = P.tmp({o, v});
  P.axpby(1.0, t1, 0.0, dvoT);
  {
    Tensor p = P.tmp({o, o});
    P.fill(p, 0.0);
    if (ni > 0) P.contract(1.0, slice_dim(l2, 1, i0, ni), "imef", slice_dim(t2, 1, i0, ni), "jmef", 1.0, p, "ij", "rdm1 oo");
    P.sum_ranks_add(p, D, "rdm1 oo");
    P.release(p);
    Tensor q = P.tmp({v, v});
    P.fill(q, 0.0);
    if (ni > 0) P.contract(0.5, slice0(t2, i0, ni), "mnea", slice0(l2, i0, ni), "mneb", 1.0, q, "ab", "rdm1 vv");
    P.sum_ranks_add(q, dvv, "rdm1 vv");
    P.release(q);
    Tensor r = P.tmp({o, v});
    P.fill(r, 0.0);
    if (ni > 0) P.contract(1.0, slice0(t2, i0, ni), "imae", l1, "me", 1.0, slice0(r, i0, ni), "ia", "rdm1 vo");
    P.sum_ranks_add(r, dvoT, "rdm1 vo");
    P.release(r);
  }
  Tensor doo = P.tmp({o, o});
  P.axpby(-0.5, D, 0.0, doo);
  P.contract(-1.0, l1, "ie", t1, "je", 1.0, doo, "ij");
  P.contract(1.0, t1, "ma", l1, "mb", 1.0, dvv, "ab");
  P.contract(-0.5, D, "mi", t1, "ma", 1.0, dvoT, "ia");
  P.contract(-1.0, t1, "ie", dvv, "ae", 1.0, dvoT, "ia");
  P.rdm1(doo, dvoT, l1, dvv, s.rdm1);   // CCSD.py:154-160
  P.release(D); P.release(doo); P.release(dvv); P.release(dvoT);
}

}  // namespace ecw
