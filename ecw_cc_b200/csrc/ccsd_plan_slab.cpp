// ccsd_plan_slab.cpp — the packed (antisymmetric-amplitude) T and Lambda plans.
//
// The contractions of oracle/refactored_np.py (reference: CCSD.py:248-338 tupdate, :346-413 T intermediates, :419-535
// lupdate, :543-623 Linter), organised so that every o^2v^2-sized piece of work is done on a SLAB — the rows
// [i0, i0+ni) of the leading occupied index that belong to this rank — and only small or packed tensors are replicated:
//
//   * The amplitudes are replicated INPUTS, so any layout or slice of them (t2ph, l2ph, packed pairs, slabs) is
//     produced locally at HBM speed; nothing of them is ever exchanged.
//   * All contributions to the doubles residual that carry an antisymmetriser are collected in ONE slab tensor z,
//         R2 = oovv (+ m3) + P(ij)P(ab) z + unpack(packed ladder terms),
//     using  X - X^(ab) = 1/2 P(ij)P(ab) X  for X antisymmetric in (ij)  (and the mirror statement), and the freedom to
//     enter a term as X or as X^(ji)(ba): every product can then be formed with ITS distributed index leading —
//     ring products as column slabs  ring^T[(j in slab, b),(i,a)],  ovvv products on the rank's own rows of ovvv.
//     z is all-gathered once (2 GB at (40,400)) and one fused kernel (OP_ASYM4) applies the antisymmetriser.
//   * One-body intermediates and the singles residual are sums of slab contributions: partial results (o x v, v x v,
//     o x o) are summed over ranks in a fixed order (sum_ranks_add).
//   * The only exchanged o^2v^2 intermediate besides z is the ovvv.t1 part of Wovvo, which is produced on rows m of
//     ovvv but consumed on columns j: an all-to-all of 1/world of it (OP_ALLTOALL).
// With one rank the slab is everything and the collectives vanish; the gain there is the fused antisymmetriser
// (one pass over z instead of a dozen permute passes).
#include "ccsd_plan_detail.h"

namespace ecw {

using namespace detail;

namespace {

struct Slab {
  int64_t i0 = 0, ni = 0, chunk = 0;
  int world = 1, rank = 0;
  explicit Slab(const Plan& P, int64_t o) : world(P.world), rank(P.rank) {
    chunk = P.lead_chunk(o);
    P.my_range(o, &i0, &ni);
  }
  Tensor rows(const Tensor& t) const { return slice0(t, i0, ni); }            // leading index in the slab
  Tensor at(const Tensor& t, int d) const { return slice_dim(t, d, i0, ni); }  // index d in the slab
};

// all-gather of a tensor whose leading extent is padded to world * chunk rows (tmp_lead_padded)
void gather_rows(Plan& P, const Slab& g, const Tensor& full, const char* note) {
  if (P.world == 1) return;
  Tensor mine = full;
  mine.off = full.off + (int64_t)P.rank * g.chunk * full.str[0];
  mine.dim[0] = g.chunk;
  Tensor all = full;
  all.dim[0] = g.chunk * P.world;
  P.allgather(mine, g.chunk * full.str[0], all, note);
}

// out[i,a] += alpha * sum_{m in [m0,m0+nm)} sum_{e,f} amp[i,m,e,f] ovvv[m,a,e,f]   (CCSD.py:294, :585-586, :499-500)
// from the constant digit planes OZ1 (rows (m,a), k = ef_p): one product per m, partial results summed in order.
void pair_ovvv_rows(Plan& P, const Slots& s, double alpha, const Tensor& amp, const Tensor& out, int64_t m0, int64_t nm,
                    const char* note) {
  const int64_t o = s.o, v = s.v, pv = s.pv;
  Tensor av = amp;                                   // view [m,i,e,f]
  std::swap(av.dim[0], av.dim[1]);
  std::swap(av.str[0], av.str[1]);
  av = slice0(av, m0, nm);
  Tensor Tp = P.tmp({nm * o, pv});
  P.pack(1.0, av, 2 | 4, 0.0, Tp);
  OzSet T = P.oz_cut(Tp, nm * o, pv, 1, 0, pv, 1, note);
  P.release(Tp);
  Tensor part = P.tmp({nm, o, v});                   // [m, i, a]
  OzSel sa, sb;
  sa.row0 = m0 * v;                                  // rows (m, a) of OZ1, m from m0
  sa.rowb = v;
  sb.rowb = o;                                       // rows (m, i) of the amplitude planes
  P.oz_mm(1.0, P.oz_const_ovvv1(), sa, T, sb, v, o, nm, 0.0, part, 1, v, o * v, note);
  P.oz_release(T);
  Op r;
  r.kind = OP_REDUCE;
  r.a = part;
  r.i0 = nm;
  r.M = o; r.N = v;
  r.c = out;
  r.i1 = out.str[0]; r.i2 = out.str[1];
  r.alpha = alpha; r.beta = 1.0;
  r.note = std::string(note) + " [sum over m]";
  P.ops.push_back(r);
  P.release(part);
}

// xp[j - j0, i, ab_p] = alpha * sum_e amp1[i,e] ovvv[j,e,a,b], a < b, j in [j0, j0+nj)   (CCSD.py:311-312, :484-486):
// one product per j over the single k1 = j of the plane set OZ2 (rows ab_p, k = (j, e)).
void t1_ovvv_rows(Plan& P, const Slots& s, double alpha, const Tensor& amp1, const Tensor& xp, int64_t j0, int64_t nj,
                  const char* note) {
  const int64_t o = s.o, v = s.v, pv = s.pv;
  OzSet T = P.oz_cut(amp1, o, amp1.str[0], 1, 0, v, amp1.str[1], note);
  OzSel sa, sb;
  sa.k10 = j0; sa.k1b = 1; sa.nk1 = 1;               // k1 = j
  P.oz_mm(alpha, P.oz_const_ovvv2(), sa, T, sb, pv, o, nj, 0.0, xp, 1, pv, o * pv, note);
  P.oz_release(T);
}

}  // namespace

// ======================================================================================================= T1 / T2
void build_ccsd_tupdate(Plan& P, const Sizes& z, int has_alpha, int equation) {
  z.apply(P);
  Slots s(z);
  const int64_t o = s.o, v = s.v, po = s.po, pv = s.pv;
  const bool shift = !equation && !has_alpha;  // CCSD.py:283-285
  const Tensor &t1 = s.t1, &t2 = s.t2, &r1 = s.out1, &r2 = s.out2;
  const Slab g(P, o);
  const int64_t i0 = g.i0, ni = g.ni, W = P.world;
  const bool planes = P.ovvv_planes;
  const bool mine = ni > 0;

  // ---- replicated (cheap, from the replicated inputs): packed tau, ph layout of t2
  Tensor tau = P.tmp({o, o, v, v});
  P.tau(t2, t1, 1.0, 1.0, tau);                                   // make_tau, CCSD.py:346-353
  Tensor tau_p = P.tmp({po, pv});
  P.pack(1.0, tau, 3, 0.0, tau_p);
  P.release(tau);
  Tensor t2ph = P.tmp({o, v, o, v});
  P.permute(1.0, t2, "ijab", 0.0, t2ph, "iajb", "t2 ph layout");
  Tensor ttl;                                                     // tau_tilde (fac = 0.5), rows of the slab
  if (mine) {
    ttl = P.tmp({ni, o, v, v});
    P.tau_rows(g.rows(t2), t1, i0, 0.5, 0.5, ttl);
  }

  // ---- one-body intermediates, CCSD.py:355-387: replicated small terms + slab contributions summed over ranks
  Tensor Fov = P.tmp({o, v});
  P.axpby(1.0, s.fov, 0.0, Fov);
  {
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) P.contract(1.0, g.rows(s.oovv_ph), "menf", t1, "nf", 0.0, g.rows(p), "me", "cc_Fov");
    P.sum_ranks_add(p, Fov, "cc_Fov");
    P.release(p);
  }
  Tensor Fvv = P.tmp({v, v});
  P.axpby(1.0, s.fvv, 0.0, Fvv);
  P.contract(-0.5, s.fov, "me", t1, "ma", 1.0, Fvv, "ae", "cc_Fvv");
  {
    Tensor p = P.tmp({v, v});
    P.fill(p, 0.0);
    if (mine) {
      P.contract(-1.0, g.rows(s.ovvv), "maef", g.rows(t1), "mf", 1.0, p, "ae", "cc_Fvv vovv");
      P.contract(-0.5, ttl, "mnfa", g.rows(s.oovv), "mnfe", 1.0, p, "ae", "cc_Fvv tau~");
    }
    P.sum_ranks_add(p, Fvv, "cc_Fvv");
    P.release(p);
  }
  Tensor Foo = P.tmp({o, o});
  P.axpby(1.0, s.foo, 0.0, Foo);
  P.contract(0.5, s.fov, "me", t1, "ie", 1.0, Foo, "mi", "cc_Foo");
  P.contract(1.0, s.ooov, "mnie", t1, "ne", 1.0, Foo, "mi", "cc_Foo ooov");
  {
    Tensor p = P.tmp({o, o});
    P.fill(p, 0.0);
    if (mine) P.contract(0.5, s.oovv, "mnef", ttl, "inef", 1.0, g.at(p, 1), "mi", "cc_Foo tau~");   // columns i of the slab
    P.sum_ranks_add(p, Foo, "cc_Foo");
    P.release(p);
  }
  if (mine) P.release(ttl);
  if (shift) {
    P.diag_add(Fvv, -1.0, s.fock, o);
    P.diag_add(Foo, -1.0, s.fock, 0);
  }

  // ---- T1 residual, CCSD.py:288-294
  P.axpby(1.0, s.fov, 0.0, r1);
  P.contract(1.0, t1, "ie", Fvv, "ae", 1.0, r1, "ia");
  P.contract(-1.0, Foo, "mi", t1, "ma", 1.0, r1, "ia");
  {
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) {
      P.contract(1.0, g.rows(t2ph), "iame", Fov, "me", 1.0, g.rows(p), "ia");
      P.contract(-1.0, g.rows(s.ovov_ph), "ianf", t1, "nf", 1.0, g.rows(p), "ia");
      if (planes) pair_ovvv_rows(P, s, -0.5, t2, p, i0, ni, "T1 ovvv");
      else P.contract(-0.5, g.at(t2, 1), "imef", g.rows(s.ovvv), "maef", 1.0, p, "ia", "T1 ovvv");
      P.contract(0.5, g.rows(t2), "mnea", g.rows(s.ooov), "mnie", 1.0, p, "ia");
    }
    P.sum_ranks_add(p, r1, "T1 slab terms");
    P.release(p);
  }

  // ---- packed accumulator [ij_p, ab_p]: hh ladder + pp ladder + (t1.ovvv part of Wvvvv)   (CCSD.py:304-305)
  Tensor w4 = P.tmp({o, o, o, o});
  P.contract(1.0, s.ooov, "mnie", t1, "je", 0.0, w4, "mnij");
  Tensor Woo_p = P.tmp({po, po});
  P.axpby(1.0, s.oooo_p, 0.0, Woo_p);
  P.pack(1.0, w4, 3 | 4, 1.0, Woo_p);
  P.release(w4);
  P.contract_split(1.0, s.oovv_p, "mf", tau_p, "if", Woo_p, "mi", 'f', "Woooo tau.oovv (K3 folded)");
  Tensor acc_p = P.tmp({po, pv});
  P.contract(1.0, Woo_p, "mi", tau_p, "ma", 0.0, acc_p, "ia", "hh ladder");
  P.release(Woo_p);
  ladder_dist(P, s, tau_p, acc_p, 1.0, "K1 pp ladder");
  Tensor Z = P.tmp({po, v, v});
  if (W == 1) {
    Tensor Y_p = P.tmp({po, o * v});
    P.contract(-2.0, tau_p, "if", s.ovvv_p2, "qf", 0.0, Y_p, "iq", "R9 Y[ijma]");
    P.contract(1.0, reshape(Y_p, {po, o, v}), "pma", t1, "mb", 0.0, Z, "pab");
    P.release(Y_p);
  } else {
    Tensor YT = P.tmp_lead_padded({o, v, po});      // Y[ij,m,a] stored [m,a,ij], distributed over m
    P.contract_lead_dist(-2.0, s.ovvv_p, "maf", tau_p, "if", YT, "mai", "R9 Y[ijma]");
    P.contract(1.0, YT, "map", t1, "mb", 0.0, Z, "pab");
    P.release(YT);
  }
  P.release(tau_p);
  P.pack(-0.5, reshape(Z, {po, 1, v, v}), 2 | 4, 1.0, acc_p);
  P.release(Z);

  // ---- z: everything of the T2 residual that carries an antisymmetriser, slab rows only   (CCSD.py:297-314)
  Tensor zf = P.tmp_lead_padded({o, o, v, v});
  if (mine) {
    Tensor zg = g.rows(zf);
    Tensor F1 = P.tmp({v, v});
    P.axpby(1.0, Fvv, 0.0, F1);
    P.contract(-0.5, t1, "mb", Fov, "me", 1.0, F1, "be");
    Tensor F2 = P.tmp({o, o});
    P.axpby(1.0, Foo, 0.0, F2);
    P.contract(0.5, t1, "je", Fov, "me", 1.0, F2, "mj");
    // P(ab) terms u = t2.F1 - t1.ooov, antisymmetric in (ij): u - u^(ab) = 1/2 P(ij)P(ab) u
    P.contract(0.5, g.rows(t2), "ijae", F1, "be", 0.0, zg, "ijab");
    P.contract(-0.5, t1, "ma", g.rows(s.ooov), "ijmb", 1.0, zg, "ijab");
    // P(ij) terms w = -F2.t2 + x, x[ijab] = -t1[ie] ovvv[jeab], antisymmetric in (ab).  x enters with j leading
    // (this rank's rows of ovvv): -(x^(ji)) contributes with the opposite sign.
    P.contract(-0.5, F2, "mj", g.rows(t2), "imab", 1.0, zg, "ijab");
    P.release(F2);
    P.release(F1);
    if (planes) {
      Tensor xp = P.tmp({ni, o, pv});                              // [j in slab, i, ab_p]
      t1_ovvv_rows(P, s, 1.0, t1, xp, i0, ni, "t1.ovvv (packed pair, INT8)");
      P.unpack(0.5, reshape(xp, {ni * o, pv}), 2, 1.0, zg);
      P.release(xp);
    } else {
      P.contract(0.5, g.rows(s.ovvv), "jeab", t1, "ie", 1.0, zg, "jiab", "t1.ovvv");
    }
    // t1[ie] t1[ma] ovov[mbje] (CCSD.py:307), entered as its (ji)(ba) image with j leading
    Tensor Q = P.tmp({ni, v, o, o});
    P.contract(1.0, g.rows(s.ovov_ph), "jbme", t1, "ie", 0.0, Q, "jbmi");
    P.contract(1.0, Q, "jbmi", t1, "ma", 1.0, zg, "jiba");
    P.release(Q);
  }

  // ---- ring, CCSD.py:306 with Wovvo (CCSD.py:404-413) as the column slab W^T[(j in slab, b),(m,e)]
  Tensor WcT;
  if (mine) {
    WcT = P.tmp({ni, v, o, v});
    P.contract(0.5, g.rows(t2ph), "jbnf", s.oovv_ph, "nfme", 0.0, WcT, "jbme", "R1 Wovvo");
    // -t1[nb] (oovv[mnef] t1[jf] - ooov[mnje]): the two o^3v operands are combined first
    Tensor U = P.tmp({o, o, ni, v});
    P.axpby(-1.0, g.at(s.ooov, 2), 0.0, U);
    P.contract(1.0, s.oovv, "mnef", g.rows(t1), "jf", 1.0, U, "mnje");
    P.contract(-1.0, U, "mnje", t1, "nb", 1.0, WcT, "jbme");
    P.release(U);
    P.axpby(-1.0, g.rows(s.ovov_ph), 1.0, WcT);                   // ovvo[mbej] = -ovov[mbje]; ovov_ph is symmetric
  }
  // t1[jf] ovvv[mbef]: formed on this rank's rows m of ovvv for all j, then moved to the owners of j
  if (W == 1) {
    P.contract(1.0, s.ovvv, "mbef", t1, "jf", 1.0, WcT, "jbme", "Wovvo ovvv.t1");
  } else {
    const int64_t cnt = g.chunk * g.chunk * v * v;
    Tensor snd = P.tmp({W * g.chunk, g.chunk, v, v});             // [j (padded), m local (padded), b, e]
    Tensor rcv = P.tmp({W, g.chunk, g.chunk, v, v});              // [source rank, j local, m local, b, e]
    P.fill(snd, 0.0);
    if (mine) {
      Tensor sv = snd;
      sv.dim[0] = o;
      sv.dim[1] = ni;
      P.contract(1.0, t1, "jf", g.rows(s.ovvv), "mbef", 0.0, sv, "jmbe", "Wovvo ovvv.t1 (rows m of ovvv)");
    }
    P.alltoall(snd, cnt, rcv, "Wovvo ovvv.t1: rows m -> columns j");
    if (mine) {
      for (int q = 0; q < W; ++q) {
        const int64_t m0 = std::min<int64_t>(o, (int64_t)q * g.chunk), nm = std::min<int64_t>(o, m0 + g.chunk) - m0;
        if (nm <= 0) continue;
        Tensor src = make_tensor(rcv.slot, rcv.off + (int64_t)q * cnt, {g.chunk, g.chunk, v, v});
        src.dim[0] = ni;
        src.dim[1] = nm;
        P.permute(1.0, src, "jmbe", 1.0, slice_dim(WcT, 2, m0, nm), "jbme", "Wovvo ovvv.t1 (received)");
      }
    }
    P.release(rcv);
    P.release(snd);
  }
  if (mine) {
    Tensor zg = g.rows(zf);
    Tensor ringT = P.tmp({ni, v, o, v});                          // ring^T[(j in slab, b),(i,a)]
    P.contract(1.0, WcT, "jbme", t2ph, "iame", 0.0, ringT, "jbia", "R2 ring");          // t2ph symmetric
    P.release(WcT);
    P.permute(1.0, ringT, "jbia", 1.0, zg, "jiba", "ring -> z");
    P.release(ringT);
  }
  P.release(t2ph);
  P.release(Fov);
  P.release(Fvv);
  P.release(Foo);

  // ---- assemble: R2 = oovv + P(ij)P(ab) z + unpack(acc_p)
  gather_rows(P, g, zf, "z (T2)");
  P.asym4(1.0, &s.oovv, zf, 0.0, r2, "T2 = oovv + P(ij)P(ab) z");
  P.release(zf);
  P.unpack(1.0, acc_p, 3, 1.0, r2);
  P.release(acc_p);

  P.finish(r1, t1, s.fock, (int)o, 2, has_alpha, equation, 0.0, r1);
  P.finish(r2, t2, s.fock, (int)o, 4, has_alpha, equation, 0.0, r2);
}

// ======================================================================================================= L1 / L2
void build_ccsd_lupdate(Plan& P, const Sizes& z, int has_alpha, int equation) {
  z.apply(P);
  Slots s(z);
  const int64_t o = s.o, v = s.v, po = s.po, pv = s.pv;
  const bool shift = !equation && !has_alpha;  // CCSD.py:449-456 (Q2)
  const Tensor &t1 = s.t1, &t2 = s.t2, &l1 = s.l1, &l2 = s.l2, &r1 = s.out1, &r2 = s.out2;
  const Slab g(P, o);
  const int64_t i0 = g.i0, ni = g.ni, W = P.world;
  const bool planes = P.ovvv_planes;
  const bool mine = ni > 0;

  // ---- replicated, from the replicated inputs
  Tensor tau = P.tmp({o, o, v, v});
  P.tau(t2, t1, 1.0, 1.0, tau);     // antisymmetric part of CCSD.py:565 (all uses contract an antisymmetric pair)
  Tensor tau_p = P.tmp({po, pv});
  P.pack(1.0, tau, 3, 0.0, tau_p);
  Tensor l2_p = P.tmp({po, pv});
  P.pack(1.0, l2, 3, 0.0, l2_p);
  Tensor t2ph = P.tmp({o, v, o, v});
  P.permute(1.0, t2, "ijab", 0.0, t2ph, "iajb", "t2 ph layout");
  Tensor l2ph = P.tmp({o, v, o, v});
  P.permute(1.0, l2, "ijab", 0.0, l2ph, "iajb", "l2 ph layout");

  // ---- Linter one-body pieces, CCSD.py:543-623
  Tensor Fov = P.tmp({o, v});   // = fov1 (:474) = tmp (:504) = (:580)
  P.axpby(1.0, s.fov, 0.0, Fov);
  {
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) P.contract(1.0, g.rows(s.oovv_ph), "menf", t1, "nf", 0.0, g.rows(p), "me");
    P.sum_ranks_add(p, Fov, "fov1");
    P.release(p);
  }
  Tensor v1 = P.tmp({v, v});
  P.axpby(1.0, s.fvv, 0.0, v1);
  P.contract(-1.0, s.fov, "ja", t1, "jb", 1.0, v1, "ba");
  {
    Tensor p = P.tmp({v, v});
    P.fill(p, 0.0);
    if (mine) {
      P.contract(-1.0, g.rows(s.ovvv), "jbac", g.rows(t1), "jc", 1.0, p, "ba", "v1 ovvv");
      P.contract(-0.5, g.rows(tau), "jkcb", g.rows(s.oovv), "jkca", 1.0, p, "ba", "v1 tau.oovv");
    }
    P.sum_ranks_add(p, v1, "v1");
    P.release(p);
  }
  Tensor v2 = P.tmp({o, o});
  P.axpby(1.0, s.foo, 0.0, v2);
  P.contract(1.0, s.fov, "ib", t1, "jb", 1.0, v2, "ij");
  P.contract(-1.0, s.ooov, "kijb", t1, "kb", 1.0, v2, "ij");
  {
    Tensor p = P.tmp({o, o});
    P.fill(p, 0.0);
    if (mine) P.contract(0.5, s.oovv, "ikbc", g.rows(tau), "jkbc", 1.0, g.at(p, 1), "ij", "v2 tau.oovv");   // columns j of the slab
    P.sum_ranks_add(p, v2, "v2");
    P.release(p);
  }
  P.release(tau);

  // v4 as the column slab v4^T[(j in slab, b),(k,c)] = v4[j,c,b,k]  (CCSD.py:575-576); oovv_ph, ovov_ph, t2ph symmetric
  Tensor v4T;
  if (mine) {
    v4T = P.tmp({ni, v, o, v});
    P.contract(1.0, g.rows(s.oovv_ph), "jbld", t2ph, "kcld", 0.0, v4T, "jbkc", "R3 v4");   // same view of t2ph as below: one cut
    P.axpby(-1.0, g.rows(s.ovov_ph), 1.0, v4T);
  }

  // v5^T, w3^T (CCSD.py:578-590): replicated small terms + slab contributions
  Tensor w3T = P.tmp({o, v});          // w3T[k,c] = w3[c,k]
  P.permute(1.0, s.fvo, "bj", 0.0, w3T, "jb");
  {
    Tensor q = P.tmp({o, o});
    P.contract(1.0, Fov, "kc", t1, "jc", 0.0, q, "kj");
    P.contract(1.0, q, "kj", t1, "kb", 1.0, w3T, "jb");
    P.release(q);
  }
  P.contract(1.0, t1, "kb", v1, "cb", 1.0, w3T, "kc");
  P.contract(-1.0, v2, "jk", t1, "jc", 1.0, w3T, "kc");
  {
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) {
      P.contract(1.0, g.rows(t2ph), "jbkc", s.fov, "kc", 1.0, g.rows(p), "jb");
      P.contract(0.5, g.rows(s.ooov), "kljc", g.rows(t2), "klcb", 1.0, p, "jb");
      if (planes) pair_ovvv_rows(P, s, -0.5, t2, p, i0, ni, "v5 ovvv");
      else P.contract(-0.5, g.at(t2, 1), "jkdc", g.rows(s.ovvv), "kbdc", 1.0, p, "jb", "v5 ovvv");
      P.contract(1.0, v4T, "jbkc", g.rows(t1), "jb", 1.0, p, "kc", "w3: v4.t1");
    }
    P.sum_ranks_add(p, w3T, "w3 slab terms");
    P.release(p);
  }

  // hole-hole pieces, packed [ij_p, kl_p]
  Tensor woo_p = P.tmp({po, po});
  P.axpby(0.5, s.oooo_p, 0.0, woo_p);
  P.contract_split(0.5, s.oovv_p, "if", tau_p, "kf", woo_p, "ik", 'f', "v3");
  Tensor y4 = P.tmp({o, o, o, o});
  P.contract(1.0, s.ooov, "jilc", t1, "kc", 0.0, y4, "jilk");
  P.pack(0.5, y4, 3 | 4, 1.0, woo_p);
  P.release(y4);
  Tensor lt_p = P.tmp({po, po});
  P.fill(lt_p, 0.0);
  P.contract_split(2.0, l2_p, "if", tau_p, "kf", lt_p, "ik", 'f', "l2.tau");

  // wovvo as the column slab w^T[(j in slab, b),(k,c)]  (CCSD.py:596-598)
  Tensor wT;
  if (mine) {
    wT = P.tmp({ni, v, o, v});
    P.axpby(1.0, v4T, 0.0, wT);
    Tensor S = P.tmp({o, ni, o, v});                               // [l, j in slab, k, b]
    P.axpby(-1.0, g.at(s.ooov, 1), 0.0, S);
    P.contract(1.0, g.at(s.oovv, 1), "ljbd", t1, "kd", 1.0, S, "ljkb");
    P.contract(1.0, S, "ljkb", t1, "lc", 1.0, wT, "jbkc");
    P.release(S);
    P.contract(1.0, g.rows(s.ovvv), "jcbd", t1, "kd", 1.0, wT, "jbkc", "wovvo ovvv.t1");
  }

  // wovoo, rows i of the slab  (CCSD.py:600-603)
  Tensor wovoo;
  if (mine) {
    Tensor wo_p = P.tmp({ni, v, po});
    P.contract(0.5, g.rows(s.ovvv_p), "icf", tau_p, "kf", 0.0, wo_p, "ick", "R4 wovoo");
    wovoo = P.tmp({ni, v, o, o});
    P.unpack(1.0, reshape(wo_p, {ni * v, po}), 2, 0.0, wovoo);
    P.release(wo_p);
    P.permute(0.5, g.at(s.ooov, 2), "jkic", 1.0, wovoo, "icjk");
    P.contract(1.0, v4T, "ibkc", t1, "jb", 1.0, wovoo, "icjk");
    P.contract(-1.0, t2ph, "kclb", g.at(s.ooov, 1), "lijb", 1.0, wovoo, "icjk", "wovoo ooov.t2");
  }
  P.release(tau_p);

  // ---- m3, CCSD.py:461-470, packed [ij_p, ab_p] (replicated small products, distributed ladder and R6)
  Tensor m3_p = P.tmp({po, pv});
  P.contract(2.0, woo_p, "ik", l2_p, "ka", 0.0, m3_p, "ia", "l2.woooo");
  P.release(woo_p);
  P.contract(0.5, lt_p, "ik", s.oovv_p, "ka", 1.0, m3_p, "ia");
  Tensor l2t1 = P.tmp({o, o, v, o});
  P.contract(1.0, l2, "ijcd", t1, "kd", 0.0, l2t1, "ijck");
  Tensor a_full = P.tmp({o, o, o, v});
  P.permute(1.0, l2t1, "ijck", 0.0, a_full, "ijkc");
  Tensor a_p = P.tmp({po, o * v});
  P.pack(1.0, reshape(a_full, {o, o, o * v, 1}), 1, 0.0, a_p);
  P.release(a_full);
  if (W == 1) {
    P.contract(1.0, a_p, "pq", s.ovvv_p2, "qa", 1.0, m3_p, "pa", "R6 ovvv.(l2 t1)");
  } else {
    Tensor r6 = P.tmp_lead_padded({po, pv});
    P.contract_lead_dist(1.0, a_p, "pq", s.ovvv_p2, "qa", r6, "pa", "R6 ovvv.(l2 t1)");
    P.axpby(1.0, r6, 1.0, m3_p);
    P.release(r6);
  }
  P.release(a_p);
  ladder_dist(P, s, l2_p, m3_p, 1.0, "K2 pp ladder");
  P.release(l2_p);

  // small symmetric products of the amplitudes (CCSD.py:459-460): contraction over the slab index, summed over ranks
  Tensor m_vv = P.tmp({v, v});
  P.fill(m_vv, 0.0);
  Tensor m_oo = P.tmp({o, o});
  P.fill(m_oo, 0.0);
  {
    Tensor p = P.tmp({v, v});
    P.fill(p, 0.0);
    if (mine) P.contract(0.5, g.rows(t2), "klcb", g.rows(l2), "klca", 1.0, p, "ba");
    P.sum_ranks_add(p, m_vv, "mba");
    P.release(p);
    Tensor q = P.tmp({o, o});
    P.fill(q, 0.0);
    if (mine) P.contract(0.5, g.rows(l2), "kicd", g.rows(t2), "kjcd", 1.0, q, "ij");
    P.sum_ranks_add(q, m_oo, "mij");
    P.release(q);
  }
  Tensor x_vv = P.tmp({v, v});
  P.axpby(1.0, m_vv, 0.0, x_vv);
  P.contract(1.0, l1, "ka", t1, "kb", 1.0, x_vv, "ba");
  Tensor x_oo = P.tmp({o, o});
  P.axpby(1.0, m_oo, 0.0, x_oo);
  P.contract(1.0, l1, "ic", t1, "kc", 1.0, x_oo, "ik");
  if (shift) {  // after w3 (which uses the unshifted v1, v2)
    P.diag_add(v1, -1.0, s.fock, o);
    P.diag_add(v2, -1.0, s.fock, 0);
  }

  // ---- R2 starts as unpack(m3): the L1 term m3.t1 (CCSD.py:498) reads its slab rows from there
  P.unpack(1.0, m3_p, 3, 0.0, r2);
  P.release(m3_p);

  // ---- z: the antisymmetrised part of the L2 residual, CCSD.py:474-488
  Tensor zf = P.tmp_lead_padded({o, o, v, v});
  if (mine) {
    Tensor zg = g.rows(zf);
    // ring^T[(j in slab, b),(i,a)] = w^T . l2ph + fov1[jb] l1[ia]
    Tensor ringT = P.tmp({ni, v, o, v});
    P.contract(1.0, wT, "jbkc", l2ph, "iakc", 0.0, ringT, "jbia", "R7 ring");           // l2ph symmetric; same view as R8: one cut
    P.release(wT);
    P.contract(1.0, g.rows(Fov), "jb", l1, "ia", 1.0, ringT, "jbia");
    P.permute(1.0, ringT, "jbia", 0.0, zg, "jiba", "ring -> z");
    P.release(ringT);
    // -(y - y^(ab)), y = l1.ooov - l2.v1 - oovv.x_vv antisymmetric in (ij): -1/2 P(ij)P(ab) y
    P.contract(-0.5, l1, "ka", g.rows(s.ooov), "ijkb", 1.0, zg, "ijab");
    P.contract(0.5, g.rows(l2), "ijac", v1, "cb", 1.0, zg, "ijab");
    P.contract(0.5, g.rows(s.oovv), "ijbc", x_vv, "ca", 1.0, zg, "ijab");     // oovv[ijcb] = -oovv[ijbc] (Eris.py:128)
    // +(y2 - y2^(ij)), y2[pqrs] = l1[qc] ovvv[pcrs] + v2[qk] l2[kprs] - x_oo[pk] oovv[kqrs] antisymmetric in (rs)
    if (planes) {
      Tensor yp = P.tmp({ni, o, pv});                              // [p in slab, q, rs_p]
      t1_ovvv_rows(P, s, 1.0, l1, yp, i0, ni, "l1.ovvv (packed pair, INT8)");
      P.unpack(0.5, reshape(yp, {ni * o, pv}), 2, 1.0, zg);
      P.release(yp);
    } else {
      P.contract(0.5, g.rows(s.ovvv), "pcrs", l1, "qc", 1.0, zg, "pqrs", "l1.ovvv");
    }
    P.contract(-0.5, g.rows(l2), "pkrs", v2, "qk", 1.0, zg, "pqrs");           // l2[kprs] = -l2[pkrs]
    P.contract(-0.5, g.rows(x_oo), "pk", s.oovv, "kqrs", 1.0, zg, "pqrs");
  }

  // ---- L1 residual, CCSD.py:490-506: replicated small terms + slab contributions
  P.axpby(1.0, s.fov, 0.0, r1);
  P.contract(1.0, l1, "ib", v1, "ba", 1.0, r1, "ia");
  P.contract(-1.0, v2, "ij", l1, "ja", 1.0, r1, "ia");
  {
    Tensor lt = P.tmp({o, o, o, o});
    P.unpack(1.0, lt_p, 3, 0.0, lt);
    P.contract(-0.25, lt, "ikjl", s.ooov, "jlka", 1.0, r1, "ia", "wvvvo: ooov.tau");
    P.release(lt);
  }
  P.release(lt_p);
  P.contract(-1.0, s.ooov, "jika", x_oo, "kj", 1.0, r1, "ia");
  P.contract(-1.0, m_oo, "ik", Fov, "ka", 1.0, r1, "ia");
  P.contract(-1.0, m_vv, "ca", Fov, "ic", 1.0, r1, "ia");
  Tensor zz = P.tmp({o, v});
  P.axpby(1.0, t1, 0.0, zz);
  P.contract(-1.0, x_vv, "bd", t1, "jd", 1.0, zz, "jb");
  P.contract(-1.0, m_oo, "lj", t1, "lb", 1.0, zz, "jb");
  {
    // zz also holds t2ph.l1 (CCSD.py:502): rows of the slab, summed over ranks
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) P.contract(1.0, g.rows(t2ph), "jbkc", l1, "kc", 1.0, g.rows(p), "jb");
    P.sum_ranks_add(p, zz, "t2.l1");
    P.release(p);
  }
  {
    Tensor p = P.tmp({o, v});
    P.fill(p, 0.0);
    if (mine) {
      Tensor pr = g.rows(p);
      P.contract(-1.0, g.rows(s.ovov_ph), "iajb", l1, "jb", 1.0, pr, "ia");             // ovov_ph symmetric
      P.contract(-1.0, wovoo, "icjk", l2, "kjca", 1.0, pr, "ia");
      P.release(wovoo);
      // -(l2 . wvvvo) with wvvvo never formed (four pieces):
      P.contract(1.0, g.at(l2t1, 3), "ikcj", v4T, "jakc", 1.0, p, "ia", "wvvvo: v4.t1");
      P.release(v4T);
      if (planes) pair_ovvv_rows(P, s, -0.5, l2, p, i0, ni, "wvvvo: ovvv");
      else P.contract(-0.5, g.at(l2, 1), "ikbc", g.rows(s.ovvv), "kabc", 1.0, p, "ia", "wvvvo: ovvv");
      Tensor XT = P.tmp({ni, v, o, v});                            // X^T[(k in slab, d),(i,b)] = sum_jc t2ph[(kd),(jc)] l2ph[(jc),(ib)]
      P.contract(1.0, g.rows(t2ph), "kdjc", l2ph, "ibjc", 0.0, XT, "kdib", "R8 l2.t2");
      P.contract(1.0, XT, "kdib", g.rows(s.ovvv), "kbda", 1.0, p, "ia", "wvvvo: ovvv.t2 (K4 refactored)");
      P.release(XT);
      P.contract(1.0, g.rows(r2), "ijab", t1, "jb", 1.0, pr, "ia", "m3.t1");
      P.contract(1.0, g.rows(l2ph), "iajb", w3T, "jb", 1.0, pr, "ia");
      P.contract(1.0, g.rows(s.oovv_ph), "iajb", zz, "jb", 1.0, pr, "ia");
      // ovvv[icba] x_vv[bc]: one matrix-vector product per i (K = v^2 split over the SMs; a batched lowering would run
      // one CTA column per i)
      for (int64_t i = 0; i < ni; ++i) {
        Tensor oi = slice0(g.rows(s.ovvv), i, 1), ri = slice0(pr, i, 1);
        P.contract(-1.0, reshape(oi, {v, v, v}), "cba", x_vv, "bc", 1.0, reshape(ri, {v}), "a", "L1 ovvv.x_vv");
      }
    }
    P.sum_ranks_add(p, r1, "L1 slab terms");
    P.release(p);
  }
  P.release(zz);
  P.release(l2t1);
  P.release(l2ph);
  P.release(t2ph);

  // ---- assemble: R2 = oovv + m3 + P(ij)P(ab) z
  gather_rows(P, g, zf, "z (L2)");
  P.asym4(1.0, &s.oovv, zf, 1.0, r2, "L2 = oovv + m3 + P(ij)P(ab) z");
  P.release(zf);

  if (shift) {  // energy term, CCSD.py:509-510
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

}  // namespace ecw
