"""Host-side mirror of the reference `CCS.Gccs` class and the module-level rdm1 builders
(CCS.py:23-1518): CCS ground state (T1/Lambda1 intermediates and updates incl. the ES coupling
terms), EOM-like right/left excited-state residuals for H + Vexp, and the four rdm1 variants.

Same names, argument order, tuple layouts and in-place quirks as the reference, so the unchanged
`Solver_GS.Solver_CCS` / `Solver_ES.Solver_ES` loops drive it.  Every arithmetic operation runs on
the device: the four intermediate builders (everything that reads an integral block) are single calls
of the C ABI — `ecw_ccs_t1inter / l1inter / r1inter / esl1inter`, cached plans replayed as CUDA graphs
(csrc/ccs_plan.cpp) — and the singles-sized updates are sequences of the primitive ops (`ecw_op_*`:
contraction engine + FP64 tensor-core GEMM, strided axpby, denominators, dot) with the reference's
host-side scalar logic between them.  Only canonical integral blocks are kept on
the device; the reference's other blocks follow from Eris.py:128:
    ovvo[jabi] = -ovov_ph[iajb]   voov[bija] = -ovov_ph[jbia]   oovo[kjbi] = -ooov[kjib]
    vovv[bica] = -ovvv[ibca]      with ovov_ph[(ia),(nf)] = ovov[naif].
numpy in -> numpy out.  The o^2v^2 intermediates (Wbija / Wakic) additionally stay cached on the
device, so the update that follows does not upload them again.
"""
import numpy as np

from ._lib import lib, EcwError, ECW_HAS_ALPHA, ECW_SUBDIFF_SINGLES
from .devops import ArgBlocks, _scalar
from .eris import DeviceEris


def _like_amp0(em, amp0):
    """The reference forms Em from `... + r0 * Zia[o, v]` (CCS.py:897-904, 1310-1317): a shape-(1,) r0 / l0 (what the
    solver carries after the first iteration) makes Em a shape-(1,) ARRAY — which `l0_fromE` then changes in place (Q12)."""
    if isinstance(amp0, np.ndarray) and amp0.ndim > 0:
        return em * np.ones_like(amp0, dtype=np.float64)
    return em


class InterTuple(tuple):
    """Reference-shaped tuple of intermediates + device copies of its large members."""
    dev = None


def _is_num(x):
    return isinstance(x, (float, int))


class Gccs(object):
    def __init__(self, eris, fock=None, M_tot=None, device=None, gemm=None):
        if not isinstance(eris, DeviceEris):
            eris = DeviceEris.from_geris(eris, device=device, gemm=gemm)
        self.M_tot = 1 if M_tot is None else M_tot                   # CCS.py:207-210
        self.eris = eris
        self.fock = np.asarray(eris.fock) if fock is None else fock  # CCS.py:212-215
        self.nocc = eris.nocc
        self.nvir = self.fock.shape[0] - self.nocc
        self.ops = eris.ops
        self._blocks = None           # ArgBlocks of _inter
        if fock is not None:
            eris.set_fock(fock)

    # ------------------------------------------------------------------ helpers
    def _G(self, ts):
        """G[jb] = sum_kc ts[kc] oovv[jkbc]"""
        return self.ops.contract('kc,jkbc->jb', ts, self.eris.block("oovv"))

    def _w_dev(self, inter, idx, shape):
        """Device copy of the o^2v^2 member of an intermediate tuple (cached when it is ours)."""
        w = inter[idx]
        dev = getattr(inter, "dev", None)
        if dev is not None and dev.get("host_id") == id(w):
            return dev["W"]
        return self.ops.to_dev(np.asarray(w, dtype=np.float64).reshape(shape))

    def _pack(self, host_items, W_dev, w_index):
        t = InterTuple(host_items)
        t.dev = {"W": W_dev, "host_id": id(host_items[w_index])}
        return t

    def _q6(self, Fv_h, Fo_h):
        """Q6: an update subtracts the Fock diagonal from the vv and oo blocks of its intermediate tuple IN PLACE, so
        the caller's arrays change as in the reference.  Returns the shifted device copies."""
        ops = self.ops
        Fv, Fo = ops.to_dev(Fv_h), ops.to_dev(Fo_h)
        ops.diag_shift(Fv, -1.0, self.nocc)
        ops.diag_shift(Fo, -1.0, 0)
        Fv_h[...] = ops.to_host(Fv)
        Fo_h[...] = ops.to_host(Fo)
        return Fv, Fo

    def _inter(self, func, ts, fsp, vm=None, e_term=True):
        """One of the four intermediate builders as ONE call of the C ABI (ecw_ccs_t1inter / l1inter / r1inter /
        esl1inter: a cached plan, replayed as a CUDA graph).  The arguments go through persistent device blocks so that
        the pointers the library sees never change; returns (F [n,n] device, W [v,o,o,v] device or None, X [o,v] device
        or None, scalar or None) — F and X are views of the persistent blocks (read them before the next call), W is a
        fresh tensor (it is cached for the update that follows)."""
        ops = self.ops
        e = self.eris
        o, v = self.nocc, self.nvir
        n = o + v
        st = self._blocks
        if st is None:
            st = self._blocks = ArgBlocks(e.device, ts=(o, v), fsp=(n, n), vm=(n, n), F=(n, n), W=(v, o, o, v),
                                          X=(o, v), e=(1,))
        st.put(ts=ops.to_dev(ts), fsp=e.fock_dev if fsp is None else ops.to_dev(fsp))
        if vm is not None:
            st.put(vm=ops.to_dev(vm))
        p = lambda k: st[k].data_ptr()                                                           # noqa: E731
        if func == "t1":
            e.execute("ccs_t1inter", 0, lambda: lib.ecw_ccs_t1inter(e._h, p("ts"), p("fsp"), p("F"), e.stream()),
                      "ecw_ccs_t1inter")
            return st["F"], None, None, None
        if func == "l1":
            fl = 1 if e_term else 0
            e.execute("ccs_l1inter", fl, lambda: lib.ecw_ccs_l1inter(e._h, p("ts"), p("fsp"), fl, p("F"), p("W"), p("e"),
                                                                      e.stream()), "ecw_ccs_l1inter")
            return st["F"], st["W"].clone(), None, (ops.scalar(st["e"]) if e_term else 0.)
        name = {"r1": "ccs_r1inter", "esl1": "ccs_esl1inter"}[func]
        fn = lib.ecw_ccs_r1inter if func == "r1" else lib.ecw_ccs_esl1inter
        fl = 1 if vm is not None else 0
        e.execute(name, fl, lambda: fn(e._h, p("ts"), p("fsp"), (p("vm") if vm is not None else None), p("F"), p("W"),
                                       p("X"), p("e"), e.stream()), "ecw_" + name)
        return st["F"], st["W"].clone(), st["X"], ops.scalar(st["e"])

    # ------------------------------------------------------------------ energy (CCS.py:226-249)
    def energy_ccs(self, ts, fsp, rsn=None, r0n=None, vn=None):
        ops = self.ops
        o = self.nocc
        d_ts = ops.to_dev(ts)
        foo, fov, fvo, fvv = self.eris.fock_blocks(fsp)
        e = ops.dot(fov, d_ts) + 0.5 * ops.dot(d_ts, self._G(d_ts))
        if rsn is not None:
            for rs, v, r0 in zip(rsn, vn, r0n):
                if v is not None:
                    d_v = ops.to_dev(v)
                    e += -ops.dot(d_v[:o, o:], ops.to_dev(rs)) - r0 * ops.dot(d_v[:o, o:], d_ts) \
                         - r0 * ops.trace(d_v[:o, :o])
        return e

    # ------------------------------------------------------------------ rdm1 (CCS.py:255-265)
    def gamma(self, ts, ls):
        return gamma_CCS(ts, ls, self)

    def gamma_unsym(self, ts, ls):
        return gamma_unsym_CCS(ts, ls, self)

    def gamma_es(self, ts, ln, rn, r0n, l0n):
        return gamma_es_CCS(ts, ln, rn, r0n, l0n, self)

    def gamma_tr(self, ts, ln, rk, r0k, l0n):
        return gamma_tr_CCS(ts, ln, rk, r0k, l0n, self)

    # ------------------------------------------------------------------ T1 (CCS.py:271-440)
    def T1inter(self, ts, fsp):
        ops = self.ops
        o = self.nocc
        F, _, _, _ = self._inter("t1", ts, fsp)
        return ops.to_host(F[o:, o:]), ops.to_host(F[:o, :o]), ops.to_host(F[o:, :o])     # Fab, Fji, Fai

    def _t1(self, d_ts, Fab, Fji, Fai):
        ops = self.ops
        T1 = ops.copy(Fai, 'ai->ia')
        ops.contract('ib,ab->ia', d_ts, Fab, out=T1, beta=1.0)
        ops.contract('ja,ji->ia', d_ts, Fji, alpha=-1.0, out=T1, beta=1.0)
        return T1

    def T1eq(self, ts, fsp):
        ops = self.ops
        Fab, Fji, Fai = self.T1inter(ts, fsp)
        return ops.to_host(self._t1(ops.to_dev(ts), ops.to_dev(Fab), ops.to_dev(Fji), ops.to_dev(Fai)))

    def tsupdate(self, ts, T1inter, rsn=None, r0n=None, vn=None):
        ops = self.ops
        o, v = self.nocc, self.nvir
        Fab_h, Fji_h, Fai_h = T1inter
        d_ts = ops.to_dev(ts)
        Fab, Fji = self._q6(Fab_h, Fji_h)                  # CCS.py:307-308
        new = self._t1(d_ts, Fab, Fji, ops.to_dev(Fai_h))
        if rsn is not None:                                # ES coupling, CCS.py:316-347
            if r0n is None:
                raise ValueError('if Vexp are to be calculated, list of r0 amp must be given')
            if len(vn) != len(rsn):
                raise ValueError('Number of experimental potentials must be equal to number of r amplitudes')
            for r, vm, r0 in zip(rsn, vn, r0n):
                if vm is None:
                    continue
                mv = ops.copy(ops.to_dev(vm), alpha=-1.0)
                v_oo, v_ov, v_vv = mv[:o, :o], mv[:o, o:], mv[o:, o:]
                d_r = ops.to_dev(r)
                Z = ops.trace(v_oo) + ops.dot(v_ov, d_ts)
                Z0 = ops.copy(v_ov)
                ops.contract('ib,ab->ia', d_ts, v_vv, out=Z0, beta=1.0)
                ops.contract('ja,ji->ia', d_ts, v_oo, alpha=-1.0, out=Z0, beta=1.0)
                tmp = ops.contract('ja,jb->ab', d_ts, v_ov)
                ops.contract('ab,ib->ia', tmp, d_ts, alpha=-1.0, out=Z0, beta=1.0)
                Zab = ops.copy(v_vv)
                ops.add(Zab, tmp, -1.0)
                Zji = ops.copy(v_oo, alpha=-1.0)
                ops.contract('ib,jb->ji', d_ts, v_ov, alpha=-1.0, out=Zji, beta=1.0)
                ops.scale_add(new, d_r, Z)
                ops.scale_add(new, Z0, r0)
                ops.contract('ab,ib->ia', Zab, d_r, out=new, beta=1.0)
                ops.contract('ji,ja->ia', Zji, d_r, out=new, beta=1.0)
        return ops.to_host(ops.denom(new, d_ts))

    def tsupdate_L1(self, ts, T1inter, alpha):             # CCS.py:353-384
        ops = self.ops
        Fab, Fji, Fai = T1inter
        d_ts = ops.to_dev(ts)
        T1 = self._t1(d_ts, ops.to_dev(Fab), ops.to_dev(Fji), ops.to_dev(Fai))
        return ops.to_host(ops.denom(T1, d_ts, ECW_HAS_ALPHA | ECW_SUBDIFF_SINGLES, alpha))

    # ------------------------------------------------------------------ Lambda1 (CCS.py:490-698)
    def L1inter(self, ts, fsp, E_term=True):
        ops = self.ops
        o = self.nocc
        F, W, _, E = self._inter("l1", ts, fsp, e_term=E_term)
        host = (ops.to_host(F[:o, o:]), ops.to_host(F[o:, o:]), ops.to_host(F[:o, :o]), ops.to_host(W), E)   # Fia, Fba, Fij
        return self._pack(host, W, 3)

    def _l1(self, d_ls, Fia, Fba, Fij, W, E):
        ops = self.ops
        L1 = ops.copy(Fia)
        ops.contract('ib,ba->ia', d_ls, Fba, out=L1, beta=1.0)
        ops.contract('ja,ij->ia', d_ls, Fij, alpha=-1.0, out=L1, beta=1.0)
        ops.contract('jb,bija->ia', d_ls, W, out=L1, beta=1.0)
        ops.scale_add(L1, d_ls, E)
        return L1

    def L1eq(self, ts, ls, fsp, E_term=True):
        ops = self.ops
        inter = self.L1inter(ts, fsp, E_term=E_term)
        L1 = self._l1(ops.to_dev(ls), ops.to_dev(inter[0]), ops.to_dev(inter[1]), ops.to_dev(inter[2]),
                      inter.dev["W"], _scalar(inter[4]))
        return ops.to_host(L1)

    def lsupdate(self, ts, ls, L1inter, rsn=None, lsn=None, r0n=None, l0n=None, vn=None):
        ops = self.ops
        o, v = self.nocc, self.nvir
        Fia_h, Fba_h, Fij_h, W_h, E = L1inter
        d_ts, d_ls = ops.to_dev(ts), ops.to_dev(ls)
        W = self._w_dev(L1inter, 3, (v, o, o, v))
        Fba, Fij = self._q6(Fba_h, Fij_h)                  # CCS.py:529-530
        new = self._l1(d_ls, ops.to_dev(Fia_h), Fba, Fij, W, _scalar(E))
        if rsn is not None:                                # CCS.py:539-579
            if len(lsn) != len(rsn) or len(vn) != len(rsn):
                raise ValueError('v0n, l and r list must be of same length')
            if r0n is None or l0n is None:
                raise ValueError('r0 and l0 values must be given')
            for r, l, vm, r0, l0 in zip(rsn, lsn, vn, r0n, l0n):
                if vm is None:
                    continue
                mv = ops.copy(ops.to_dev(vm), alpha=-1.0)
                v_oo, v_ov, v_vv = mv[:o, :o], mv[:o, o:], mv[o:, o:]
                d_r, d_l = ops.to_dev(r), ops.to_dev(l)
                tr = ops.trace(v_oo)
                tv = ops.dot(d_ts, v_ov)
                Pl = ops.dot(d_r, v_ov) + r0 * tv + r0 * tr
                P = tr + tv
                Pba = ops.copy(v_vv)
                ops.contract('jb,ja->ba', d_ts, v_ov, alpha=-1.0, out=Pba, beta=1.0)
                Pij = ops.copy(v_oo, alpha=-1.0)
                ops.contract('jb,ib->ij', d_ts, v_ov, alpha=-1.0, out=Pij, beta=1.0)
                ops.scale_add(new, d_ls, Pl)
                ops.scale_add(new, v_ov, l0)
                ops.scale_add(new, d_l, P)
                ops.contract('ib,ba->ia', d_l, Pba, out=new, beta=1.0)
                ops.contract('ja,ij->ia', d_l, Pij, out=new, beta=1.0)
        return ops.to_host(ops.denom(new, d_ls))

    def lsupdate_L1(self, ls, L1inter, alpha):             # CCS.py:585-617
        ops = self.ops
        o, v = self.nocc, self.nvir
        d_ls = ops.to_dev(ls)
        L1 = self._l1(d_ls, ops.to_dev(L1inter[0]), ops.to_dev(L1inter[1]), ops.to_dev(L1inter[2]),
                      self._w_dev(L1inter, 3, (v, o, o, v)), _scalar(L1inter[4]))
        return ops.to_host(ops.denom(L1, d_ls, ECW_HAS_ALPHA | ECW_SUBDIFF_SINGLES, alpha))

    # ------------------------------------------------------------------ ES right (CCS.py:774-1158)
    def R1inter(self, ts, fsp, vm):
        ops = self.ops
        o = self.nocc
        F, W, X, Er = self._inter("r1", ts, (self.fock if fsp is None else fsp), vm)
        host = (ops.to_host(F[o:, o:]), ops.to_host(F[:o, :o]), ops.to_host(W), Er, ops.to_host(F[:o, o:]),
                ops.to_host(X))                                                          # Fab, Fji, Wakic, Er, Tia, Pia
        return self._pack(host, W, 2)

    def _r1core(self, d_rs, Fab, Fji, W):
        ops = self.ops
        R = ops.contract('ab,ib->ia', Fab, d_rs)
        ops.contract('ji,ja->ia', Fji, d_rs, alpha=-1.0, out=R, beta=1.0)
        ops.contract('akic,kc->ia', W, d_rs, out=R, beta=1.0)
        return R

    def _es1full(self, core, amp, amp0, inter, shifted=None):
        """core(amp, Fv, Fo, W) + amp F + amp0 Zia + P for an excited-state intermediate tuple (Fv, Fo, W, F, Zia, P:
        R1inter / es_L1inter); shifted: the device Fv, Fo of an update (_q6).  Returns it and the device amp."""
        ops = self.ops
        o, v = self.nocc, self.nvir
        d = ops.to_dev(amp)
        Fv, Fo = shifted or (ops.to_dev(inter[0]), ops.to_dev(inter[1]))
        R = core(d, Fv, Fo, self._w_dev(inter, 2, (v, o, o, v)))
        ops.scale_add(R, d, _scalar(inter[3]))
        ops.scale_add(R, ops.to_dev(inter[4]), _scalar(amp0))
        ops.scale_add(R, ops.to_dev(inter[5]), 1.0)
        return R, d

    def Extract_Em_r(self, rs, r0, Rinter, ov=None):       # CCS.py:874-906
        ops = self.ops
        rs = np.asarray(rs)
        if ov is None:
            o, v = np.unravel_index(np.argmax(abs(rs), axis=None), rs.shape)
        else:
            o, v = ov
        R, _ = self._es1full(self._r1core, rs, r0, Rinter)
        q = ops.to_host(R)
        return _like_amp0(q[o, v] / rs[o, v], r0), o, v

    def rsupdate(self, rs, r0, Rinter, Em, force_alpha=True):   # CCS.py:908-943
        ops = self.ops
        R, d_rs = self._es1full(self._r1core, rs, r0, Rinter, self._q6(Rinter[0], Rinter[1]))   # CCS.py:927-928
        new = ops.denom(R, d_rs, shift=float(np.asarray(Em).reshape(-1)[0]))
        if force_alpha:
            ops.fill(new[0::2, :], 0.0)                    # force alpha transition (Q9)
        return ops.to_host(new)

    def get_ov(self, ls, l0, rs, r0, ind):                 # CCS.py:945-963
        ops = self.ops
        o, v = ind
        ls = np.asarray(ls)
        rs = np.asarray(rs)
        d_r = ops.to_dev(rs).clone()
        for i, a in zip(np.ravel(o), np.ravel(v)):         # scalars, or the index arrays of np.where (Solver_ES.py:172)
            ops.fill(d_r[int(i):int(i) + 1, int(a):int(a) + 1], 0.0)
        rov = 1. - r0 * l0 - ops.dot(d_r, ops.to_dev(ls))
        return rov / ls[o, v]

    def R1eq(self, rs, r0, Rinter):                        # CCS.py:965-985
        R, _ = self._es1full(self._r1core, rs, r0, Rinter)
        return self.ops.to_host(R)

    def R0inter(self, ts, fsp, vm):                        # CCS.py:987-1034
        ops = self.ops
        o = self.nocc
        d_ts = ops.to_dev(ts)
        foo, fov, fvo, fvv = self.eris.fock_blocks(self.fock if fsp is None else fsp)
        Fjb = ops.copy(fov)
        ops.contract('kc,kjcb->jb', d_ts, self.eris.block("oovv"), out=Fjb, beta=1.0)
        E = ops.dot(d_ts, fov) + 0.5 * ops.dot(d_ts, self._G(d_ts))
        d_v = ops.to_dev(vm)
        P = ops.trace(d_v[:o, :o]) + ops.dot(d_ts, d_v[:o, o:])
        return ops.to_host(Fjb), E, P

    def Extract_r0(self, r1, ts, fsp, vm):                 # CCS.py:1036-1079
        """r0 from the R1 and R0 equations for a given r1 — contractions on the device, the scalar quadratic on the
        host exactly as the reference writes it (roots divided by c, `0` when c == 0., ValueError when both roots are
        negative; the square root of a negative discriminant is numpy's nan + RuntimeWarning, as there)."""
        r1 = np.asarray(r1)
        f = self.fock if fsp is None else fsp
        Rinter = self.R1inter(ts, f, vm)
        Fjb, Z, P = self.R0inter(ts, f, vm)
        R, d_rs = self._es1full(self._r1core, r1, 0.0, Rinter)  # Fab.r1 - Fji.r1 + W.r1 + r1 F + Pia (r0 = 0: no Zia term)
        R1 = self.ops.to_host(R)
        Zia = np.asarray(Rinter[4])
        c = -self.ops.dot(d_rs, self.ops.to_dev(Fjb)) - P
        if c == 0.:
            return 0
        i, j = np.unravel_index(np.argmax(abs(r1), axis=None), r1.shape)
        a = Zia[i, j] / r1[i, j]
        b = R1[i, j] / r1[i, j]
        b -= Z
        r0_1 = (-b + np.sqrt((b ** 2) - (4 * a * c))) / c
        r0_2 = (-b - np.sqrt((b ** 2) - (4 * a * c))) / c
        if r0_1 > 0:
            return r0_1
        elif r0_2 > 0:
            return r0_2
        raise ValueError('Both solution for r0 are negative')

    def r0update(self, rs, r0, Em, R0inter):               # CCS.py:1081-1096
        Fjb, E, P = R0inter
        F = self.ops.dot(self.ops.to_dev(rs), self.ops.to_dev(Fjb))
        return (F + P + (r0 * E)) / Em

    def R0eq(self, rs, r0, R0inter):                       # CCS.py:1098-1114
        Fjb, E, P = R0inter
        return self.ops.dot(self.ops.to_dev(rs), self.ops.to_dev(Fjb)) + r0 * E + P

    def r0_fromE(self, En, t1, r1, vm0, fsp=None):         # CCS.py:1116-1158
        ops = self.ops
        o = self.nocc
        d_t, d_r = ops.to_dev(t1), ops.to_dev(r1)
        foo, fov, fvo, fvv = self.eris.fock_blocks(self.fock if fsp is None else fsp)
        G = self._G(d_t)
        d = En - ops.dot(d_t, fov) - 0.5 * ops.dot(d_t, G)
        r0 = ops.dot(d_r, fov) + ops.dot(d_r, G)           # 'kc,jb,jkbc' = r1 . G (oovv[jkbc] = oovv[kjcb])
        if vm0 is not None:
            d_v = ops.to_dev(vm0)
            r0 += -ops.dot(d_t, d_v[:o, o:]) - ops.trace(d_v[:o, :o])
        return r0 / d

    # ------------------------------------------------------------------ ES left (CCS.py:1164-1518)
    def es_L1inter(self, ts, fsp, vm):
        ops = self.ops
        o = self.nocc
        F, W, X, El = self._inter("esl1", ts, fsp, vm)
        host = (ops.to_host(F[o:, o:]), ops.to_host(F[:o, :o]), ops.to_host(W), El, ops.to_host(F[:o, o:]),
                ops.to_host(X))                                                          # Fba, Fij, W, El, Zia, P
        return self._pack(host, W, 2)

    def L0inter(self, ts, fsp, vm):                        # CCS.py:1236-1286
        ops, B = self.ops, self.eris.block
        o = self.nocc
        d_ts = ops.to_dev(ts)
        foo, fov, fvo, fvv = self.eris.fock_blocks(self.fock if fsp is None else fsp)
        Fbj = ops.copy(fvo)
        ops.contract('kb,kj->bj', d_ts, foo, alpha=-1.0, out=Fbj, beta=1.0)
        ops.contract('ja,ba->bj', d_ts, fvv, out=Fbj, beta=1.0)
        q = ops.contract('kb,kc->bc', d_ts, fov)                                             # 'jc,kb,kc->bj'
        ops.contract('jc,bc->bj', d_ts, q, alpha=-1.0, out=Fbj, beta=1.0)
        x = ops.copy(B("ovov_ph"), 'jbkc->kbcj', alpha=-1.0)                                  # ovvo[kbcj] = -ovov[kbjc]
        a = ops.contract('lb,lkcd->bkcd', d_ts, B("oovv"))                                   # 'lb,jd,lkcd->kbcj'
        ops.contract('jd,bkcd->kbcj', d_ts, a, out=x, beta=1.0)
        ops.contract('lb,kljc->kbcj', d_ts, B("ooov"), out=x, beta=1.0)                      # -(oovo[klcj] = -ooov[kljc])
        ops.contract('jd,kbcd->kbcj', d_ts, B("ovvv"), out=x, beta=1.0)
        Wjb = ops.contract('kc,kbcj->jb', d_ts, x)
        Z = ops.dot(d_ts, fov) + 0.5 * ops.dot(d_ts, self._G(d_ts))
        d_v = ops.to_dev(vm)
        P = ops.dot(d_ts, d_v[:o, o:]) + ops.trace(d_v[:o, :o])
        return ops.to_host(Fbj), ops.to_host(Wjb), Z, P

    def _l1core(self, d_ls, Fba, Fij, W):
        ops = self.ops
        L = ops.contract('ib,ba->ia', d_ls, Fba)
        ops.contract('ja,ij->ia', d_ls, Fij, alpha=-1.0, out=L, beta=1.0)
        ops.contract('jb,bija->ia', d_ls, W, out=L, beta=1.0)
        return L

    def Extract_Em_l(self, ls, l0, L1inter, ov=None):      # CCS.py:1288-1319
        ls = np.asarray(ls)
        if ov is None:
            o, v = np.unravel_index(np.argmax(abs(ls), axis=None), ls.shape)
        else:
            o, v = ov
        L = self.ops.to_host(self._es1full(self._l1core, ls, l0, L1inter)[0])
        return _like_amp0(L[o, v] / ls[o, v], l0), o, v

    def Extract_l0(self, l1, ts, fsp, vm):
        raise EcwError("Extract_l0 is broken in the reference (operator precedence '/ 2*c', CCS.py:1356-1357) "
                       "and unused by any solver; not provided")

    def es_lsupdate(self, ls, l0, Em, L1inter, force_alpha=True):   # CCS.py:1366-1399
        ops = self.ops
        L, d_ls = self._es1full(self._l1core, ls, l0, L1inter, self._q6(L1inter[0], L1inter[1]))   # CCS.py:1384-1385
        new = ops.denom(L, d_ls, shift=float(np.asarray(Em).reshape(-1)[0]))
        if force_alpha:
            ops.fill(new[0::2, :], 0.0)
        return ops.to_host(new)

    def es_L1eq(self, ls, l0, es_L1inter):                 # CCS.py:1401-1421
        return self.ops.to_host(self._es1full(self._l1core, ls, l0, es_L1inter)[0])

    def l0update(self, ls, l0, Em, L0inter):               # CCS.py:1423-1439
        ops = self.ops
        Fbj, Wjb, Z, P = L0inter
        d_ls = ops.to_dev(ls)
        F = ops.dot(d_ls, ops.to_dev(Fbj).t())
        W = ops.dot(d_ls, ops.to_dev(Wjb))
        return (F + W + P + (l0 * Z)) / Em

    def L0eq(self, ls, l0, L0inter):                       # CCS.py:1441-1457
        ops = self.ops
        Fbj, Wjb, El, P = L0inter
        d_ls = ops.to_dev(ls)
        return ops.dot(d_ls, ops.to_dev(Fbj).t()) + ops.dot(d_ls, ops.to_dev(Wjb)) + l0 * El + P

    def l0_fromE(self, En, t1, l1, v0m, fsp=None):         # CCS.py:1459-1518
        ops, B = self.ops, self.eris.block
        o = self.nocc
        d_t, d_l = ops.to_dev(t1), ops.to_dev(l1)
        foo, fov, fvo, fvv = self.eris.fock_blocks(self.fock if fsp is None else fsp)
        G = self._G(d_t)
        shift = 0.5 * ops.dot(d_t, G)
        if isinstance(En, np.ndarray):                     # Q12: `d = En; d -= ...` (CCS.py:1488-1490) changes the
            En -= shift                                    # caller's energy array — Solver_ES records it AFTER this call
            d = En
        else:
            d = En - shift
        l0 = ops.dot(d_l, fov)
        l0 += ops.dot(ops.contract('jb,ab->ja', d_t, fvv), d_l)                              # 'jb,ab,ja'
        l0 -= ops.dot(ops.contract('jb,kb->kj', d_l, d_t), foo)                              # 'jb,kb,kj'
        q = ops.contract('kb,kc->bc', d_t, fov)                                              # 'jc,kb,kc,jb'
        l0 -= ops.dot(ops.contract('jc,bc->jb', d_t, q), d_l)
        w = ops.contract('kc,jbkc->jb', d_t, B("ovov_ph"), alpha=-1.0)                       # ovvo[kbcj] = -ovov_ph[jbkc]
        l0 += ops.dot(d_l, w)
        x = ops.contract('jb,jd->bd', d_l, d_t)
        y = ops.contract('lc,klcd->kd', d_t, B("oovv"))                                      # 'bd,kb,lc,klcd'
        l0 += ops.dot(ops.contract('kb,kd->bd', d_t, y), x)
        m = ops.contract('jb,lb->jl', d_l, d_t)
        n2 = ops.contract('kc,kljc->jl', d_t, B("ooov"))                                     # -'jl,kc,klcj' oovo = +ooov
        l0 += ops.dot(m, n2)
        l0 += ops.dot(ops.contract('kc,kbcd->bd', d_t, B("ovvv")), x)                        # 'bd,kc,kbcd'
        if v0m is not None:
            d_v = ops.to_dev(v0m)
            l0 += ops.dot(d_t, d_v[:o, o:]) + ops.trace(d_v[:o, :o])
        return l0 / d


# ---------------------------------------------------------------------- module-level rdm1 (CCS.py:23-190)
def _need(mycc):
    if mycc is None:
        raise EcwError("the device rdm1 builders need the owning Gccs object (device context): "
                       "call Gccs.gamma / gamma_unsym / gamma_es / gamma_tr")
    return mycc.ops


def _assemble(ops, oo, ov, vo, vv, unit_occ):
    o, v = ov.shape
    dm = ops.empty(o + v, o + v)
    ops.axpby(1.0, oo, 'pq', 0.0, dm[:o, :o], 'pq')
    ops.axpby(1.0, ov, 'pq', 0.0, dm[:o, o:], 'pq')
    ops.axpby(1.0, vo, 'pq', 0.0, dm[o:, :o], 'pq')
    ops.axpby(1.0, vv, 'pq', 0.0, dm[o:, o:], 'pq')
    if unit_occ:
        diag = ops.torch.as_strided(dm, (o,), (dm.stride(0) + dm.stride(1),))
        ops.mul(1.0, None, None, 1.0, diag)
    return dm


def gamma_unsym_CCS(ts, ls, mycc=None):                    # CCS.py:23-48
    ops = _need(mycc)
    t, l = ops.to_dev(ts), ops.to_dev(ls)
    oo = ops.contract('ie,je->ij', t, l, alpha=-1.0)
    vv = ops.contract('ib,ia->ab', t, l)
    x = ops.contract('ib,jb->ij', t, l)                    # 'ja,ib,jb->ia'
    ov = ops.copy(t)
    ops.contract('ij,ja->ia', x, t, alpha=-1.0, out=ov, beta=1.0)
    return ops.to_host(_assemble(ops, oo, ov, l.t(), vv, True))


def _es_blocks(ops, t, l, r, r0k, l0n):                    # CCS.py:75-91 / 130-146
    oo = ops.contract('ie,je->ij', t, l, alpha=-r0k)
    ops.contract('ie,je->ij', r, l, alpha=-1.0, out=oo, beta=1.0)
    vo = ops.copy(l, 'ia->ai', alpha=r0k)
    vv = ops.contract('mb,ma->ab', t, l, alpha=r0k)
    ops.contract('mb,ma->ab', r, l, out=vv, beta=1.0)
    x = ops.contract('ja,jb->ab', t, l)
    ov = ops.contract('ib,ab->ia', t, x, alpha=-r0k)
    y = ops.contract('ie,me->im', r, l)                    # 'ma,ie,me->ia'
    ops.contract('im,ma->ia', y, t, alpha=-1.0, out=ov, beta=1.0)
    z = ops.contract('ie,me->im', t, l)                    # 'ie,ma,me->ia'
    ops.contract('im,ma->ia', z, r, alpha=-1.0, out=ov, beta=1.0)
    ops.scale_add(ov, t, 1.0)
    ops.scale_add(ov, r, l0n)
    return oo, ov, vo, vv


def gamma_es_CCS(ts, ln, rk, r0k, l0n, mycc=None):         # CCS.py:51-102
    ops = _need(mycc)
    t, l = ops.to_dev(ts), ops.to_dev(ln)
    if rk is None or _is_num(rk):
        r, r0k, l0n = ops.fill(ops.empty(*t.shape), 0.0), 1., 0.
    else:
        r = ops.to_dev(rk)
    return ops.to_host(_assemble(ops, *_es_blocks(ops, t, l, r, _scalar(r0k), _scalar(l0n)), unit_occ=True))


def gamma_tr_CCS(ts, ln, rk, r0k, l0n, mycc=None):         # CCS.py:105-154
    ops = _need(mycc)
    t, l = ops.to_dev(ts), ops.to_dev(ln)
    if rk is None or _is_num(rk) or r0k is None:
        r, r0k = ops.fill(ops.empty(*t.shape), 0.0), 1.
    else:
        r = ops.to_dev(rk)
    return ops.to_host(_assemble(ops, *_es_blocks(ops, t, l, r, _scalar(r0k), _scalar(l0n)), unit_occ=False))


def gamma_CCS(ts, ls, mycc=None):                          # CCS.py:157-190
    ops = _need(mycc)
    t, l = ops.to_dev(ts), ops.to_dev(ls)
    o, v = t.shape
    doo = ops.contract('ja,ia->ij', t, l, alpha=-1.0)
    dvv = ops.contract('ia,ib->ab', t, l)
    xtv = ops.contract('ie,me->im', t, l)
    dvoT = ops.copy(t)                                     # dvo^T[i,a]
    ops.contract('im,ma->ia', xtv, t, alpha=-1.0, out=dvoT, beta=1.0)
    oo = ops.copy(doo, alpha=0.5)
    ops.axpby(0.5, doo, 'ji', 1.0, oo, 'ij')
    vv = ops.copy(dvv, alpha=0.5)
    ops.axpby(0.5, dvv, 'ba', 1.0, vv, 'ab')
    ov = ops.copy(l, alpha=0.5)
    ops.scale_add(ov, dvoT, 0.5)
    return ops.to_host(_assemble(ops, oo, ov, ov.t(), vv, True))
