"""Host-side mirror of the reference `CCSD.GCC` class (CCSD.py:185-623).

Same constructor and method signatures as the reference so that the unchanged
solver loop (`Solver_GS.Solver_CCSD.SCF`, Solver_GS.py:621-742) drives the CUDA
kernels:  `gamma`, `energy`, `tupdate`, `lupdate`.  numpy arrays in -> fresh
numpy arrays out (inputs are never mutated); torch CUDA tensors in -> torch
CUDA tensors out (device-resident mode used by bench.py's `value` leg).
"""
import numpy as np

from ._lib import lib, EcwError, ECW_HAS_ALPHA, ECW_EQUATION, ECW_ANTISYM
from .devops import ArgBlocks
from .eris import DeviceEris


# Amplitudes whose antisymmetry defect max|x[ijab]+x[jiab]|, |x[ijab]+x[ijba]| is below this (times max(1, max|x|)) run
# the fully packed path (the defect only enters the result multiplied by O(1) integrals/amplitudes,
# far below the 1e-10 parity bar); anything larger — e.g. after an L1-regularised update, which
# breaks antisymmetry in the reference (utilities.py:59-67) — runs the general path.
ANTISYM_TOL = 1e-13


def _flags(alpha, equation, antisym=False):
    return ((ECW_HAS_ALPHA if alpha is not None else 0) | (ECW_EQUATION if equation else 0)
            | (ECW_ANTISYM if antisym else 0))


class GCC(object):
    TRACK_MIN_BYTES = 1 << 20   # smaller outputs are not worth a device copy kept alive
    # Shapes with o^2 v^2 up to this many elements (every molecular configuration of BASELINE.json) are bound by the
    # launch rate of the several hundred kernels of an evaluation, not by their run time.  Their calls go through
    # persistent argument blocks owned by this object — inputs copied in, results copied out (device to device,
    # microseconds) — so the pointer arguments of the C entry points never change and the library replays one CUDA
    # graph per function (include/ecw_b200.h, ecw_ctx_set_graphs).  Larger shapes pass the caller's tensors directly.
    STAGE_MAX_ELEMS = 1 << 24

    def __init__(self, eris, fock=None, device=None, assume_antisym=None, rank=0, world=1, group=None, gemm=None,
                 int8_digits=None, track_outputs=True):
        """:param eris: a `DeviceEris`, or any object with the reference's
        `Eris.geris` attribute surface (uploaded once).
        :param gemm, int8_digits: GEMM engine of the uploaded container ("int8" default / "dmma"; eris.py)
        :param track_outputs: returned host arrays are read-only and keep their device copies (see `_to_host`)
        :param assume_antisym: None (default) = measure the antisymmetry of the doubles amplitudes
        on the device at every call and pick the packed or the general path; True/False = force."""
        self.assume_antisym = assume_antisym
        if not isinstance(eris, DeviceEris):
            eris = DeviceEris.from_geris(eris, device=device, rank=rank, world=world, group=group, gemm=gemm,
                                         int8_digits=int8_digits)
        self.eris = eris
        self.ops = eris.ops
        self.nocc = eris.nocc
        if fock is None:                       # CCSD.py:196-198
            self.fock = eris.fock
        self.nvir = self.fock.shape[0] - self.nocc
        o, v, n = self.nocc, self.nvir, self.fock.shape[0]
        self._shapes = dict(t1=(o, v), t2=(o, o, v, v), l1=(o, v), l2=(o, o, v, v), fsp=(n, n), o1=(o, v),
                            o2=(o, o, v, v), rdm1=(n, n), e=(1,))    # arguments and results of the four entry points
        self._pin = {}
        self._tracked = {}      # id(host array this object returned) -> (weakref, its device copy)
        self._blocks = None     # ArgBlocks of the small-shape route (_stage)
        self.track_outputs = bool(track_outputs)
        self.h2d_bytes = 0      # bytes staged host->device / device->host by this object
        self.d2h_bytes = 0
        self.h2d_reused = 0     # bytes NOT copied because the device copy of a returned array was reused
        self.host_seconds = {"to_host_alloc": 0.0, "to_host_copy": 0.0}    # wall time of the result downloads

    # -- host <-> device staging ---------------------------------------------
    def _torch(self):
        import torch
        return torch

    def _to_dev(self, name, x, shape):
        """numpy -> device.  An array THIS OBJECT handed out (`_to_host`: read-only, so its contents cannot have
        changed) is not copied again: its device copy is reused — in the solver loop (Solver_GS.py:683-705) every
        amplitude a call receives is an array an earlier call returned.  Other arrays that already live in pinned
        host memory are DMA'd directly; the rest is staged through a persistent pinned buffer."""
        torch = self._torch()
        if isinstance(x, torch.Tensor):
            if x.dtype != torch.float64 or tuple(x.shape) != tuple(shape):
                raise ValueError("%s: expected float64 tensor of shape %s" % (name, (shape,)))
            return x.contiguous(), True
        ent = self._tracked.get(id(x)) if isinstance(x, np.ndarray) else None
        if ent is not None and ent[0]() is x and not x.flags.writeable and x.shape == tuple(shape):
            self.h2d_reused += x.nbytes
            return ent[1], False
        a = np.asarray(x, dtype=np.float64)
        if a.shape != tuple(shape):
            raise ValueError("%s: expected shape %s, got %s" % (name, tuple(shape), a.shape))
        self.h2d_bytes += a.nbytes
        if a.flags.c_contiguous and a.flags.writeable:
            t = torch.from_numpy(a)
            if t.is_pinned():
                return t.to(self.eris.device, non_blocking=True), False
        key = (name, tuple(shape))
        pin = self._pin.get(key)
        if pin is None:
            pin = torch.empty(shape, dtype=torch.float64, pin_memory=True)
            self._pin[key] = pin
        else:
            torch.cuda.current_stream(self.eris.device).synchronize()   # previous DMA out of this buffer
        pin.numpy()[...] = a
        return pin.to(self.eris.device, non_blocking=True), False

    def _to_host(self, *ts):
        """device -> fresh numpy arrays in pinned blocks of the context's download pool (devops.PinnedPool).  With
        `track_outputs` (default) the arrays of TRACK_MIN_BYTES or more are READ-ONLY and the object remembers their
        device copies for as long as the caller keeps the arrays (weak references): passing one back costs no transfer.
        (The reference returns writable arrays; its solvers never write into them — `GCC(..., track_outputs=False)`
        restores that.)"""
        import weakref
        import time
        torch = self._torch()
        pool = self.ops.pinned
        torch.cuda.current_stream(self.eris.device).synchronize()          # the results are complete
        t0 = time.perf_counter()
        outs = [pool.take(t.shape, t.dtype) for t in ts]
        t1 = time.perf_counter()
        for h, t in zip(outs, ts):
            h.copy_(t, non_blocking=True)
            self.d2h_bytes += t.numel() * 8
        torch.cuda.current_stream(self.eris.device).synchronize()
        self.host_seconds["to_host_alloc"] += t1 - t0
        self.host_seconds["to_host_copy"] += time.perf_counter() - t1
        arrs = [pool.hand_out(h) for h in outs]
        for a, t in zip(arrs, ts):
            if self.track_outputs and a.nbytes >= self.TRACK_MIN_BYTES:
                a.setflags(write=False)
                key = id(a)
                self._tracked[key] = (weakref.ref(a, lambda _r, k=key, d=self._tracked: d.pop(k, None)), t)
        return arrs[0] if len(arrs) == 1 else tuple(arrs)

    def to_numpy(self, t):
        """Download a device tensor the way every method of this class returns its results (pinned, read-only,
        device copy remembered)."""
        return self._to_host(t)

    def _stage(self):
        """Persistent argument blocks of the small-shape (CUDA-graph) route, or None."""
        o, v = self.nocc, self.nvir
        e = self.eris
        if o * o * v * v > self.STAGE_MAX_ELEMS or getattr(e, "world", 1) > 1:
            return None
        if self._blocks is None:
            self._blocks = ArgBlocks(e.device, **self._shapes)
        return self._blocks

    def antisym_stats(self, d_x):
        """(max |x[ijab]+x[jiab]|, |x[ijab]+x[ijba]|, max |x|) of a device doubles amplitude."""
        torch = self._torch()
        e = self.eris
        out = torch.zeros(2, dtype=torch.float64, device=e.device)
        if lib.ecw_antisym_defect(d_x.data_ptr(), self.nocc, self.nvir, out.data_ptr(), e.stream()) != 0:
            raise EcwError("ecw_antisym_defect failed")
        h = out.cpu()
        return float(h[0]), float(h[1])

    def antisym_defect(self, d_x):
        return self.antisym_stats(d_x)[0]

    def _is_antisym(self, *amps):
        """Packed path when every amplitude is antisymmetric to ANTISYM_TOL relative to max(1, max|x|)."""
        if self.assume_antisym is not None:
            return bool(self.assume_antisym)
        for a in amps:
            defect, amax = self.antisym_stats(a)
            if not defect <= ANTISYM_TOL * max(1.0, amax):
                return False
        return True

    def _fsp(self, fsp):
        n = self.nocc + self.nvir
        if fsp is None:
            return self.eris.fock_dev, True
        return self._to_dev("fsp", fsp, (n, n))

    def _call(self, func, launch, inputs, outputs, antisym=(), alpha=None, equation=False):
        """The sequence of the four entry points: upload `inputs` (name -> array; the first one decides between device
        and host results; "fsp" may be None = the Fock matrix), measure the antisymmetry of the doubles named in
        `antisym`, stage everything into the persistent blocks when the shape allows, allocate the `outputs`, and run
        launch(flags, pointers by name) through the guarded executor.  Returns (device results?, [outputs])."""
        torch = self._torch()
        e = self.eris
        shapes = self._shapes
        args, dev = {}, None
        for k, x in inputs.items():
            args[k], d = self._fsp(x) if k == "fsp" else self._to_dev(k, x, shapes[k])
            dev = d if dev is None else dev
        fl = _flags(alpha, equation, bool(antisym) and self._is_antisym(*(args[k] for k in antisym)))
        st = self._stage()
        if st is not None:
            args = dict(zip(args, st.put(**args)))
            outs = [st[k] for k in outputs]
        else:
            outs = [torch.empty(shapes[k], dtype=torch.float64, device=e.device) for k in outputs]
        p = {k: t.data_ptr() for k, t in list(args.items()) + list(zip(outputs, outs))}
        e.execute(func, fl, lambda: launch(fl, p), "ecw_ccsd_" + func)
        if st is not None:
            outs = [t.clone() for t in outs]
        return dev, outs

    # -- rdm1 (CCSD.py:204-208 -> :136-182) -------------------------------------
    def gamma(self, t1, t2, l1, l2):
        e = self.eris
        dev, outs = self._call("gamma", lambda fl, p: lib.ecw_ccsd_gamma(
            e._h, p["t1"], p["t2"], p["l1"], p["l2"], p["rdm1"], e.stream()),
            dict(t1=t1, t2=t2, l1=l1, l2=l2), ("rdm1",))
        return outs[0] if dev else self._to_host(*outs)

    # -- energy (CCSD.py:224-242) -------------------------------------------------
    def energy(self, t1, t2, fsp):
        e = self.eris
        dev, (out,) = self._call("energy", lambda fl, p: lib.ecw_ccsd_energy(
            e._h, p["t1"], p["t2"], p["fsp"], p["e"], e.stream()), dict(t1=t1, t2=t2, fsp=fsp), ("e",))
        if dev:
            return out[0]
        self.d2h_bytes += 8
        return float(out.cpu()[0])

    # -- T1/T2 (CCSD.py:248-338) ---------------------------------------------------
    def tupdate(self, t1, t2, fsp=None, alpha=None, equation=False):
        e = self.eris
        dev, outs = self._call("tupdate", lambda fl, p: lib.ecw_ccsd_tupdate(
            e._h, p["t1"], p["t2"], p["fsp"], e.fock_dev.data_ptr(), fl, float(alpha or 0.0), p["o1"], p["o2"],
            e.stream()), dict(t1=t1, t2=t2, fsp=fsp), ("o1", "o2"), ("t2",), alpha, equation)
        return tuple(outs) if dev else self._to_host(*outs)

    # -- L1/L2 (CCSD.py:419-535, Linter :543-623) --------------------------------------
    def lupdate(self, t1, t2, l1, l2, fsp=None, alpha=None, equation=False):
        e = self.eris
        dev, outs = self._call("lupdate", lambda fl, p: lib.ecw_ccsd_lupdate(
            e._h, p["t1"], p["t2"], p["l1"], p["l2"], p["fsp"], e.fock_dev.data_ptr(), fl, float(alpha or 0.0),
            p["o1"], p["o2"], e.stream()), dict(t1=t1, t2=t2, l1=l1, l2=l2, fsp=fsp), ("o1", "o2"), ("t2", "l2"),
            alpha, equation)
        return tuple(outs) if dev else self._to_host(*outs)

    # -- intermediates of the reference API (CCSD.py:207-208, 346-413, 543-623) ------------------
    # Not used by the fused tupdate/lupdate plans (which never form Wvvvv / wvvvo); provided so
    # that every public GCC method exists.  numpy in -> numpy out, arithmetic on the device
    # through the primitive ops (same index strings as the reference, canonical integral blocks).
    def _tau_dev(self, t2, t1a, t1b, fac=1.):
        ops = self.ops
        x = ops.contract('ia,jb->ijab', t1a, t1b, alpha=0.5 * fac)          # CCSD.py:348
        y = ops.copy(x)
        ops.axpby(-1.0, x, 'jiab', 1.0, y, 'ijab')                          # :349
        tau = ops.copy(y)
        ops.axpby(-1.0, y, 'ijba', 1.0, tau, 'ijab')                        # :350
        ops.add(tau, t2)                                                    # :351
        return tau

    def make_tau(self, t2, t1a, t1b, fac=1.):
        ops = self.ops
        return ops.to_host(self._tau_dev(ops.to_dev(t2), ops.to_dev(t1a), ops.to_dev(t1b), fac))

    def gamma_inter(self, t1, t2, l1, l2):                                  # CCSD.py:165-182
        ops = self.ops
        t1, t2, l1, l2 = (ops.to_dev(x) for x in (t1, t2, l1, l2))
        doo = ops.contract('ie,je->ij', l1, t1, alpha=-1.0)
        ops.contract('imef,jmef->ij', l2, t2, alpha=-0.5, out=doo, beta=1.0)
        dvv = ops.contract('ma,mb->ab', t1, l1)
        ops.contract('mnea,mneb->ab', t2, l2, alpha=0.5, out=dvv, beta=1.0)
        xt1 = ops.contract('mnef,inef->mi', l2, t2, alpha=0.5)
        xt2 = ops.contract('mnfa,mnfe->ae', t2, l2, alpha=0.5)
        ops.contract('ma,me->ae', t1, l1, out=xt2, beta=1.0)
        dvo = ops.contract('imae,me->ai', t2, l1)
        ops.contract('mi,ma->ai', xt1, t1, alpha=-1.0, out=dvo, beta=1.0)
        ops.contract('ie,ae->ai', t1, xt2, alpha=-1.0, out=dvo, beta=1.0)
        ops.add(dvo, t1, 1.0, 'ia->ai')
        return ops.to_host(doo), ops.to_host(l1), ops.to_host(dvo), ops.to_host(dvv)

    def cc_Fvv(self, t1, t2, fsp):                                          # CCSD.py:355-368
        ops, B = self.ops, self.eris.block
        t1, t2 = ops.to_dev(t1), ops.to_dev(t2)
        foo, fov, fvo, fvv = self.eris.fock_blocks(fsp)
        tt = self._tau_dev(t2, t1, t1, fac=0.5)
        Fae = ops.copy(fvv)
        ops.contract('me,ma->ae', fov, t1, alpha=-0.5, out=Fae, beta=1.0)
        ops.contract('mf,maef->ae', t1, B("ovvv"), alpha=-1.0, out=Fae, beta=1.0)      # vovv[amef] = -ovvv[maef]
        ops.contract('mnaf,mnef->ae', tt, B("oovv"), alpha=-0.5, out=Fae, beta=1.0)
        return ops.to_host(Fae)

    def cc_Foo(self, t1, t2, fsp):                                          # CCSD.py:370-381
        ops, B = self.ops, self.eris.block
        t1, t2 = ops.to_dev(t1), ops.to_dev(t2)
        foo, fov, fvo, fvv = self.eris.fock_blocks(fsp)
        tt = self._tau_dev(t2, t1, t1, fac=0.5)
        Fmi = ops.copy(foo)
        ops.contract('me,ie->mi', fov, t1, alpha=0.5, out=Fmi, beta=1.0)
        ops.contract('ne,mnie->mi', t1, B("ooov"), out=Fmi, beta=1.0)
        ops.contract('inef,mnef->mi', tt, B("oovv"), alpha=0.5, out=Fmi, beta=1.0)
        return ops.to_host(Fmi)

    def cc_Fov(self, t1, t2, fsp):                                          # CCSD.py:383-387
        ops, B = self.ops, self.eris.block
        t1 = ops.to_dev(t1)
        foo, fov, fvo, fvv = self.eris.fock_blocks(fsp)
        Fme = ops.copy(fov)
        ops.contract('nf,mnef->me', t1, B("oovv"), out=Fme, beta=1.0)
        return ops.to_host(Fme)

    def cc_Woooo(self, t1, t2):                                             # CCSD.py:389-394
        ops, B = self.ops, self.eris.block
        t1, t2 = ops.to_dev(t1), ops.to_dev(t2)
        tau = self._tau_dev(t2, t1, t1)
        tmp = ops.contract('je,mnie->mnij', t1, B("ooov"))
        W = ops.copy(B("oooo"))
        ops.add(W, tmp)
        ops.axpby(-1.0, tmp, 'mnji', 1.0, W, 'mnij')
        ops.contract('ijef,mnef->mnij', tau, B("oovv"), alpha=0.25, out=W, beta=1.0)
        return ops.to_host(W)

    def _vvvv_dense(self):
        ops = self.ops
        v = self.nvir
        if self.eris.world != 1:
            raise EcwError("dense vvvv is not available on a sharded context")
        pv = v * (v - 1) // 2
        if "vvvv_p" not in self.eris.buf:
            raise EcwError("dense vvvv is not available: the packed vvvv is held as INT8 digit planes only "
                           "(DeviceEris.synthetic(..., keep_fp64_vvvv=True) keeps the FP64 layout)")
        return ops.unpack(self.eris.buf["vvvv_p"][: pv * pv].view(pv, pv), 3, ops.empty(v, v, v, v))

    def cc_Wvvvv(self, t1, t2):                                             # CCSD.py:396-402 (small sizes only: v^4)
        ops, B = self.ops, self.eris.block
        t1, t2 = ops.to_dev(t1), ops.to_dev(t2)
        tau = self._tau_dev(t2, t1, t1)
        tmp = ops.contract('mb,mafe->bafe', t1, B("ovvv"))
        W = self._vvvv_dense()
        ops.add(W, tmp, -1.0)
        ops.axpby(1.0, tmp, 'bafe', 1.0, W, 'abfe')
        ops.contract('mnab,mnef->abef', tau, B("oovv"), alpha=0.25, out=W, beta=1.0)
        return ops.to_host(W)

    def _wovvo_dev(self, t1, t2):
        ops, B = self.ops, self.eris.block
        W = ops.contract('jf,mbef->mbej', t1, B("ovvv"))                                    # CCSD.py:408
        ops.contract('nb,mnje->mbej', t1, B("ooov"), out=W, beta=1.0)                       # -(oovo = -ooov)
        ops.contract('jnfb,mnef->mbej', t2, B("oovv"), alpha=-0.5, out=W, beta=1.0)
        x = ops.contract('jf,mnef->mnej', t1, B("oovv"))
        ops.contract('nb,mnej->mbej', t1, x, alpha=-1.0, out=W, beta=1.0)
        ops.axpby(-1.0, B("ovov_ph"), 'jbme', 1.0, W, 'mbej')                               # ovvo[mbej] = -ovov[mbje]
        return W

    def cc_Wovvo(self, t1, t2):                                             # CCSD.py:404-413
        ops = self.ops
        return ops.to_host(self._wovvo_dev(ops.to_dev(t1), ops.to_dev(t2)))

    def Linter(self, t1, t2, fsp=None):                                     # CCSD.py:543-623
        ops, B = self.ops, self.eris.block
        t1, t2 = ops.to_dev(t1), ops.to_dev(t2)
        foo, fov, fvo, fvv = self.eris.fock_blocks(fsp)
        tau = ops.contract('ia,jb->ijab', t1, t1, alpha=2.0)
        ops.add(tau, t2)
        v1 = ops.copy(fvv)
        ops.contract('ja,jb->ba', fov, t1, alpha=-1.0, out=v1, beta=1.0)
        ops.contract('jbac,jc->ba', B("ovvv"), t1, alpha=-1.0, out=v1, beta=1.0)
        ops.contract('jkca,jkbc->ba', B("oovv"), tau, alpha=0.5, out=v1, beta=1.0)
        v2 = ops.copy(foo)
        ops.contract('ib,jb->ij', fov, t1, out=v2, beta=1.0)
        ops.contract('kijb,kb->ij', B("ooov"), t1, alpha=-1.0, out=v2, beta=1.0)
        ops.contract('ikbc,jkbc->ij', B("oovv"), tau, alpha=0.5, out=v2, beta=1.0)
        v3 = ops.contract('ijcd,klcd->ijkl', B("oovv"), tau)
        v4 = ops.contract('ljdb,klcd->jcbk', B("oovv"), t2)
        ops.axpby(-1.0, B("ovov_ph"), 'kcjb', 1.0, v4, 'jcbk')                              # ovvo[jcbk] = -ovov[jckb]
        v5 = ops.copy(fvo)
        ops.contract('kc,jkbc->bj', fov, t2, out=v5, beta=1.0)
        tmp = ops.copy(fov)
        ops.contract('kldc,ld->kc', B("oovv"), t1, alpha=-1.0, out=tmp, beta=1.0)
        q = ops.contract('kc,jc->kj', tmp, t1)                                              # 'kc,kb,jc->bj'
        ops.contract('kb,kj->bj', t1, q, out=v5, beta=1.0)
        ops.contract('kljc,klbc->bj', B("ooov"), t2, alpha=-0.5, out=v5, beta=1.0)
        ops.contract('kbdc,jkcd->bj', B("ovvv"), t2, alpha=0.5, out=v5, beta=1.0)
        w3 = ops.copy(v5)
        ops.contract('jcbk,jb->ck', v4, t1, out=w3, beta=1.0)
        ops.contract('cb,jb->cj', v1, t1, out=w3, beta=1.0)
        ops.contract('jk,jb->bk', v2, t1, alpha=-1.0, out=w3, beta=1.0)
        woooo = ops.copy(B("oooo"), alpha=0.5)
        ops.add(woooo, v3, 0.25)
        ops.contract('jilc,kc->jilk', B("ooov"), t1, out=woooo, beta=1.0)
        wovvo = ops.copy(v4)
        s1 = ops.contract('ljdb,kd->ljbk', B("oovv"), t1)                                   # 'ljdb,lc,kd->jcbk'
        ops.contract('ljbk,lc->jcbk', s1, t1, alpha=-1.0, out=wovvo, beta=1.0)
        ops.contract('ljkb,lc->jcbk', B("ooov"), t1, alpha=-1.0, out=wovvo, beta=1.0)
        ops.contract('jcbd,kd->jcbk', B("ovvv"), t1, out=wovvo, beta=1.0)
        wovoo = ops.contract('icdb,jkdb->icjk', B("ovvv"), tau, alpha=0.25)
        ops.axpby(0.5, B("ooov"), 'jkic', 1.0, wovoo, 'icjk')
        ops.contract('icbk,jb->icjk', v4, t1, out=wovoo, beta=1.0)
        ops.contract('lijb,klcb->icjk', B("ooov"), t2, alpha=-1.0, out=wovoo, beta=1.0)
        wvvvo = ops.contract('jcak,jb->bcak', v4, t1)
        ops.contract('jlka,jlbc->bcak', B("ooov"), tau, alpha=0.25, out=wvvvo, beta=1.0)
        ops.axpby(-0.5, B("ovvv"), 'jacb', 1.0, wvvvo, 'bcaj')
        ops.contract('kbad,jkcd->bcaj', B("ovvv"), t2, out=wvvvo, beta=1.0)
        G = ops.contract('menf,nf->me', B("oovv_ph"), t1)
        E = ops.dot(fov, t1) + 0.25 * ops.dot(t2, B("oovv")) + 0.5 * ops.dot(t1, G)

        class _IMDS:
            pass
        imds = _IMDS()
        imds.woooo, imds.wovvo, imds.wovoo, imds.wvvvo = (ops.to_host(x) for x in (woooo, wovvo, wovoo, wvvvo))
        imds.v1, imds.v2, imds.w3, imds.E = ops.to_host(v1), ops.to_host(v2), ops.to_host(w3), E
        return imds

    # -- introspection ---------------------------------------------------------------
    def plan_json(self, func, alpha=None, equation=False, antisym=True):
        import ctypes
        fl = _flags(alpha, equation, antisym)
        n = 1 << 22
        while True:
            buf = ctypes.create_string_buffer(n)
            r = lib.ecw_plan_dump(self.eris._h, func.encode(), fl, buf, n)
            if r >= 0:
                return buf.value.decode()
            if r == -1:
                self.eris.check(-1, "ecw_plan_dump")
            n = int(-r) + 16

    def plan_flops(self, func, alpha=None, equation=False, antisym=True):
        return lib.ecw_plan_flops(self.eris._h, func.encode(), _flags(alpha, equation, antisym))

    def plan_launches(self, func, alpha=None, equation=False, antisym=True):
        return lib.ecw_plan_launches(self.eris._h, func.encode(), _flags(alpha, equation, antisym))


def gamma_CCSD(t1, t2, l1, l2, mycc=None):
    """Module-level rdm1 of the reference (CCSD.py:136-162); needs a GCC for the device context."""
    if mycc is None:
        raise EcwError("gamma_CCSD needs the owning GCC object (device context)")
    return mycc.gamma(t1, t2, l1, l2)
