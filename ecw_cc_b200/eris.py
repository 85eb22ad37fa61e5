"""Device-resident integral container.

Consumes the attribute surface of the reference `Eris.geris` (Eris.py:132-154:
`fock, nocc, oooo, ooov, oovv, ovov, ovvv, vvvv`, numpy arrays of
antisymmetrised <pq||rs>) and keeps the constant layouts the kernels read
(include/ecw_b200.h, "integral container").  Construction of integrals from a
molecule (PySCF ao2mo, Eris.py:47-128) is out of scope.
"""
import ctypes
import os
import weakref

import numpy as np

from ._lib import lib, EcwError

_LAYOUTS = ("oooo", "ooov", "oovv", "ovvv", "oovv_ph", "ovov_ph", "oooo_p", "oovv_p", "ovvv_p", "vvvv_p")
SYNTH_KIND = dict(oooo=0, ooov=1, oovv=2, oovv_ph=3, ovov_ph=4, ovvv=5, oooo_p=6, oovv_p=7, ovvv_p=8, vvvv_p=9,
                  fock=10, fsp=11, t1=12, l1=13, t2=14, l2=15)
_BLOCK_INDEX = dict(oooo="oooo", ooov="ooov", oovv="oovv", ovvv="ovvv", ovov_ph="ovov", oovv_ph="ovov")


# GEMM engine of the contraction plans (include/ecw_b200.h, ecw_ctx_set_gemm):
#   "int8" (default) - large unbatched GEMMs on the INT8 tcgen05 tensor pipe: FP64 operands cut into
#                      base-256 int8 digits (csrc/ozaki.cu); the packed vvvv lives on the device as digit
#                      planes only;
#   "dmma"           - everything on the FP64 DMMA kernels.
# Digits: 6 (48 bits) when the worst-case error bound of the longest contraction (the pp ladder, K = P_v),
#   4 (NS+3) 256^-NS K max|<pq||rs>| max|tau|  with max|tau| taken as 1/4, stays below AUTO_DIGIT_BOUND; else 7 (or 8).
# Environment overrides for experiments: ECW_GEMM, ECW_INT8_DIGITS, ECW_INT8_MIN_FLOPS (-1: every GEMM).
INT8_MIN_FLOPS = 2e10
AUTO_DIGIT_BOUND = 5e-11
# Run-time guard (include/ecw_b200.h, ecw_int8_error_bound): after every call the worst-case absolute error of its INT8
# products, (NS+3) 256^-NS K |alpha| max s_m max s_n from the row scales actually cut, is read back.  Above INT8_TOL the
# call is repeated on the FP64 DMMA kernels when the FP64 integral layouts are on the device (containers built with
# from_geris, or synthetic(..., keep_fp64_vvvv=True)); otherwise it fails loudly (rebuild with more digits).  The bound
# is a strict worst case (every digit error aligned): half the 1e-10 parity bar; observed errors are >= 100x smaller
# (they add like a random walk over K: profiles/r1_engine_check_40_400.json, 1.8e-12 at the benchmark shape).
INT8_TOL = 5e-11


def auto_digits(nvir, eri_max):
    k = nvir * (nvir - 1) // 2
    for nd in (6, 7):
        if 4.0 * (nd + 3) * 256.0 ** (-nd) * k * float(eri_max) * 0.25 <= AUTO_DIGIT_BOUND:
            return nd
    return 8


def _gemm_config(gemm, int8_digits, int8_min_flops, nvir, eri_max):
    gemm = gemm or os.environ.get("ECW_GEMM", "int8")
    if gemm not in ("int8", "dmma"):
        raise ValueError("gemm must be 'int8' or 'dmma', got %r" % (gemm,))
    if gemm == "dmma":
        return 0, 0.0
    nd = int8_digits if int8_digits is not None else os.environ.get("ECW_INT8_DIGITS")
    nd = int(nd) if nd is not None else auto_digits(nvir, eri_max)
    mf = float(int8_min_flops if int8_min_flops is not None else os.environ.get("ECW_INT8_MIN_FLOPS", INT8_MIN_FLOPS))
    return nd, mf


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: the ECW-CC residual path has no CPU implementation")
    return torch


class TorchDistComm(object):
    """Collectives of a sharded call over torch.distributed (NCCL over NVLink between the GPUs of one box)."""

    def __init__(self, group=None):
        self.group = group

    def all_gather(self, eris, recv, send):
        import torch.distributed as dist
        dist.all_gather_into_tensor(recv, send, group=self.group)

    def all_to_all(self, eris, recv, send):
        """block q of `send` goes to rank q, block q of `recv` comes from rank q"""
        import torch.distributed as dist
        dist.all_to_all_single(recv, send, group=self.group)

    def max_scalar(self, eris, x):
        """max over ranks of a one-element device tensor -> float"""
        import torch.distributed as dist
        dist.all_reduce(x, op=dist.ReduceOp.MAX, group=self.group)
        return float(x.cpu()[0])


class DeviceEris(object):
    """Owns the C context, the bound integral layouts and the workspace."""

    def __init__(self, nocc, nvir, device=None, rank=0, world=1, group=None, gemm=None, int8_digits=None,
                 int8_min_flops=None, eri_max=1.0, ovvv_planes=None, int8_tol=None):
        """rank/world/group: one process per GPU; `vvvv_p` is then row-sharded over the packed
        virtual pair index and the heavy contractions are distributed (include/ecw_b200.h).
        gemm: "int8" | "dmma"; int8_digits: None = chosen from eri_max = max |<pq||rs>| (module header)."""
        torch = _torch()
        self.nocc = int(nocc)
        self.nvir = int(nvir)
        self.rank, self.world, self.group = int(rank), int(world), group
        self.comm = TorchDistComm(group)     # who performs the collectives of a sharded call (tests: virtual ranks)
        self.own_nccl = False                # the context holds its own ncclComm_t (init_nccl)
        self.device = torch.device(device if device is not None else ("cuda:%d" % torch.cuda.current_device()))
        self._h = ctypes.c_void_p()
        if lib.ecw_ctx_create(ctypes.byref(self._h), self.nocc, self.nvir) != 0:
            raise EcwError("ecw_ctx_create failed")
        if self.world > 1 and lib.ecw_ctx_set_shard(self._h, self.rank, self.world) != 0:
            raise EcwError("ecw_ctx_set_shard failed")
        self.int8_digits, self.int8_min_flops = _gemm_config(gemm, int8_digits, int8_min_flops, self.nvir, eri_max)
        self.check(lib.ecw_ctx_set_gemm(self._h, self.int8_digits, self.int8_min_flops), "ecw_ctx_set_gemm")
        # constant digit planes of ovvv_p (both orientations): sub-blocks of a plane set start on 8-row groups
        if ovvv_planes is None:
            ovvv_planes = os.environ.get("ECW_OVVV_PLANES", "1") != "0"
        self.use_ovvv_planes = bool(ovvv_planes and self.int8_digits and self.nocc % 8 == 0 and self.nvir % 8 == 0)
        self.int8_tol = float(os.environ.get("ECW_INT8_TOL", INT8_TOL) if int8_tol is None else int8_tol)
        self.guard_trips = 0      # calls whose INT8 error bound exceeded int8_tol (each was repeated on DMMA)
        self.last_bound = 0.0     # bound of the last guarded call (a plan or a primitive contraction)
        self.max_bound = 0.0      # the largest finite bound of those calls that stayed within int8_tol
        self.buf = {}
        self._views = {}          # block(): shaped views of the canonical integral blocks
        self._ops = None
        self._ws = None
        self._scal = torch.zeros(16, dtype=torch.float64, device=self.device)
        self._bind("scal", self._scal)
        self.fock = None          # host numpy (reference attribute `eris.fock`)
        self.fock_dev = None
        self.mo_occ = np.concatenate([np.ones(self.nocc), np.zeros(self.nvir)])
        self.EHF = 0.0

    # -- plumbing ------------------------------------------------------------
    def __del__(self):
        try:
            if self._h:
                lib.ecw_ctx_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def check(self, rc, what):
        if rc != 0:
            msg = lib.ecw_last_error(self._h)
            raise EcwError("%s: %s" % (what, msg.decode() if msg else "error"))

    def stream(self):
        return _torch().cuda.current_stream(self.device).cuda_stream

    def _bind(self, name, tensor):
        self.check(lib.ecw_bind(self._h, name.encode(), tensor.data_ptr()), "ecw_bind(%s)" % name)

    def _alloc_layout(self, name):
        torch = _torch()
        n = lib.ecw_slot_elems(self._h, name.encode())
        if n < 0:
            raise EcwError("unknown layout %s" % name)
        t = torch.empty(max(int(n), 1), dtype=torch.float64, device=self.device)
        self.buf[name] = t
        self._bind(name, t)
        return t

    def grow_workspace(self, nbytes):
        """Give the context a workspace of at least `nbytes` (never shrinks).  The stream is synchronised before the
        old buffer is dropped: work already enqueued may still read it."""
        if self._ws is not None and self._ws.numel() >= nbytes:
            return
        torch = _torch()
        if self._ws is not None:
            torch.cuda.current_stream(self.device).synchronize()
        self._ws = None
        self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        self.check(lib.ecw_set_workspace(self._h, self._ws.data_ptr(), self._ws.numel()), "ecw_set_workspace")

    def ensure_workspace(self, func, flags):
        need = lib.ecw_workspace_bytes(self._h, func.encode(), flags)
        if need < 0:
            self.check(-1, "ecw_workspace_bytes(%s)" % func)
        self.grow_workspace(max(int(need), 256))

    def run(self, rc, what):
        """Drive a (possibly distributed) call to completion: while the library reports a pending
        collective, perform it through `self.comm` (default: torch.distributed / NCCL on the workspace) and resume."""
        torch = _torch()
        while rc == 1:
            desc = (ctypes.c_int64 * 6)()
            if lib.ecw_pending_collective(self._h, desc) != 0:
                raise EcwError("%s: no pending collective" % what)
            kind, soff, count, roff, world, rank = [int(x) for x in desc]
            if kind not in (1, 2) or world != self.world:
                raise EcwError("%s: unexpected collective %r" % (what, list(desc)))
            ws = self._ws.view(torch.float64)
            if kind == 1:
                self.comm.all_gather(self, ws[roff: roff + world * count], ws[soff: soff + count])
            else:
                self.comm.all_to_all(self, ws[roff: roff + world * count], ws[soff: soff + world * count])
            rc = lib.ecw_resume(self._h, self.stream())
        self.check(rc, what)

    def init_nccl(self):
        """Give the context its own NCCL communicator (include/ecw_b200.h): rank 0 draws the unique id, torch.distributed
        broadcasts it, every rank joins.  The executor then enqueues the collectives itself.  Returns False (and keeps
        the host-driven protocol) when torch.distributed is not running on NCCL or ECW_HOST_COLLECTIVES=1."""
        torch = _torch()
        if self.world < 2 or os.environ.get("ECW_HOST_COLLECTIVES", "0") == "1":
            return False
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized() and dist.get_backend(self.group) == "nccl"):
            return False
        libdir = os.path.join(os.path.dirname(os.path.dirname(torch.__file__)), "nvidia", "nccl", "lib")
        path = os.path.join(libdir, "libnccl.so.2")
        path = path.encode() if os.path.exists(path) else b""
        ident = (ctypes.c_char * 128)()
        if self.rank == 0:
            self.check(lib.ecw_nccl_unique_id(path, ident), "ecw_nccl_unique_id")
        t = torch.frombuffer(bytearray(ident.raw), dtype=torch.uint8).to(self.device)
        src = dist.get_global_rank(self.group, 0) if self.group is not None else 0
        dist.broadcast(t, src=src, group=self.group)
        raw = bytes(t.cpu().numpy().tobytes())
        torch.cuda.current_stream(self.device).synchronize()
        self.check(lib.ecw_ctx_init_nccl(self._h, path, raw, self.rank, self.world), "ecw_ctx_init_nccl")
        self.own_nccl = True
        return True

    # -- guarded execution of one C entry point ----------------------------------------
    def int8_bound(self):
        """Worst-case absolute error of the INT8 products of the last call (max over ranks); NaN when an operand
        held a non-finite value."""
        torch = _torch()
        if self.world > 1:
            b = self._scal[15:16].clone()
            b = torch.where(torch.isnan(b), torch.full_like(b, float("inf")), b)
            v = self.comm.max_scalar(self, b)
            return float("nan") if v == float("inf") else v
        out = ctypes.c_double(0.0)
        self.check(lib.ecw_int8_error_bound(self._h, ctypes.byref(out), self.stream()), "ecw_int8_error_bound")
        return out.value

    def can_dmma(self):
        """The FP64 layouts the DMMA plans read are on the device."""
        return "vvvv_p" in self.buf and "ovvv_p" in self.buf

    def execute(self, func, flags, launch, what):
        """One plan call: `launch` (a closure around the C entry point) through `guarded`, with the workspace sized
        for the plan of `func` / `flags` before every launch."""
        self.guarded(launch, what, prepare=lambda: self.ensure_workspace(func, flags))

    def guarded(self, launch, what, prepare=None, repeat=True):
        """prepare() + launch() (a closure around a C entry point, returns its rc) + the INT8 accuracy guard: when the
        bound of the call exceeds int8_tol the same call is repeated without the INT8 route.  repeat=False: the call
        accumulates into its output (beta != 0), so a repeat would count its product twice; it raises instead.  A plan
        call (the calls with a prepare step) reads the FP64 integral layouts when it runs on DMMA: without them it
        raises too.  The primitive contractions only guard calls large enough for the INT8 route (DevOps.contract):
        on a sharded context reading the bound is a collective."""
        if prepare is not None:
            prepare()
        self.run(launch(), what)
        if not self.int8_digits or not self.int8_tol > 0.0:
            return
        b = self.last_bound = self.int8_bound()
        if b != b or b <= self.int8_tol:        # NaN: non-finite operands; the outputs are NaN as in the reference
            self.max_bound = max(self.max_bound, b) if b == b else self.max_bound
            return
        self.guard_trips += 1
        if not repeat:
            raise EcwError("%s: INT8 error bound %.2e > %.1e on an accumulating contraction; use more digits "
                           "(int8_digits) or gemm='dmma'" % (what, b, self.int8_tol))
        if prepare is not None and not self.can_dmma():
            raise EcwError("%s: the INT8 engine cannot guarantee its accuracy for these operands (worst-case error "
                           "bound %.2e > %.1e with %d digits) and the FP64 integral layouts are not on the device: "
                           "build the container with int8_digits=%d or gemm='dmma'"
                           % (what, b, self.int8_tol, self.int8_digits, min(self.int8_digits + 1, 8)))
        self.check(lib.ecw_ctx_set_engine_override(self._h, 1), "ecw_ctx_set_engine_override")
        try:
            if prepare is not None:
                prepare()
            self.run(launch(), what + " (FP64 DMMA after the INT8 guard)")
        finally:
            lib.ecw_ctx_set_engine_override(self._h, 0)

    def set_fock(self, fock):
        torch = _torch()
        self.fock = np.ascontiguousarray(fock, dtype=np.float64)
        self.fock_dev = torch.from_numpy(self.fock).to(self.device)

    # -- constructors ----------------------------------------------------------
    @classmethod
    def from_geris(cls, eris, device=None, rank=0, world=1, group=None, gemm=None, int8_digits=None,
                   int8_min_flops=None, ovvv_planes=None, int8_tol=None):
        """Upload a reference-style container (numpy blocks, Eris.py:132-150)."""
        torch = _torch()
        fock = np.asarray(eris.fock)
        nocc = int(eris.nocc)
        eri_max = max(float(np.abs(np.asarray(getattr(eris, k))).max()) if np.asarray(getattr(eris, k)).size else 0.0
                      for k in ("oooo", "ooov", "oovv", "ovov", "ovvv", "vvvv"))
        self = cls(nocc, fock.shape[0] - nocc, device, gemm=gemm, int8_digits=int8_digits,
                   int8_min_flops=int8_min_flops, eri_max=eri_max, ovvv_planes=ovvv_planes,
                   int8_tol=int8_tol)   # packed whole, sharded below
        self.set_fock(fock)
        for name in ("oooo", "ooov", "oovv", "ovvv"):
            t = torch.from_numpy(np.ascontiguousarray(getattr(eris, name), dtype=np.float64)).to(self.device)
            self.buf[name] = t.reshape(-1)
            self._bind(name, self.buf[name])
        for name in ("oovv_ph", "ovov_ph", "oooo_p", "oovv_p", "ovvv_p", "vvvv_p"):
            self._alloc_layout(name)
        ovov = torch.from_numpy(np.ascontiguousarray(eris.ovov, dtype=np.float64)).to(self.device)
        vvvv = torch.from_numpy(np.ascontiguousarray(eris.vvvv, dtype=np.float64)).to(self.device)
        self.check(lib.ecw_eris_pack_from_dense(self._h, ovov.data_ptr(), vvvv.data_ptr(), self.stream()),
                   "ecw_eris_pack_from_dense")
        torch.cuda.current_stream(self.device).synchronize()
        if world > 1:
            self.rank, self.world, self.group = int(rank), int(world), group
            self.comm = TorchDistComm(group)
            if lib.ecw_ctx_set_shard(self._h, self.rank, self.world) != 0:
                raise EcwError("ecw_ctx_set_shard failed")
            pv = self.nvir * (self.nvir - 1) // 2
            nshmax = (pv + world - 1) // world
            n0 = min(pv, rank * nshmax)
            n1 = min(pv, n0 + nshmax)
            shard = self.buf["vvvv_p"][n0 * pv: n1 * pv].clone() if n1 > n0 else torch.zeros(
                1, dtype=torch.float64, device=self.device)
            self.buf["vvvv_p"] = shard
            self._bind("vvvv_p", shard)
        if self.int8_digits:
            # a dense upload is small: the FP64 shard stays (cc_Wvvvv / Linter getters read it), the
            # residual plans read the digit planes
            self._cut_vvvv_planes(lambda r0, nr: self.buf["vvvv_p"][r0 * self._pv(): (r0 + nr) * self._pv()])
        if self.use_ovvv_planes:
            self._cut_ovvv_planes(keep_fp64=True)
        for attr in ("mo_occ", "EHF", "orbspin"):
            if hasattr(eris, attr):
                setattr(self, attr, getattr(eris, attr))
        self.init_nccl()
        return self

    @classmethod
    def synthetic(cls, nocc, nvir, device=None, scale=0.01, rank=0, world=1, group=None, gemm=None,
                  int8_digits=None, int8_min_flops=None, keep_fp64_vvvv=False, ovvv_planes=None, int8_tol=None):
        """Function-defined synthetic integrals generated in place on the device (each rank
        generates only its own rows of the packed vvvv).  With the INT8 engine the packed vvvv is
        generated in row chunks and kept as digit planes only (keep_fp64_vvvv: also the FP64 layout)."""
        torch = _torch()
        self = cls(nocc, nvir, device, rank=rank, world=world, group=group, gemm=gemm, int8_digits=int8_digits,
                   int8_min_flops=int8_min_flops, eri_max=abs(float(scale)), ovvv_planes=ovvv_planes, int8_tol=int8_tol)
        planes_only = bool(self.int8_digits) and not keep_fp64_vvvv
        for name in _LAYOUTS:
            if name == "vvvv_p" and planes_only:
                continue
            self._alloc_layout(name)
        self.check(lib.ecw_eris_synthetic(self._h, float(scale), self.stream()), "ecw_eris_synthetic")
        if self.int8_digits:
            if planes_only:
                n0 = self._shard_rows()[0]
                pv = self._pv()
                chunk_rows = max(128, min(4096, (1 << 28) // max(pv, 1) // 128 * 128))     # <= 2 GiB of FP64 rows
                tmp = torch.empty(chunk_rows * pv, dtype=torch.float64, device=self.device)

                def rows(r0, nr):
                    rc = lib.ecw_synth_tensor(SYNTH_KIND["vvvv_p"], tmp.data_ptr(), self.nocc, self.nvir, n0 + r0, nr,
                                              float(scale), self.stream())
                    if rc != 0:
                        raise EcwError("ecw_synth_tensor(vvvv_p rows) failed")
                    return tmp
                self._cut_vvvv_planes(rows, chunk_rows)
                del tmp
            else:
                self._cut_vvvv_planes(lambda r0, nr: self.buf["vvvv_p"][r0 * self._pv(): (r0 + nr) * self._pv()])
        if self.use_ovvv_planes:
            self._cut_ovvv_planes(keep_fp64=keep_fp64_vvvv)
        n = self.nocc + self.nvir
        self.fock_dev = self.synth_tensor("fock", (n, n))
        self.fock = self.fock_dev.cpu().numpy()
        torch.cuda.current_stream(self.device).synchronize()
        self.init_nccl()
        return self

    def _pv(self):
        return self.nvir * (self.nvir - 1) // 2

    def _shard_rows(self):
        """(first row, number of rows) of this rank's shard of the packed vvvv."""
        pv = self._pv()
        nshmax = (pv + self.world - 1) // self.world
        n0 = min(pv, self.rank * nshmax)
        return n0, min(pv, n0 + nshmax) - n0

    def _cut_vvvv_planes(self, rows_of, chunk_rows=None):
        """Cut this rank's packed-vvvv rows into int8 digit planes (ecw_eris_vvvv_planes).
        rows_of(r0, nr) -> device tensor holding the FP64 rows [r0, r0+nr) of the shard."""
        torch = _torch()
        nsh = self._shard_rows()[1]
        for name, dt, unit in (("vvvv_oz", torch.int8, 8), ("vvvv_ozs", torch.float64, 1)):
            n = lib.ecw_slot_elems(self._h, name.encode())
            if n < 0:
                self.check(-1, "ecw_slot_elems(%s)" % name)
            self.buf[name] = torch.empty(max(int(n), 1) * unit, dtype=dt, device=self.device)
            self._bind(name, self.buf[name])
        chunk_rows = int(chunk_rows or max(nsh, 1))
        r0 = 0
        while True:
            nr = min(chunk_rows, nsh - r0)
            src = rows_of(r0, nr) if nr > 0 else self.buf["vvvv_ozs"]
            self.check(lib.ecw_eris_vvvv_planes(self._h, src.data_ptr(), r0, nr, self.stream()), "ecw_eris_vvvv_planes")
            r0 += nr
            if r0 >= nsh:
                break
        torch.cuda.current_stream(self.device).synchronize()

    def _cut_ovvv_planes(self, keep_fp64=False):
        """ovvv_p -> int8 digit planes in both orientations (ecw_eris_ovvv_planes); the FP64 layout is then
        dropped unless keep_fp64."""
        torch = _torch()
        for name in ("ovvv_oz1", "ovvv_oz1s", "ovvv_oz2", "ovvv_oz2s"):
            n = lib.ecw_slot_elems(self._h, name.encode())
            if n < 0:
                self.check(-1, "ecw_slot_elems(%s)" % name)
            planes = not name.endswith("s")
            self.buf[name] = torch.empty(max(int(n), 1) * (8 if planes else 1),
                                         dtype=torch.int8 if planes else torch.float64, device=self.device)
            self._bind(name, self.buf[name])
        self.check(lib.ecw_eris_ovvv_planes(self._h, self.stream()), "ecw_eris_ovvv_planes")
        torch.cuda.current_stream(self.device).synchronize()
        if not keep_fp64:
            self.check(lib.ecw_bind(self._h, b"ovvv_p", None), "ecw_bind(ovvv_p)")
            del self.buf["ovvv_p"]

    def synth_tensor(self, kind, shape, scale=0.01):
        """Synthetic fock / fsp / t1 / l1 / t2 / l2 on the device."""
        torch = _torch()
        out = torch.empty(shape, dtype=torch.float64, device=self.device)
        rc = lib.ecw_synth_tensor(SYNTH_KIND[kind], out.data_ptr(), self.nocc, self.nvir, 0, int(shape[0]),
                                  float(scale), self.stream())
        if rc != 0:
            raise EcwError("ecw_synth_tensor(%s) failed" % kind)
        return out

    # -- device views, the primitive ops, the Fock blocks ---------------------------
    def block(self, name):
        """Device view of a canonical integral block in its index shape (ovov_ph / oovv_ph: [ia, jb] as (o, v, o, v))."""
        t = self._views.get(name)
        if t is None:
            shape = tuple(self.nocc if c == "o" else self.nvir for c in _BLOCK_INDEX[name])
            t = self._views[name] = self.buf[name][: int(np.prod(shape))].view(shape)
        return t

    @property
    def ops(self):
        """The primitive device ops of this context (one DevOps, shared by every class built on it)."""
        if self._ops is None:
            from .devops import DevOps
            self._ops = DevOps(weakref.proxy(self))    # no reference cycle: the context is freed with its last owner
        return self._ops

    def fock_blocks(self, fsp=None):
        """oo, ov, vo, vv views of the device one-body operator: fsp (uploaded when it is a host array) or the Fock
        matrix."""
        o = self.nocc
        F = self.fock_dev if fsp is None else self.ops.to_dev(fsp)
        return F[:o, :o], F[:o, o:], F[o:, :o], F[o:, o:]

    # -- reference attribute surface (host copies on demand) ----------------------
    @property
    def oovv(self):
        return self.block("oovv").cpu().numpy()

    @property
    def ooov(self):
        return self.block("ooov").cpu().numpy()

    @property
    def oooo(self):
        return self.block("oooo").cpu().numpy()

    @property
    def ovvv(self):
        return self.block("ovvv").cpu().numpy()
