"""Thin host wrapper over the primitive device ops of the C ABI (`ecw_op_*`,
include/ecw_b200.h): einsum-style contraction, axpby/permutes, element-wise
product, diagonal shift, denominators and dot products on torch CUDA tensors.
Torch only allocates the memory and provides the stream; every arithmetic
operation is one of this repo's kernels.
"""
import ctypes
import weakref

import numpy as np

from ._lib import lib


class _TensorDesc(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("nd", ctypes.c_int32),
                ("dim", ctypes.c_int64 * 6), ("str", ctypes.c_int64 * 6)]


def _desc(t):
    if t is None:
        return None
    d = _TensorDesc()
    d.ptr = t.data_ptr()
    d.nd = t.dim()
    for i in range(t.dim()):
        d.dim[i] = t.shape[i]
        d.str[i] = t.stride(i)
    return d


def _scalar(x):
    """Python float from a number or a one-element array (the solvers pass r0 / l0 / E as shape-(1,) arrays)."""
    return float(np.asarray(x, dtype=np.float64).reshape(-1)[0])


def _ref(d):
    return ctypes.byref(d) if d is not None else None


class PinnedPool(object):
    """Pinned host blocks for device -> host downloads (a pageable D2H runs at ~2.5 GB/s).  Page-locking gigabytes
    costs far more than the transfer itself (cudaHostAlloc), so the block of a returned array of MIN_BYTES or more
    goes back to the pool when the caller drops the array (per shape and dtype, at most DEPTH kept); smaller ones come
    from torch's caching host allocator."""
    MIN_BYTES = 1 << 20
    DEPTH = 4

    def __init__(self):
        self._free = {}

    def take(self, shape, dtype):
        import torch
        free = self._free.get((tuple(shape), dtype))
        if free:
            h = free.pop()
            del free[self.DEPTH:]
            return h
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    def hand_out(self, h):
        """numpy view of a filled block; a large block returns to the pool when the array is dropped."""
        a = h.numpy()
        if a.nbytes >= self.MIN_BYTES:
            weakref.finalize(a, self._free.setdefault((tuple(h.shape), h.dtype), []).append, h)
        return a


class ArgBlocks(object):
    """Persistent device argument blocks, name -> tensor.  A C entry point that always receives the same pointers
    replays its CUDA graph (include/ecw_b200.h, ecw_ctx_set_graphs) instead of launching its kernels one by one."""

    def __init__(self, device, **shapes):
        import torch
        self.blocks = {k: torch.empty(s, dtype=torch.float64, device=device) for k, s in shapes.items()}

    def __getitem__(self, name):
        return self.blocks[name]

    def put(self, **named):
        """Copy device tensors into the blocks of the same names (device to device); returns the blocks in order."""
        out = []
        for k, t in named.items():
            b = self.blocks[k]
            if t.data_ptr() != b.data_ptr():
                b.copy_(t)
            out.append(b)
        return out


class DevOps(object):
    def __init__(self, eris):
        import torch
        self.torch = torch
        self.e = eris
        self.dev = eris.device
        self.pinned = PinnedPool()

    # -- memory -----------------------------------------------------------------
    def to_dev(self, x):
        torch = self.torch
        if isinstance(x, torch.Tensor):
            return x
        return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(self.dev)

    def empty(self, *shape):
        return self.torch.empty(shape, dtype=self.torch.float64, device=self.dev)

    def to_host(self, t):
        """device -> fresh numpy array in a pinned block of `self.pinned`."""
        h = self.pinned.take(t.shape, t.dtype)
        h.copy_(t, non_blocking=True)
        self.torch.cuda.current_stream(self.dev).synchronize()
        return self.pinned.hand_out(h)

    def scalar(self, t):
        """Device scalar -> Python float (one synchronising D2H read)."""
        return float(t.cpu().reshape(-1)[0])

    # -- dispatch with workspace growth ---------------------------------------------
    def _launch(self, fn, *args):
        """fn(ctx, *args, stream) -> rc; a call that needs more workspace than the context has (rc -2) is repeated
        with the workspace grown to what the library asks for."""
        e = self.e
        if e._ws is None:
            e.grow_workspace(1 << 20)
        rc = fn(e._h, *args, e.stream())
        if rc == -2:
            e.grow_workspace(max(int(lib.ecw_op_workspace_needed(e._h)), 256) + 4096)
            rc = fn(e._h, *args, e.stream())
        return rc

    def _call(self, fn, *args):
        self.e.check(self._launch(fn, *args), getattr(fn, "__name__", "ecw_op"))

    # -- ops ---------------------------------------------------------------------------
    def contract(self, spec, A, B, alpha=1.0, out=None, beta=0.0):
        """out[sc] = alpha * einsum(spec, A, B) + beta * out.  spec like 'jb,jabi->ai'."""
        lhs, sc = spec.split("->")
        sa, sb = lhs.split(",")
        if out is None:
            dims = {}
            for s, t in ((sa, A), (sb, B)):
                for ch, n in zip(s, t.shape):
                    dims[ch] = n
            out = self.empty(*[dims[ch] for ch in sc])
            beta = 0.0
        da, db, dc = _desc(A), _desc(B), _desc(out)
        args = (_scalar(alpha), _ref(da), sa.encode(), _ref(db), sb.encode(), _scalar(beta), _ref(dc), sc.encode())
        e = self.e
        if 2.0 * A.numel() * B.numel() >= e.int8_min_flops >= 0.0:
            # a contraction this large may have taken the INT8 route (2MNK <= 2|A||B|): accuracy guard (eris.py)
            e.guarded(lambda: self._launch(lib.ecw_op_contract, *args), "ecw_op_contract",
                      repeat=_scalar(beta) == 0.0)
        else:
            self._call(lib.ecw_op_contract, *args)
        return out

    def axpby(self, alpha, A, sa, beta, C, sc):
        da, dc = _desc(A), _desc(C)
        self._call(lib.ecw_op_axpby, _scalar(alpha), _ref(da), sa.encode(), _scalar(beta), _ref(dc), sc.encode())
        return C

    def copy(self, A, spec=None, alpha=1.0):
        """Fresh contiguous tensor = alpha * A (optionally permuted: spec 'ai->ia')."""
        lab = "pqrstu"[: A.dim()]
        sa, sc = (spec.split("->") if spec else (lab, lab))
        dims = dict(zip(sa, A.shape))
        out = self.empty(*[dims[ch] for ch in sc])
        return self.axpby(alpha, A, sa, 0.0, out, sc)

    def add(self, C, A, alpha=1.0, spec=None):
        """C += alpha * A (optionally permuted)."""
        lab = "pqrstu"[: A.dim()]
        sa, sc = (spec.split("->") if spec else (lab, lab))
        return self.axpby(alpha, A, sa, 1.0, C, sc)

    def mul(self, alpha, A, B, beta, C):
        da, db, dc = _desc(A), _desc(B), _desc(C)
        self._call(lib.ecw_op_mul, _scalar(alpha), _ref(da), _ref(db), _scalar(beta), _ref(dc))
        return C

    def fill(self, C, value):
        return self.mul(value, None, None, 0.0, C)

    def scale_add(self, C, A, alpha):
        """C += alpha * A (same shape, any strides)."""
        return self.mul(alpha, A, None, 1.0, C)

    def unpack(self, A2, flags, C4, alpha=1.0, beta=0.0):
        da, dc = _desc(A2), _desc(C4)
        self._call(lib.ecw_op_unpack, _scalar(alpha), _ref(da), int(flags), _scalar(beta), _ref(dc))
        return C4

    def diag_shift(self, C, alpha, offset):
        dc, df = _desc(C), _desc(self.e.fock_dev)
        self._call(lib.ecw_op_diag_shift, _ref(dc), _scalar(alpha), _ref(df), int(offset))
        return C

    def denom(self, resid, amp, flags=0, alpha=0.0, shift=0.0, out=None):
        if out is None:
            out = self.empty(*resid.shape)
        dr, da, df, do = _desc(resid), _desc(amp), _desc(self.e.fock_dev), _desc(out)
        self._call(lib.ecw_op_denom, _ref(dr), _ref(da), _ref(df), int(self.e.nocc), int(flags), _scalar(alpha),
                   _scalar(shift), _ref(do))
        return out

    def dot_into(self, out, A, B, alpha=1.0, beta=1.0):
        """out[0] = alpha * <A, B> + beta * out[0] on the device, without synchronising (out: one-element tensor)."""
        da, db = _desc(A), _desc(B)
        self._call(lib.ecw_op_dot, _scalar(alpha), _ref(da), _ref(db), _scalar(beta), ctypes.c_void_p(out.data_ptr()))
        return out

    def dot(self, A, B, alpha=1.0):
        """alpha * <A, B> as a Python float."""
        out = self.torch.zeros(1, dtype=self.torch.float64, device=self.dev)
        return self.scalar(self.dot_into(out, A, B, alpha, 0.0))

    def trace(self, M):
        """sum_i M[i,i] through the dot kernel (diagonal view x ones)."""
        n = M.shape[0]
        diag = self.torch.as_strided(M, (n,), (M.stride(0) + M.stride(1),))
        ones = self.fill(self.empty(n), 1.0)
        return self.dot(diag, ones)
