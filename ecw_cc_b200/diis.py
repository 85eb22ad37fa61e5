"""Pulay DIIS for the solver loops, with the call surface of `pyscf.lib.diis.DIIS` as the reference uses it
(Solver_GS.py:666-674, 683-686, 709-718: `space`, `min_space`, `update(x)`; error vector = x_k - previous returned x).

Two stores behind one algorithm:
  * `DIIS(ops)`  — device resident: the vector is a list of device tensors (the amplitude sets [ls, ts, ld, td]), the
    history (`space` x 2 vectors + xprev) lives in HBM, differences / Gram row / extrapolation run through the C ABI's
    primitive kernels (`ecw_op_axpby`, `ecw_op_dot`), and only the `nd` new Gram entries come to the host, where the
    (space+1)^2 bordered system is solved;
  * `DIIS()`     — host numpy, for the n x n rdm1 ('rdm1' mode), which is on the host anyway for `exp_pot.Exp`.

The steps follow PySCF's published algorithm (ring of `space` slots; first vector only becomes `xprev`; below
`min_space` stored vectors the input is returned unchanged and `xprev` is kept; eigenvalues |w| < 1e-14 of the bordered
Gram matrix are projected out).  PySCF itself is outside the reference tree: DIIS-accelerated runs are pinned to the
restatement in oracle/pyscf_stub and to the fixed point of the plain iteration, not to PySCF ("parity unpinned").
HBM need on the device: (2*space + 1) vectors — 2*(ov + o^2v^2) doubles each; choose `maxdiis` accordingly.
"""
import numpy as np


def solve_coefficients(h):
    g = np.zeros(h.shape[0])
    g[0] = 1.0
    w, v = np.linalg.eigh(h)
    if np.any(abs(w) < 1e-14):
        idx = abs(w) > 1e-14
        return np.dot(v[:, idx] * (1.0 / w[idx]), np.dot(v[:, idx].T, g))
    return np.linalg.solve(h, g)


class _HostStore(object):
    def setup(self, x, space):
        x = np.asarray(x, dtype=np.float64)
        self.shape = x.shape
        self.x = np.empty((space, x.size))
        self.e = np.empty((space, x.size))
        self.xprev = np.empty(x.size)

    def put_prev(self, x):
        self.xprev[:] = np.ravel(x)

    def put(self, slot, x):
        self.x[slot] = np.ravel(x)
        self.e[slot] = self.x[slot] - self.xprev

    def gram_row(self, slot, nd):
        return self.e[:nd] @ self.e[slot]

    def combine(self, c):
        self.xprev[:] = c @ self.x[:len(c)]
        return self.xprev.reshape(self.shape).copy()

    def passthrough(self, x):
        return x


class _DeviceStore(object):
    def __init__(self, ops):
        self.ops = ops

    def setup(self, parts, space):
        torch = self.ops.torch
        self.shapes = [tuple(p.shape) for p in parts]
        self.sizes = [p.numel() for p in parts]
        n = sum(self.sizes)
        try:
            self.x = torch.empty((space, n), dtype=torch.float64, device=self.ops.dev)
            self.e = torch.empty((space, n), dtype=torch.float64, device=self.ops.dev)
            self.xprev = torch.empty(n, dtype=torch.float64, device=self.ops.dev)
        except RuntimeError as err:                              # out of HBM: say what it takes
            raise MemoryError("DIIS history needs %.1f GB of HBM (space=%d); lower maxdiis: %s"
                              % ((2 * space + 1) * n * 8 / 1e9, space, err))
        self.gram = torch.zeros(space, dtype=torch.float64, device=self.ops.dev)

    def _segments(self, flat):
        off = 0
        for n in self.sizes:
            yield flat[off:off + n]
            off += n

    def put_prev(self, parts):
        for dst, p in zip(self._segments(self.xprev), parts):
            self.ops.axpby(1.0, p.reshape(-1), "p", 0.0, dst, "p")

    def put(self, slot, parts):
        segs = zip(self._segments(self.x[slot]), self._segments(self.e[slot]), self._segments(self.xprev), parts)
        for xs, es, prev, p in segs:
            flat = p.reshape(-1)
            self.ops.axpby(1.0, flat, "p", 0.0, xs, "p")
            self.ops.axpby(1.0, flat, "p", 0.0, es, "p")
            self.ops.axpby(-1.0, prev, "p", 1.0, es, "p")

    def gram_row(self, slot, nd):
        ops = self.ops
        ops.fill(self.gram, 0.0)
        for i in range(nd):
            for a, b in zip(self._segments(self.e[slot]), self._segments(self.e[i])):
                ops.dot_into(self.gram[i:i + 1], a, b)
        return self.gram[:nd].cpu().numpy()                      # nd doubles: the only D2H of an update

    def combine(self, c):
        ops = self.ops
        for k, dst in enumerate(self._segments(self.xprev)):
            for i, ci in enumerate(c):
                src = list(self._segments(self.x[i]))[k]
                ops.axpby(float(ci), src, "p", 0.0 if i == 0 else 1.0, dst, "p")
        return [seg.reshape(s).clone() for seg, s in zip(self._segments(self.xprev), self.shapes)]

    def passthrough(self, parts):
        return list(parts)


class DIIS(object):
    def __init__(self, ops=None):
        self.space = 6
        self.min_space = 1
        self._store = _DeviceStore(ops) if ops is not None else _HostStore()
        self._head = 0
        self._book = []
        self._H = None
        self._have_prev = False

    def get_num_vec(self):
        return len(self._book)

    def update(self, x):
        """x: numpy array (host store) or list of device tensors (device store); returns the same kind."""
        st = self._store
        if self._H is None:
            st.setup(x, self.space)
            self._H = np.zeros((self.space + 1, self.space + 1))
            self._H[0, 1:] = self._H[1:, 0] = 1.0
        while len(self._book) >= self.space:
            self._book.pop(0)
        if not self._have_prev:
            st.put_prev(x)
            self._have_prev = True
        else:
            if self._head >= self.space:
                self._head = 0
            self._book.append(self._head)
            st.put(self._head, x)
            self._head += 1
        nd = self.get_num_vec()
        if nd < self.min_space:
            return st.passthrough(x)
        row = st.gram_row(self._head - 1, nd)
        self._H[self._head, 1:nd + 1] = row
        self._H[1:nd + 1, self._head] = row
        c = solve_coefficients(self._H[:nd + 1, :nd + 1])
        return st.combine(c[1:])
