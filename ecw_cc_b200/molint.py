"""Integral source without PySCF (SURVEY §8f-1): Gaussian one- and two-electron integrals over s, p and (spherical) d
shells (McMurchie-Davidson), restricted Hartree-Fock, and the spin-orbital antisymmetrised MO integrals of the reference's
`Eris.geris` container (Eris.py:24-154: `<pq||rs> = <pq|rs> - <pq|sr>`, blocks `oooo ... vvvv`, `fock = diag(mo_energy)`),
built the way `Main.ECW.__init__` does (Main.py:151-217: RHF -> GHF spin orbitals in `[a, b, a, b, ...]` order).

Host-side numpy on purpose: this is the producer of the path's inputs (a 13-function basis for config 1, H2O/6-31G),
not the path.  Basis sets embedded for H, C, N, O: the 6-31G family — 6-31G, 6-31G*, 6-31G**, 6-31+G*, 6-31++G** ...
(Pople's standard polarisation / diffuse exponents; five spherical d functions per shell, PySCF's default) — and
cc-pVDZ for H, C, O.  Anchor: E_HF(H2O/6-31G) = -75.9839 (ECW_CC/__init__.py:39).
"""
import re
from fractions import Fraction

import numpy as np
from scipy.special import hyp1f1

ANGSTROM = 1.0 / 0.52917721092                 # bohr per Angstrom (the value PySCF uses)
FOBS_ZERO = 1e-12                              # 'Fobs': |F_calc| <= FOBS_ZERO max |F_calc| counts as zero

# 6-31G: per element a list of (kind, exponents, s coefficients, p coefficients)
BASIS_631G = {
    1: [("S", [18.7311370, 2.8253937, 0.6401217], [0.03349460, 0.23472695, 0.81375733], None),
        ("S", [0.1612778], [1.0], None)],
    6: [("S", [3047.5249, 457.36952, 103.94869, 29.210155, 9.2866630, 3.1639270],
         [0.0018347, 0.0140373, 0.0688426, 0.2321844, 0.4679413, 0.3623120], None),
        ("SP", [7.8682724, 1.8812885, 0.5442493], [-0.1193324, -0.1608542, 1.1434564], [0.0689991, 0.3164240, 0.7443083]),
        ("SP", [0.1687144], [1.0], [1.0])],
    7: [("S", [4173.5110, 627.45790, 142.90210, 40.234330, 12.820210, 4.3904370],
         [0.0018348, 0.0139950, 0.0685870, 0.2322410, 0.4690700, 0.3604550], None),
        ("SP", [11.626358, 2.7162800, 0.7722180], [-0.1149610, -0.1691180, 1.1458520], [0.0675800, 0.3239070, 0.7408950]),
        ("SP", [0.2120313], [1.0], [1.0])],
    8: [("S", [5484.6717, 825.23495, 188.04696, 52.964500, 16.897570, 5.7996353],
         [0.0018311, 0.0139501, 0.0684451, 0.2327143, 0.4701930, 0.3585209], None),
        ("SP", [15.539616, 3.5999336, 1.0137618], [-0.1107775, -0.1480263, 1.1307670], [0.0708743, 0.3397528, 0.7271586]),
        ("SP", [0.2700058], [1.0], [1.0])],
}


# polarisation / diffuse functions of the 6-31G family: d exponent ('*'), diffuse sp exponent ('+') of the heavy atoms,
# p exponent ('**') and diffuse s exponent ('++') of hydrogen
POPLE_D = {6: 0.8, 7: 0.8, 8: 0.8}
POPLE_DIFFUSE_SP = {6: 0.0438, 7: 0.0639, 8: 0.0845}
POPLE_H_P, POPLE_H_DIFFUSE_S = 1.1, 0.036

# cc-pVDZ (Dunning 1989): general contractions written out per contracted function
BASIS_CCPVDZ = {
    1: [("S", [13.01, 1.962, 0.4446], [0.019685, 0.137977, 0.478148], None),
        ("S", [0.122], [1.0], None),
        ("P", [0.727], None, [1.0])],
    6: [("S", [6665.0, 1000.0, 228.0, 64.71, 21.06, 7.495, 2.797, 0.5215],
         [0.000692, 0.005329, 0.027077, 0.101718, 0.27474, 0.448564, 0.285074, 0.015204], None),
        ("S", [6665.0, 1000.0, 228.0, 64.71, 21.06, 7.495, 2.797, 0.5215],
         [-0.000146, -0.001154, -0.005725, -0.023312, -0.063955, -0.149981, -0.127262, 0.544529], None),
        ("S", [0.1596], [1.0], None),
        ("P", [9.439, 2.002, 0.5456], None, [0.038109, 0.20948, 0.508557]),
        ("P", [0.1517], None, [1.0]),
        ("D", [0.55], None, [1.0])],
    8: [("S", [11720.0, 1759.0, 400.8, 113.7, 37.03, 13.27, 5.025, 1.013],
         [0.00071, 0.00547, 0.027837, 0.1048, 0.283062, 0.448719, 0.270952, 0.015458], None),
        ("S", [11720.0, 1759.0, 400.8, 113.7, 37.03, 13.27, 5.025, 1.013],
         [-0.00016, -0.001263, -0.006267, -0.025716, -0.070924, -0.165411, -0.116955, 0.557368], None),
        ("S", [0.3023], [1.0], None),
        ("P", [17.7, 3.854, 1.046], None, [0.043018, 0.228913, 0.508728]),
        ("P", [0.2753], None, [1.0]),
        ("D", [1.185], None, [1.0])],
}

# real solid harmonics of a d shell over Cartesian monomials, in PySCF's order (xy, yz, z2, xz, x2-y2); factors are
# relative to the norm of an xy-type Gaussian, N = (2a/pi)^(3/4) * 4a
_S3 = 1.0 / (2.0 * np.sqrt(3.0))
D_SPHERICAL = [[((1, 1, 0), 1.0)], [((0, 1, 1), 1.0)], [((0, 0, 2), 2 * _S3), ((2, 0, 0), -_S3), ((0, 2, 0), -_S3)],
               [((1, 0, 1), 1.0)], [((2, 0, 0), 0.5), ((0, 2, 0), -0.5)]]


def basis_shells(name, z):
    """Shell list [(kind, exponents, s coefficients, p-or-d coefficients)] of element z in the named basis."""
    key = name.lower().replace("-", "").replace("(d)", "*").replace("(d,p)", "**")
    if key == "ccpvdz":
        if z not in BASIS_CCPVDZ:
            raise NotImplementedError("cc-pVDZ is embedded for H, C, O")
        return BASIS_CCPVDZ[z]
    import re
    m = re.fullmatch(r"631(\+{0,2})g(\*{0,2})", key)
    if m is None:
        raise NotImplementedError("embedded basis sets: 6-31G family (6-31G, 6-31G*, 6-31+G*, 6-31++G**, ...) and cc-pVDZ")
    plus, star = len(m.group(1)), len(m.group(2))
    shells = list(BASIS_631G[z])
    if z == 1:
        if plus == 2:
            shells.append(("S", [POPLE_H_DIFFUSE_S], [1.0], None))
        if star == 2:
            shells.append(("P", [POPLE_H_P], None, [1.0]))
    else:
        if plus >= 1:
            shells.append(("SP", [POPLE_DIFFUSE_SP[z]], [1.0], [1.0]))
        if star >= 1:
            shells.append(("D", [POPLE_D[z]], None, [1.0]))
    return shells


class Molecule(object):
    """atoms: [(Z or element symbol, (x, y, z)), ...] in Angstrom (Main.py:104-109 style); basis: '6-31g', '6-31+g*',
    '6-31++g**', 'cc-pvdz', ... (see `basis_shells`)."""
    SYMBOLS = {"H": 1, "C": 6, "N": 7, "O": 8}

    def __init__(self, atoms, basis="6-31g", charge=0):
        for a in atoms:
            if (a[0].capitalize() if isinstance(a[0], str) else int(a[0])) not in (set(self.SYMBOLS) | set(self.SYMBOLS.values())):
                raise NotImplementedError("element %r: basis sets are embedded for H, C, N, O" % (a[0],))
        self.Z = np.array([self.SYMBOLS[a[0].capitalize()] if isinstance(a[0], str) else a[0] for a in atoms], dtype=np.float64)
        self.R = np.array([a[1] for a in atoms], dtype=np.float64) * ANGSTROM
        self.nelec = int(self.Z.sum()) - charge
        if self.nelec % 2:
            raise NotImplementedError("closed shells only (RHF)")
        # primitive Cartesian Gaussians: centre, exponent, (lx,ly,lz), coefficient incl. normalisation, AO index
        cen, ex, lmn, coef, ao, ao_atom = [], [], [], [], [], []
        nao = 0
        for iat, (z, r) in enumerate(zip(self.Z, self.R)):
            for kind, exps, cs, cp in basis_shells(basis, int(z)):
                parts = {"S": ((0, cs),), "P": ((1, cp),), "SP": ((0, cs), (1, cp)), "D": ((2, cp),)}[kind]
                for ang, cc in parts:
                    if ang == 2:                               # five spherical d functions
                        comps = D_SPHERICAL
                    else:
                        comps = [[((0, 0, 0), 1.0)]] if ang == 0 else [[(l3, 1.0)] for l3 in ((1, 0, 0), (0, 1, 0), (0, 0, 1))]
                    for comp in comps:
                        for a, c in zip(exps, cc):
                            norm = (2 * a / np.pi) ** 0.75 * (2 * np.sqrt(a)) ** ang      # s / p / xy-type d norm
                            for l3, f in comp:
                                cen.append(r); ex.append(a); lmn.append(l3); coef.append(c * norm * f); ao.append(nao)
                        ao_atom.append(iat)
                        nao += 1
        self.cen, self.ex = np.array(cen), np.array(ex)
        self.lmn, self.coef, self.ao = np.array(lmn), np.array(coef), np.array(ao)
        self.ao_atom = np.array(ao_atom, dtype=np.int64)            # atom of every AO
        self.nao = nao
        self.lmax = int(self.lmn.sum(1).max())
        # Tables of general contractions (cc-pVDZ) list contracted functions that are not unit normalised: rescale
        # those.  Segmented Pople functions are normalised to ~1e-7 as published and are left exactly as tabulated.
        sii = self._self_overlaps()
        scale = np.where(np.abs(sii - 1.0) > 1e-4, 1.0 / np.sqrt(sii), 1.0)
        self.coef = self.coef * scale[self.ao]
        d = self.R[:, None, :] - self.R[None, :, :]
        rr = np.sqrt((d ** 2).sum(-1))
        iu = np.triu_indices(len(self.Z), 1)
        self.e_nuc = float((self.Z[:, None] * self.Z[None, :])[iu].dot(1.0 / rr[iu]))
        self._origin = np.zeros(3)
        self._ints = None


    def _self_overlaps(self):
        """<mu|mu> of every AO from its own primitives (all on one centre: products of 1-D Gaussian moments)."""
        def dfact(n):                                             # (n-1)!! for even n >= 0
            return float(np.prod(np.arange(n - 1, 0, -2))) if n > 0 else 1.0
        out = np.zeros(self.nao)
        for mu in range(self.nao):
            k = np.where(self.ao == mu)[0]
            for i in k:
                for j in k:
                    n3 = self.lmn[i] + self.lmn[j]
                    if (n3 % 2).any():
                        continue
                    pq = self.ex[i] + self.ex[j]
                    val = (np.pi / pq) ** 1.5
                    for n in n3:
                        val *= dfact(n) / (2 * pq) ** (n // 2)
                    out[mu] += self.coef[i] * self.coef[j] * val
        return out

    # -- the slice of PySCF's `gto.Mole` surface that exp_pot.Exp / utilities touch (exp_pot.py:90-108) ---------------
    def atom_charges(self):
        return self.Z.copy()

    def atom_coords(self):
        return self.R.copy()                                      # Bohr, like PySCF

    def with_common_orig(self, origin):
        mol = self

        class _Origin(object):
            def __enter__(self_inner):
                self_inner.old = mol._origin
                mol._origin = np.asarray(origin, dtype=np.float64)
                return mol

            def __exit__(self_inner, *exc):
                mol._origin = self_inner.old
                return False
        return _Origin()

    def intor_symmetric(self, name, comp=None):
        if self._ints is None:
            self._ints = integrals(self)
        if name == "int1e_kin":
            return self._ints[1]
        if name == "int1e_nuc":
            return self._ints[2]
        if name == "int1e_ovlp":
            return self._ints[0]
        if name == "int1e_r":
            return dipole_integrals(self, self._origin)
        raise NotImplementedError("intor %r" % (name,))

    intor = intor_symmetric


def _boys(nmax, x):
    """F_n(x), n = 0..nmax, for an array x."""
    return np.stack([hyp1f1(n + 0.5, n + 1.5, -x) / (2 * n + 1) for n in range(nmax + 1)])


def _hermite_E(imax, jmax, p, XPA, XPB, mu, XAB):
    """1-D Hermite expansion coefficients E[i][j][t] (arrays over pairs), i <= imax, j <= jmax."""
    E = [[None] * (jmax + 1) for _ in range(imax + 1)]
    tmax = imax + jmax
    z = np.zeros_like(p)
    E[0][0] = [np.exp(-mu * XAB ** 2)] + [z] * (tmax + 1)
    for i in range(imax + 1):
        for j in range(jmax + 1):
            if i == 0 and j == 0:
                continue
            if i > 0:
                src, X = E[i - 1][j], XPA
            else:
                src, X = E[i][j - 1], XPB
            E[i][j] = [(src[t - 1] / (2 * p) if t > 0 else 0) + X * src[t] + (t + 1) * src[t + 1]
                       for t in range(tmax + 1)] + [z]
    return E


def _hermite_R(L, alpha, D):
    """Hermite Coulomb integrals R[t][u][v] (t+u+v <= L) for exponent alpha and distance vectors D[..., 3]."""
    r2 = (D ** 2).sum(-1)
    F = _boys(L, alpha * r2)
    Rn = {(0, 0, 0, n): (-2 * alpha) ** n * F[n] for n in range(L + 1)}
    X, Y, Z = D[..., 0], D[..., 1], D[..., 2]

    def get(t, u, v, n):
        key = (t, u, v, n)
        if key in Rn:
            return Rn[key]
        if t > 0:
            val = X * get(t - 1, u, v, n + 1) + ((t - 1) * get(t - 2, u, v, n + 1) if t > 1 else 0)
        elif u > 0:
            val = Y * get(t, u - 1, v, n + 1) + ((u - 1) * get(t, u - 2, v, n + 1) if u > 1 else 0)
        else:
            val = Z * get(t, u, v - 1, n + 1) + ((v - 1) * get(t, u, v - 2, n + 1) if v > 1 else 0)
        Rn[key] = val
        return val
    return {(t, u, v): get(t, u, v, 0) for t in range(L + 1) for u in range(L + 1 - t) for v in range(L + 1 - t - u)}


def _pairs(mol):
    """Unique primitive pairs I >= J and the matrix that adds a pair quantity into the AO pairs (mu nu) and (nu mu)."""
    I, J = np.tril_indices(len(mol.ex))
    nao = mol.nao
    M = np.zeros((len(I), nao * nao))
    k = np.arange(len(I))
    np.add.at(M, (k, mol.ao[I] * nao + mol.ao[J]), 1.0)
    off = I != J
    np.add.at(M, (k[off], mol.ao[J[off]] * nao + mol.ao[I[off]]), 1.0)
    return I, J, M


def integrals(mol):
    """Overlap, kinetic, nuclear-attraction [nao, nao] and electron-repulsion (mu nu|la si) [nao]*4, AO basis.
    McMurchie-Davidson over the unique primitive pairs (I >= J) and the lower triangle of pair-pairs."""
    I, J, M = _pairs(mol)
    a, b = mol.ex[I], mol.ex[J]
    p = a + b
    mu = a * b / p
    A, B = mol.cen[I], mol.cen[J]
    P = (a[:, None] * A + b[:, None] * B) / p[:, None]
    la, lb = mol.lmn[I], mol.lmn[J]
    cc = mol.coef[I] * mol.coef[J]
    lm = mol.lmax
    nt = 2 * lm + 1                                               # Hermite orders 0..2*lmax per direction
    # 1-D coefficients with j up to l_b + 2 (kinetic energy)
    Ed = [_hermite_E(lm, lm + 2, p, P[:, d] - A[:, d], P[:, d] - B[:, d], mu, A[:, d] - B[:, d]) for d in range(3)]

    def pick(d, dj, t):
        """E^{la_d, lb_d + dj}_t per pair (lb_d + dj may be -1 or -2: zero)."""
        out = np.zeros(len(p))
        for i in range(lm + 1):
            for j in range(0, lm + 3):
                if t > i + j:
                    continue
                m = (la[:, d] == i) & (lb[:, d] + dj == j)
                if m.any():
                    out[m] = Ed[d][i][j][t][m]
        return out
    S1 = [pick(d, 0, 0) * np.sqrt(np.pi / p) for d in range(3)]
    T1 = []
    for d in range(3):
        j = lb[:, d]
        T1.append((-2 * b ** 2 * pick(d, 2, 0) + b * (2 * j + 1) * pick(d, 0, 0) - 0.5 * j * (j - 1) * pick(d, -2, 0))
                  * np.sqrt(np.pi / p))
    Sp = S1[0] * S1[1] * S1[2]
    Tp = T1[0] * S1[1] * S1[2] + S1[0] * T1[1] * S1[2] + S1[0] * S1[1] * T1[2]
    # Hermite tensor of every pair: Eab[pair, t, u, v], t + u + v <= 2*lmax
    Eab = np.zeros((len(p), nt, nt, nt))
    e1 = [[pick(d, 0, t) for t in range(nt)] for d in range(3)]
    for t in range(nt):
        for u in range(nt):
            for v in range(nt):
                if t + u + v <= 2 * lm:
                    Eab[:, t, u, v] = e1[0][t] * e1[1][u] * e1[2][v]
    Vp = np.zeros(len(p))
    for Zc, C in zip(mol.Z, mol.R):
        R = _hermite_R(2 * lm, p, P - C)
        acc = np.zeros(len(p))
        for (t, u, v), r in R.items():
            acc += Eab[:, t, u, v] * r
        Vp -= Zc * 2 * np.pi / p * acc
    nao = mol.nao
    S, T, V = ((M.T @ (cc * x)).reshape(nao, nao) for x in (Sp, Tp, Vp))
    # electron repulsion: (ab|cd) = 2 pi^2.5 / (p q sqrt(p+q)) sum E_ab(tuv) (-1)^(t'+u'+v') E_cd(t'u'v') R(t+t',u+u',v+v')
    sign = np.array([[[(-1.0) ** (t + u + v) for v in range(nt)] for u in range(nt)] for t in range(nt)])
    Ecd = Eab * sign[None]
    idx = [(t, u, v) for t in range(nt) for u in range(nt) for v in range(nt) if t + u + v <= 2 * lm]
    W = np.zeros((len(p), len(p)))                                # pair-pair integrals, lower block triangle
    chunk = 64
    for s0 in range(0, len(p), chunk):
        s1 = min(len(p), s0 + chunk)
        sl, kt = slice(s0, s1), slice(0, s1)
        pq = p[sl, None] + p[None, kt]
        alpha = p[sl, None] * p[None, kt] / pq
        R = _hermite_R(4 * lm, alpha, P[sl, None, :] - P[None, kt, :])
        acc = np.zeros_like(alpha)
        for (t, u, v) in idx:
            ea = Eab[sl, t, u, v]
            if not ea.any():
                continue
            for (t2, u2, v2) in idx:
                ec = Ecd[kt, t2, u2, v2]
                if not ec.any():
                    continue
                acc += ea[:, None] * ec[None, :] * R[(t + t2, u + u2, v + v2)]
        W[sl, kt] = 2 * np.pi ** 2.5 / (p[sl, None] * p[None, kt] * np.sqrt(pq)) * acc * cc[sl, None] * cc[None, kt]
    W = np.tril(W) + np.tril(W, -1).T
    eri = M.T @ W @ M
    return S, T, V, eri.reshape(nao, nao, nao, nao)


def dipole_integrals(mol, origin=(0., 0., 0.)):
    """<mu| r - origin |nu>, [3, nao, nao] (the 'int1e_r' integrals the reference takes from PySCF with
    `mol.with_common_orig`, exp_pot.py:90-98): 1-D first moments (E_1 + (P - C) E_0) sqrt(pi/p) times the overlaps of
    the other two directions."""
    I, J, M = _pairs(mol)
    a, b = mol.ex[I], mol.ex[J]
    p = a + b
    mu = a * b / p
    A, B = mol.cen[I], mol.cen[J]
    P = (a[:, None] * A + b[:, None] * B) / p[:, None]
    la, lb = mol.lmn[I], mol.lmn[J]
    cc = mol.coef[I] * mol.coef[J]
    origin = np.asarray(origin, dtype=np.float64)
    S1, M1 = [], []
    for d in range(3):
        lm = mol.lmax
        E = _hermite_E(lm, lm, p, P[:, d] - A[:, d], P[:, d] - B[:, d], mu, A[:, d] - B[:, d])
        e0, e1 = np.zeros(len(p)), np.zeros(len(p))
        for i in range(lm + 1):
            for j in range(lm + 1):
                m = (la[:, d] == i) & (lb[:, d] == j)
                e0[m], e1[m] = E[i][j][0][m], E[i][j][1][m]
        S1.append(e0 * np.sqrt(np.pi / p))
        M1.append((e1 + (P[:, d] - origin[d]) * e0) * np.sqrt(np.pi / p))
    nao = mol.nao
    out = []
    for d in range(3):
        f = [M1[k] if k == d else S1[k] for k in range(3)]
        out.append((M.T @ (cc * f[0] * f[1] * f[2])).reshape(nao, nao))
    return np.stack(out)


def ft_aopair(mol, G):
    """Fourier-transformed AO pairs A_mu,nu(G) = int phi_mu phi_nu exp(+i G.r) d^3r (crystallographic sign), complex
    [nG, nao, nao], for scattering vectors G [nG, 3] in bohr^-1.  Symmetric in mu nu; A(0) is the overlap matrix.
    One primitive pair (exponents a, b, p = a + b, centre P) contributes, exactly,
        (pi/p)^(3/2) exp(-|G|^2/4p) exp(i G.P) prod_d sum_t E_t^(d) (i G_d)^t
    with the 1-D Hermite coefficients E_t of `_hermite_E` (the Fourier transform of the Hermite Gaussian of order t is
    (i G_d)^t times that of order 0).  This is the host path of the structure-factor target of `exp_pot.Exp` and the
    reference the device kernel (`ecw_ft_aopair`) is tested against."""
    G = np.atleast_2d(np.asarray(G, dtype=np.float64))
    if G.ndim != 2 or G.shape[1] != 3:
        raise ValueError("G must be an [nG, 3] array of scattering vectors")
    I, J, M = _pairs(mol)
    a, b = mol.ex[I], mol.ex[J]
    p = a + b
    mu = a * b / p
    A, B = mol.cen[I], mol.cen[J]
    P = (a[:, None] * A + b[:, None] * B) / p[:, None]
    la, lb = mol.lmn[I], mol.lmn[J]
    lm = mol.lmax
    re = np.ones((len(G), len(p)))
    im = np.zeros((len(G), len(p)))
    for d in range(3):
        E = _hermite_E(lm, lm, p, P[:, d] - A[:, d], P[:, d] - B[:, d], mu, A[:, d] - B[:, d])
        et = np.zeros((2 * lm + 1, len(p)))                      # E_t^{la_d, lb_d} per pair
        for i in range(lm + 1):
            for j in range(lm + 1):
                m = (la[:, d] == i) & (lb[:, d] == j)
                for t in range(i + j + 1):
                    et[t, m] = E[i][j][t][m]
        g = G[:, d:d + 1]
        pr, pi = np.zeros_like(re), np.zeros_like(im)            # sum_t E_t (i g)^t
        for t in range(2 * lm + 1):
            c = et[t][None, :] * g ** t
            if t % 4 == 0:
                pr += c
            elif t % 4 == 1:
                pi += c
            elif t % 4 == 2:
                pr -= c
            else:
                pi -= c
        re, im = re * pr - im * pi, re * pi + im * pr
    amp = mol.coef[I] * mol.coef[J] * (np.pi / p) ** 1.5 * np.exp(-(G ** 2).sum(1)[:, None] / (4 * p[None, :]))
    ph = G @ P.T
    c, s = np.cos(ph), np.sin(ph)
    vr = amp * (re * c - im * s)
    vi = amp * (re * s + im * c)
    nao = mol.nao
    return ((vr @ M) + 1j * (vi @ M)).reshape(len(G), nao, nao)


_SYMOP_TERM = re.compile(r"([+-])((?:\d+(?:\.\d*)?|\.\d+)(?:/\d+)?)?\*?([xyz])?")


def parse_symop(op):
    """One symmetry operation x' = R x + t in fractional coordinates, from a CIF `_space_group_symop_operation_xyz`
    string ('x,y,z', '-x,y+1/2,-z+1/2', 'x-y,x,z+1/6', ...) or an (R, t) pair.  R must be an integer matrix with
    det +-1.  Returns (R int [3, 3], t float [3])."""
    if isinstance(op, str):
        parts = op.replace(" ", "").lower().split(",")
        if len(parts) != 3:
            raise ValueError("symmetry operation %r: three comma-separated components expected" % (op,))
        R, t = np.zeros((3, 3)), np.zeros(3)
        for d, s in enumerate(parts):
            s = s if s[:1] in ("+", "-") else "+" + s
            pos = 0
            while pos < len(s):
                m = _SYMOP_TERM.match(s, pos)
                if m is None or (m.group(2) is None and m.group(3) is None):
                    raise ValueError("symmetry operation %r: cannot read %r" % (op, s[pos:]))
                v = float(Fraction(m.group(2))) if m.group(2) else 1.0
                v = -v if m.group(1) == "-" else v
                if m.group(3):
                    R[d, "xyz".index(m.group(3))] += v
                else:
                    t[d] += v
                pos = m.end()
    else:
        try:
            R, t = op
            R, t = np.asarray(R, dtype=np.float64), np.asarray(t, dtype=np.float64)
        except (TypeError, ValueError):
            raise ValueError("symmetry operation %r: a CIF xyz string or an (R, t) pair expected" % (op,))
        if R.shape != (3, 3) or t.shape != (3,) or not np.all(np.isfinite(R)) or not np.all(np.isfinite(t)):
            raise ValueError("symmetry operation: R must be 3 x 3 and t of length 3, finite")
    if np.any(R != np.round(R)):
        raise ValueError("symmetry operation %r: R must be an integer matrix" % (op,))
    R = np.round(R).astype(np.int64)
    if abs(round(np.linalg.det(R))) != 1:
        raise ValueError("symmetry operation %r: det R must be +-1" % (op,))
    return R, t


def symop_string(R, t):
    """The CIF xyz string of (R, t): the inverse of `parse_symop` for the standard strings."""
    out = []
    for d in range(3):
        s = ""
        for e in range(3):
            c = int(R[d][e])
            if c:
                s += ("+" if c > 0 else "-") + ("" if abs(c) == 1 else str(abs(c))) + "xyz"[e]
        f = Fraction(float(t[d])).limit_denominator(48)
        if f:
            s += ("+" if f > 0 else "-") + str(abs(f))
        out.append(s.lstrip("+") or "0")
    return ",".join(out)


def check_group(ops, tol=1e-9):
    """Raise ValueError unless the operations (R, t) are closed under composition modulo lattice translations:
    (R_s R_u, R_s t_u + t_s mod 1) must be in the list for every s, u (t to `tol`)."""
    R = np.array([r for r, _ in ops])
    t = np.array([t for _, t in ops], dtype=np.float64)
    for Rs, ts in zip(R, t):
        for Ru, tu in zip(R, t):
            dt = np.mod(Rs @ tu + ts - t + 0.5, 1.0) - 0.5
            if not np.any(np.all(R == Rs @ Ru, axis=(1, 2)) & np.all(np.abs(dt) <= tol, axis=1)):
                raise ValueError("the symmetry operations are not closed under composition (%s after %s is missing): "
                                 "for a molecule on a special position the crystal lists only coset representatives; "
                                 "pass the full space group as group=" % (symop_string(Rs, ts), symop_string(Ru, tu)))


class Crystal(object):
    """A molecular crystal for the amplitude target 'Fobs' of `exp_pot.Exp`.

    cell: (a, b, c) in Angstrom (orthorhombic) or (a, b, c, alpha, beta, gamma) in Angstrom and degrees.  The lattice
    matrix M has the lattice vectors as columns in the standard orthogonalisation (a along x, b in the xy plane):
        M = [[a, b cos g, c cos b], [0, b sin g, c (cos a - cos b cos g) / sin g], [0, 0, V / (a b sin g)]]
    and the molecule's Cartesian coordinates (`Molecule`, Angstrom) are taken in this frame (`cartesian` converts
    fractional coordinates).  The scattering vector of reflection h is G_h = 2 pi M^-T h.

    symops: operations x' = R x + t in fractional coordinates, CIF xyz strings or (R, t) pairs (`parse_symop`); the
    default is the identity.  The list must hold exactly the operations that generate the DISTINCT copies of the
    molecule in the cell, centring translations included: for a molecule on a special position give only the coset
    representatives.  One molecule in the asymmetric unit (Z' = 1).

    adp: None, or one entry per atom of the molecule: None (no smearing), a scalar U_iso, or a 3 x 3 Cartesian U tensor
    in the frame above (not the crystal-axis U_ij of a CIF), Angstrom^2."""

    def __init__(self, cell, symops=("x,y,z",), adp=None):
        cell = np.asarray(cell, dtype=np.float64)
        if cell.shape not in ((3,), (6,)) or not np.all(np.isfinite(cell)) or np.any(cell[:3] <= 0):
            raise ValueError("cell: (a, b, c) or (a, b, c, alpha, beta, gamma), positive lengths in Angstrom")
        ang = cell[3:] if len(cell) == 6 else np.full(3, 90.0)
        if np.any(ang <= 0) or np.any(ang >= 180):
            raise ValueError("cell angles must lie strictly between 0 and 180 degrees")

        def cos_sin(x):                                             # exact 0 / 1 at 90 degrees
            return (0.0, 1.0) if x == 90.0 else (np.cos(np.deg2rad(x)), np.sin(np.deg2rad(x)))
        (ca, _), (cb, _), (cg, sg) = (cos_sin(x) for x in ang)
        vf = 1.0 - ca * ca - cb * cb - cg * cg + 2.0 * ca * cb * cg
        if vf <= 0:
            raise ValueError("cell angles do not describe a cell of positive volume")
        a, b, c = cell[:3]
        self.cell = cell
        self.M = np.array([[a, b * cg, c * cb], [0.0, b * sg, c * (ca - cb * cg) / sg], [0.0, 0.0, c * np.sqrt(vf) / sg]])
        self.volume = float(a * b * c * np.sqrt(vf))
        self.ops = [parse_symop(op) for op in ([symops] if isinstance(symops, str) else symops)]
        if not self.ops:
            raise ValueError("symops: at least one operation")
        self.adp = None if adp is None else [self._adp_entry(u) for u in adp]

    @staticmethod
    def _adp_entry(u):
        if u is None:
            return np.zeros((3, 3))
        u = np.asarray(u, dtype=np.float64)
        if u.ndim == 0:
            u = float(u) * np.eye(3)
        if u.shape != (3, 3) or not np.all(np.isfinite(u)) or np.abs(u - u.T).max() > 1e-12 * max(1.0, np.abs(u).max()):
            raise ValueError("adp: each entry is None, a scalar U_iso or a symmetric 3 x 3 Cartesian tensor (A^2)")
        if np.linalg.eigvalsh(u).min() < -1e-12 * max(1.0, np.abs(u).max()):
            raise ValueError("adp: U must be positive semi-definite")
        return 0.5 * (u + u.T)

    @property
    def nsym(self):
        return len(self.ops)

    def cartesian(self, frac):
        """Fractional coordinates [..., 3] -> Cartesian Angstrom in the frame of M."""
        return np.asarray(frac, dtype=np.float64) @ self.M.T

    def G(self, hkl):
        """G_h = 2 pi M^-T h in bohr^-1, [..., 3] (M^T is lower triangular: forward substitution, which gives
        2 pi (h/a, k/b, l/c) bit for bit in an orthorhombic cell)."""
        x = 2 * np.pi * np.asarray(hkl, dtype=np.float64)
        M = self.M
        g0 = x[..., 0] / M[0, 0]
        g1 = (x[..., 1] - M[0, 1] * g0) / M[1, 1]
        g2 = (x[..., 2] - M[0, 2] * g0 - M[1, 2] * g1) / M[2, 2]
        return np.stack([g0, g1, g2], axis=-1) / ANGSTROM

    @property
    def volume_bohr3(self):
        return self.volume * ANGSTROM ** 3

    def expand(self, hkl, F, group=None):
        """Unique (or unmerged) structure factors -> the half set of the full sphere, for Fourier maps.

        Every F(h) contributes F(R_u^T h) = exp(-2 pi i h.t_u) F(h) for each operation u and, by Friedel's law,
        F(-R_u^T h) = conj of that.  Each coefficient of the expanded set is the mean of all contributions landing on
        it: equivalents and Friedel mates are averaged, systematically absent reflections cancel to zero (to rounding)
        and a consistent set such as F_calc comes out unchanged.  The operations (this crystal's, or `group`: symmetry
        operations as for `Crystal`) must form a group modulo lattice translations; that is checked, to 1e-9 in t.
        Returns (hkl_half int64 [M, 3], F_half complex [M], F000 float): h > 0, or h = 0 and k > 0, or h = k = 0 and
        l > 0, in lexicographic order; F000 is the real part of the mean at (0, 0, 0) (0 when no input lands there)."""
        hkl = np.asarray(hkl)
        F = np.asarray(F)
        if hkl.ndim != 2 or hkl.shape[1] != 3 or not np.issubdtype(hkl.dtype, np.number) \
                or not np.all(np.isfinite(hkl)) or np.any(hkl != np.round(hkl)):
            raise ValueError("hkl must be an (N_h, 3) array of integer Miller indices")
        if F.shape != (len(hkl),) or not np.issubdtype(F.dtype, np.number) or not np.all(np.isfinite(F)):
            raise ValueError("F must hold N_h finite (real or complex) structure factors, N_h = len(hkl)")
        ops = self.ops if group is None else [parse_symop(op) for op in ([group] if isinstance(group, str) else group)]
        if not ops:
            raise ValueError("group: at least one operation")
        check_group(ops)
        R = np.array([r for r, _ in ops])
        t = np.array([t for _, t in ops])
        h = np.round(hkl).astype(np.int64)
        hs = np.einsum("sdk,hd->hsk", R, h).reshape(-1, 3)          # R_u^T h
        ph = 2 * np.pi * np.mod(h @ t.T, 1.0)
        v = ((np.cos(ph) - 1j * np.sin(ph)) * F.astype(np.complex128)[:, None]).ravel()
        keys, inv = np.unique(np.concatenate([hs, -hs]), axis=0, return_inverse=True)
        inv = inv.ravel()
        s = np.zeros(len(keys), dtype=np.complex128)
        np.add.at(s, inv, np.concatenate([v, np.conj(v)]))
        mean = s / np.bincount(inv, minlength=len(keys))
        zero = np.all(keys == 0, axis=1)
        F000 = float(mean[zero][0].real) if zero.any() else 0.0
        half = (keys[:, 0] > 0) | ((keys[:, 0] == 0) & (keys[:, 1] > 0)) | \
               ((keys[:, 0] == 0) & (keys[:, 1] == 0) & (keys[:, 2] > 0))
        return keys[half], mean[half], F000

    def adp_bohr(self, natom):
        """Cartesian U per atom in bohr^2, [natom, 3, 3] (zeros without ADPs)."""
        if self.adp is None:
            return np.zeros((natom, 3, 3))
        if len(self.adp) != natom:
            raise ValueError("adp: %d entries for a molecule of %d atoms" % (len(self.adp), natom))
        return np.array(self.adp) * ANGSTROM ** 2

    def tables(self, hkl):
        """What the symmetrised planes need per (h, s), [N_h, nsym, ...]: the rotated vectors G_{h_s}, h_s = R_s^T h
        (bohr^-1), and the phases (cos, sin) of 2 pi h.t_s (h.t_s reduced mod 1 first)."""
        h = np.asarray(hkl, dtype=np.float64).reshape(-1, 3)
        R = np.array([r for r, _ in self.ops], dtype=np.float64)
        t = np.array([t for _, t in self.ops])
        Gs = self.G(np.einsum("sdk,hd->hsk", R, h))
        ph = 2 * np.pi * np.mod(h @ t.T, 1.0)
        return Gs, np.stack([np.cos(ph), np.sin(ph)], axis=-1)


def ft_aopair_cryst(mol, crystal, hkl):
    """Symmetrised, thermally smeared AO-pair transforms, complex [N_h, nao, nao]:
        B_mu,nu(h) = sum_s exp(+2 pi i h.t_s) T_mu,nu(G_{h_s}) A_mu,nu(G_{h_s}),   h_s = R_s^T h,
    A = `ft_aopair`, T_mu,nu(G) = (T_A(G) + T_B(G)) / 2 for mu on atom A and nu on atom B, T_A(G) = exp(-G^T U_A G / 2).
    For a one-centre pair T is the exact Debye-Waller factor of a rigidly displaced atom; for a two-centre pair the
    arithmetic mean is a convention.  F_calc(h) = sum D_mu,nu B_mu,nu(h) is then the structure factor of the unit cell
    (all copies of the molecule, smeared).  Host path of the 'Fobs' target and reference of `ecw_ft_aopair_cryst`."""
    Gs, ph = crystal.tables(hkl)
    U = crystal.adp_bohr(len(mol.Z))
    at = mol.ao_atom
    out = np.zeros((len(Gs), mol.nao, mol.nao), dtype=np.complex128)
    for s in range(crystal.nsym):
        G = Gs[:, s]
        T = np.exp(-0.5 * np.einsum("hi,aij,hj->ha", G, U, G))      # [N_h, natom]
        Tp = 0.5 * (T[:, at][:, :, None] + T[:, at][:, None, :])
        out += (ph[:, s, 0] + 1j * ph[:, s, 1])[:, None, None] * Tp * ft_aopair(mol, G)
    return out


def ao_values(mol, points):
    """AO values phi_mu(r), [P, nao], at points [P, 3] in bohr: phi_mu(r) = sum_{p in mu} coef_p (x-A_x)^l (y-A_y)^m
    (z-A_z)^n exp(-alpha_p |r-A|^2), each AO's primitives added in table order with no screening.  The reference of
    the AO-value kernel of `ecw_density_grid`."""
    r = np.atleast_2d(np.asarray(points, dtype=np.float64))
    if r.ndim != 2 or r.shape[1] != 3:
        raise ValueError("points must be a [P, 3] array (bohr)")
    out = np.zeros((len(r), mol.nao))
    for q in range(len(mol.ex)):
        d = r - mol.cen[q]
        r2 = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]
        lx, ly, lz = mol.lmn[q]
        out[:, mol.ao[q]] += mol.coef[q] * d[:, 0] ** lx * d[:, 1] ** ly * d[:, 2] ** lz * np.exp(-mol.ex[q] * r2)
    return out


def density_points(mol, dm, points, chunk=65536):
    """rho(r) = sum_mu,nu dm_mu,nu phi_mu(r) phi_nu(r) in e/bohr^3 at points [P, 3] (bohr), for an AO density dm
    [nao, nao] (need not be symmetric).  The reference of `ecw_density_grid`."""
    dm = np.asarray(dm, dtype=np.float64)
    if dm.shape != (mol.nao, mol.nao):
        raise ValueError("dm must be an (nao, nao) AO density matrix")
    r = np.atleast_2d(np.asarray(points, dtype=np.float64))
    out = np.empty(len(r))
    for p0 in range(0, len(r), chunk):
        phi = ao_values(mol, r[p0:p0 + chunk])
        out[p0:p0 + chunk] = ((phi @ dm) * phi).sum(1)
    return out


def fourier_synthesis(hkl_half, F_half, F000, volume_bohr3, shape, chunk=256):
    """rho(x_ijk) = (F000 + 2 sum_h (Re F_h cos 2 pi h.x + Im F_h sin 2 pi h.x)) / V at x_ijk = (i/n1, j/n2, k/n3), a
    direct sum over the half set (the Friedel mates are implied): the inverse of the exp(+i G.r) sign of `ft_aopair`.
    The phases are exact: (h_d i_d) mod n_d in integers, then a table of 2 pi m / n_d.  Returns [n1, n2, n3]."""
    shape = tuple(int(n) for n in shape)
    h = np.asarray(hkl_half, dtype=np.int64).reshape(-1, 3)
    F = np.asarray(F_half, dtype=np.complex128).reshape(-1)
    tabs = [np.exp(2j * np.pi * np.arange(n) / n) for n in shape]
    acc = np.zeros(shape)
    for c0 in range(0, len(h), chunk):
        hc = h[c0:c0 + chunk]
        e = [tabs[d][np.mod(hc[:, d:d + 1] * np.arange(shape[d]), shape[d])] for d in range(3)]
        e12 = np.conj(F[c0:c0 + chunk])[:, None, None] * e[0][:, :, None] * e[1][:, None, :]
        acc += np.einsum("cij,ck->ijk", e12, e[2]).real             # Re[conj(F) exp(2 pi i h.x)]
    return (F000 + 2 * acc) / volume_bohr3


def fourier_map(crystal, hkl, F, shape, group=None):
    """Fourier map (1/V) sum_h F(h) exp(-2 pi i h.x) in e/bohr^3 on the [n1, n2, n3] fractional grid of `crystal`, from
    structure factors F of the reflections hkl expanded to the full sphere by `crystal.expand(hkl, F, group)`.  A direct
    sum for small grids: the reference of `ecw_fourier_map`."""
    shape = tuple(int(n) for n in shape)
    if len(shape) != 3 or min(shape) < 1:
        raise ValueError("shape must be three positive grid dimensions")
    hh, Fh, F000 = crystal.expand(hkl, F, group)
    return fourier_synthesis(hh, Fh, F000, crystal.volume_bohr3, shape)


def rhf(mol, ints=None, conv=1e-11, maxiter=100):
    """Closed-shell SCF with DIIS.  Returns (E_HF, mo_energy, mo_coeff, ints)."""
    S, T, V, eri = ints if ints is not None else integrals(mol)
    h = T + V
    nocc = mol.nelec // 2
    s, U = np.linalg.eigh(S)
    X = U / np.sqrt(s)
    e, C = np.linalg.eigh(X.T @ h @ X)
    C = X @ C
    D = 2 * C[:, :nocc] @ C[:, :nocc].T
    fs, es = [], []
    E_old = 0.0
    for it in range(maxiter):
        F = h + np.einsum("mnls,ls->mn", eri, D) - 0.5 * np.einsum("mlns,ls->mn", eri, D)
        E = 0.5 * np.sum(D * (h + F)) + mol.e_nuc
        err = X.T @ (F @ D @ S - S @ D @ F) @ X
        fs.append(F); es.append(err)
        fs, es = fs[-8:], es[-8:]
        if len(fs) > 1:
            n = len(fs)
            Bm = -np.ones((n + 1, n + 1)); Bm[n, n] = 0.0
            for i in range(n):
                for j in range(n):
                    Bm[i, j] = np.sum(es[i] * es[j])
            rhs = np.zeros(n + 1); rhs[n] = -1.0
            try:
                c = np.linalg.solve(Bm, rhs)[:n]
                F = sum(ci * fi for ci, fi in zip(c, fs))
            except np.linalg.LinAlgError:
                pass
        e, C = np.linalg.eigh(X.T @ F @ X)
        C = X @ C
        D = 2 * C[:, :nocc] @ C[:, :nocc].T
        if abs(E - E_old) < conv and np.abs(err).max() < 1e-8:
            break
        E_old = E
    F = h + np.einsum("mnls,ls->mn", eri, D) - 0.5 * np.einsum("mlns,ls->mn", eri, D)
    E = 0.5 * np.sum(D * (h + F)) + mol.e_nuc
    e, C = np.linalg.eigh(X.T @ F @ X)
    return float(E), e, X @ C, (S, T, V, eri)


class geris(object):
    """The attribute surface of the reference's `Eris.geris` (Eris.py:132-154) from an RHF solution:
    spin orbitals in [alpha, beta, alpha, beta, ...] order (orbspin = 0,1,0,1,...), `fock = diag(mo_energy)`,
    `<pq||rs> = (pr|qs) - (ps|qr)` with the spin selection rules, all sixteen o/v blocks."""

    def __init__(self, mol, scf_result=None):
        ehf, e, C, (S, T, V, eri) = scf_result if scf_result is not None else rhf(mol)
        nmo = C.shape[1]
        mo = np.einsum("mp,mnls->pnls", C, eri)
        mo = np.einsum("nq,pnls->pqls", C, mo)
        mo = np.einsum("lr,pqls->pqrs", C, mo)
        mo = np.einsum("st,pqrs->pqrt", C, mo)                  # (pq|rs), spatial MOs, chemists' notation
        n = 2 * nmo
        sp = np.arange(n) // 2                                   # spatial index of spin orbital
        spin = np.arange(n) % 2
        g = mo[np.ix_(sp, sp, sp, sp)] * (spin[:, None, None, None] == spin[None, :, None, None]) \
            * (spin[None, None, :, None] == spin[None, None, None, :])       # (pq|rs) spin orbitals
        phys = g.transpose(0, 2, 1, 3)                           # <pq|rs> = (pr|qs)
        anti = phys - phys.transpose(0, 1, 3, 2)
        o = mol.nelec
        self.nocc = o
        self.fock = np.diag(np.repeat(e, 2))
        self.mo_energy = np.repeat(e, 2)
        self.mo_occ = np.concatenate([np.ones(o), np.zeros(n - o)])
        self.orbspin = spin
        self.mo_coeff = C
        nao = C.shape[0]
        self.mo_coeff_g = np.zeros((2 * nao, n))                 # G format: [[C, 0], [0, C]] with interleaved columns,
        self.mo_coeff_g[:nao, 0::2] = C                           # what scf.addons.convert_to_ghf(mf).mo_coeff holds
        self.mo_coeff_g[nao:, 1::2] = C
        self.EHF = self.e_hf = ehf
        sl = {"o": slice(0, o), "v": slice(o, n)}
        for name in ("oooo", "ooov", "oovv", "ovov", "ovvo", "ovvv", "vvvv", "vooo", "vovo", "oovo", "vovv", "vvoo", "vvvo",
                     "voov", "ovoo"):
            setattr(self, name, np.ascontiguousarray(anti[sl[name[0]], sl[name[1]], sl[name[2]], sl[name[3]]]))
