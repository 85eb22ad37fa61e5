"""Structure-factor ('F') target of `exp_pot.Exp` on the host: the AO-pair Fourier transform `molint.ft_aopair` against
the overlap and dipole integrals and against quadrature, F_calc of the HF density, the potential against finite
differences of the penalty, input validation, and the C entries without a device."""
import numpy as np
import pytest
from scipy.integrate import quad

from helpers import load_golden
from oracle.make_golden_h2o import H2O

CELL = (8.0, 9.0, 10.0)


@pytest.fixture(scope="module")
def water():
    from ecw_cc_b200 import molint
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    return mol, molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol)))


def reflections(n=24):
    hkl = [(h, k, l) for h in range(0, 3) for k in range(-2, 3) for l in range(-2, 3) if (h, k, l) != (0, 0, 0)]
    return np.array([(0, 0, 0)] + hkl[:n - 1])


def test_ft_aopair_limits(water):
    """A(0) = S, A(-G) = conj A(G), A symmetric, and dA/dG at 0 = i <mu|r|nu>."""
    from ecw_cc_b200 import molint
    mol, _ = water
    assert np.abs(molint.ft_aopair(mol, np.zeros(3))[0] - molint.integrals(mol)[0]).max() < 1e-13
    G = np.random.default_rng(3).uniform(-3, 3, (5, 3))
    A, Am = molint.ft_aopair(mol, G), molint.ft_aopair(mol, -G)
    assert np.abs(Am - A.conj()).max() < 1e-14
    assert np.abs(A - A.transpose(0, 2, 1)).max() == 0
    eps = 1e-4
    Ad = molint.ft_aopair(mol, [[eps, 0, 0], [-eps, 0, 0]])
    assert np.abs((Ad[0] - Ad[1]) / (2 * eps) - 1j * molint.dipole_integrals(mol, (0., 0., 0.))[0]).max() < 1e-7


class _Pair(object):
    """Two unit-coefficient primitives on two centres: the minimal `Molecule` surface `ft_aopair` reads."""

    def __init__(self, la, lb, a, b, A, B):
        self.cen, self.ex = np.array([A, B], dtype=float), np.array([a, b], dtype=float)
        self.lmn, self.coef = np.array([la, lb]), np.ones(2)
        self.ao, self.nao = np.array([0, 1]), 2
        self.lmax = int(self.lmn.sum(1).max())


@pytest.mark.parametrize("la", ["s", "p", "d"])
@pytest.mark.parametrize("lb", ["s", "p", "d"])
def test_ft_aopair_against_quadrature(la, lb):
    """One off-centre primitive pair: the element is the product of three 1-D transforms
    int (x-A)^i (x-B)^j exp(-a (x-A)^2 - b (x-B)^2) exp(i g x) dx, each checked by quadrature."""
    from ecw_cc_b200 import molint
    lmn_a = {"s": (0, 0, 0), "p": (1, 0, 0), "d": (2, 0, 1)}[la]
    lmn_b = {"s": (0, 0, 0), "p": (0, 1, 0), "d": (2, 1, 0)}[lb]
    a, b = 0.9, 0.45
    A, B = np.array([0.3, -0.4, 0.2]), np.array([-0.5, 0.6, 1.1])
    pair = _Pair(lmn_a, lmn_b, a, b, A, B)
    Gs = np.array([[0.0, 0.0, 0.0], [0.7, -1.3, 0.4], [-2.1, 0.5, 1.7]])
    got = molint.ft_aopair(pair, Gs)[:, 0, 1]

    def one_d(i, j, Ad, Bd, g):
        f = lambda x, trig: (x - Ad) ** i * (x - Bd) ** j * np.exp(-a * (x - Ad) ** 2 - b * (x - Bd) ** 2) * trig(g * x)
        kw = dict(limit=400, epsabs=1e-14, epsrel=1e-13)
        return quad(f, -15, 15, args=(np.cos,), **kw)[0] + 1j * quad(f, -15, 15, args=(np.sin,), **kw)[0]
    for G, val in zip(Gs, got):
        want = np.prod([one_d(lmn_a[d], lmn_b[d], A[d], B[d], G[d]) for d in range(3)])
        assert abs(val - want) < 1e-10, (G, val, want)


def test_hf_density_counts_the_electrons(water):
    from ecw_cc_b200 import exp_pot
    mol, er = water
    hkl = reflections()
    vx = exp_pot.Exp(0.1, [[['F', np.ones(len(hkl)), hkl, CELL]]], mol, er.mo_coeff_g)
    vx.Vexp_update(np.diag(er.mo_occ), np.diag(er.mo_occ), (0, 0))
    name, fc = vx.prop_calc[0]
    assert name == 'F' and fc.shape == (len(hkl),)
    assert abs(fc[0] - 10.0) < 1e-8
    assert np.all(np.abs(fc[1:]) < 10.0)


def penalty(vx, rdm1, F_exp, w):
    vx.Vexp_update(rdm1, rdm1, (0, 0))
    return 0.5 * w * np.sum(np.abs(F_exp - vx.prop_calc[0][1]) ** 2)


def test_potential_is_the_penalty_gradient(water):
    """Vexp = -dP/dgamma for P = (w/2) sum_h |F_exp - F_calc|^2: central differences along random symmetric
    directions.  Also Delta, vmax and the HF-relative Delta."""
    from ecw_cc_b200 import exp_pot
    from oracle.make_golden_solver import target_rdm1
    mol, er = water
    hkl = reflections()
    rng = np.random.default_rng(7)
    F_exp = (1 + 0.1 * rng.standard_normal(len(hkl))) * np.exp(1j * rng.uniform(0, 2 * np.pi, len(hkl)))
    w = 0.3
    vx = exp_pot.Exp(w, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g)
    rdm1 = target_rdm1(10, 16)
    Delta, vmax = vx.Vexp_update(rdm1, rdm1, (0, 0))
    V = vx.Vexp[0, 0].copy()
    fc = vx.prop_calc[0][1]
    assert np.abs(V - V.T).max() < 1e-12
    assert abs(Delta - np.sum(np.abs(F_exp - fc)) / np.sum(np.abs(F_exp))) < 1e-14 and vmax == np.max(np.abs(V))
    eps = 1e-4
    for _ in range(3):
        X = rng.standard_normal(rdm1.shape)
        X = 0.5 * (X + X.T)
        fd = (penalty(vx, rdm1 + eps * X, F_exp, w) - penalty(vx, rdm1 - eps * X, F_exp, w)) / (2 * eps)
        an = -np.sum(V * X)
        assert abs(fd - an) <= 1e-7 * abs(an), (fd, an)
    # Delta relative to the HF structure factors
    hf = np.diag(er.mo_occ)
    vx.Vexp_update(hf, hf, (0, 0))
    F_hf = vx.prop_calc[0][1]
    vh = exp_pot.Exp(w, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g, HF_prop=[[F_hf]])
    d2, _ = vh.Vexp_update(rdm1, rdm1, (0, 0))
    assert abs(d2 - np.sum(np.abs(F_exp - fc)) / np.sum(np.abs(F_exp - F_hf))) < 1e-14
    # real F_exp (phase 0) is accepted and the target applies to any diagonal state
    vr = exp_pot.Exp(w, [[['mat', rdm1]], [['F', np.abs(F_exp), hkl, CELL]]], mol, er.mo_coeff_g)
    vr.Vexp_update(rdm1, rdm1, (1, 1))
    assert vr.prop_calc[0][0] == 'F' and vr.Vexp[1, 1].shape == rdm1.shape


def test_input_validation(water):
    from ecw_cc_b200 import exp_pot
    mol, er = water
    hkl = reflections(4)
    C = er.mo_coeff_g
    with pytest.raises(NotImplementedError, match="molint.Molecule"):
        exp_pot.Exp(0.1, [[['F', np.ones(4), hkl, CELL]]], None, C)

    class Mole(object):                                         # a PySCF Mole stand-in
        def intor_symmetric(self, name, comp=None):
            raise AssertionError

    with pytest.raises(NotImplementedError, match="PySCF"):
        exp_pot.Exp(0.1, [[['F', np.ones(4), hkl, CELL]]], Mole(), C)
    bad = [
        ['F', np.ones(3), hkl, CELL],                           # length mismatch
        ['F', np.ones((4, 1)), hkl, CELL],                      # not 1-D
        ['F', [1.0, np.nan, 1.0, 1.0], hkl, CELL],              # not finite
        ['F', np.ones(4), hkl[:, :2], CELL],                    # hkl not (N_h, 3)
        ['F', np.ones(4), hkl + 0.5, CELL],                     # hkl not integer
        ['F', np.ones(4), hkl, (8.0, 9.0)],                     # cell not three lengths
        ['F', np.ones(4), hkl, (8.0, -9.0, 10.0)],              # cell length not positive
        ['F', np.ones(4), hkl],                                 # no cell
    ]
    for target in bad:
        with pytest.raises(ValueError):
            exp_pot.Exp(0.1, [[target]], mol, C)
    with pytest.raises(ValueError):
        exp_pot.Exp(0.1, [[['F', np.ones(4), hkl, CELL]]], mol, None)
    vx = exp_pot.Exp(0.1, [[['F', np.ones(4), hkl, CELL]]], mol, C)
    assert vx.device_sf_ready() and not vx.device_mat_ready()
    two = [['F', np.ones(4), hkl, CELL], ['F', np.ones(4), hkl, CELL]]
    assert not exp_pot.Exp(0.1, [two], mol, C).device_sf_ready()


def test_c_entries_without_a_device(built_lib, water):
    import torch
    if torch.cuda.is_available():
        return
    from ecw_cc_b200 import EcwError, exp_pot
    assert built_lib.ecw_ft_aopair(None, 1, None, 1, None, 1, None, None) != 0
    assert built_lib.ecw_vexp_sf(None, 2, None, 1, None, 1, None, 0.1, None, None, None, None, None, None, None) != 0
    assert built_lib.ecw_vexp_sf_workspace_bytes(26, 13, 24) > 8 * (2 * 13 * 26 + 2 * 169 + 48)
    assert built_lib.ecw_vexp_sf_workspace_bytes(0, 13, 24) < 0
    mol, _ = water
    with pytest.raises(EcwError, match="no CUDA device"):
        exp_pot.ft_aopair_device(mol, np.zeros((1, 3)), "cpu")
