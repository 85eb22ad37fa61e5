"""Amplitude target 'Fobs' of `exp_pot.Exp` on the host: the cell metric of `molint.Crystal`, the symop parser, the
symmetrised smeared planes `molint.ft_aopair_cryst` against explicit symmetry copies of the molecule, the electron
count, the closed-form scale, the potential against finite differences of the penalty, the statistics, input
validation, and the C entries without a device."""
import numpy as np
import pytest
from scipy.optimize import minimize_scalar

from helpers import load_golden
from oracle.make_golden_h2o import H2O

P21C = ['x,y,z', '-x,y+1/2,-z+1/2', '-x,-y,-z', 'x,-y+1/2,z+1/2']
MONO = (7.0, 8.0, 9.0, 90.0, 104.0, 90.0)


@pytest.fixture(scope="module")
def water():
    from ecw_cc_b200 import molint
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    return mol, molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol)))


def aniso_adp(natom, seed):
    """Random positive-definite Cartesian U tensors, Angstrom^2."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(natom):
        x = 0.03 * rng.standard_normal((3, 3))
        out.append(0.01 * np.eye(3) + x @ x.T)
    return out


def reflections(n, seed=0, r=3):
    rng = np.random.default_rng(seed)
    hkl = np.array([(h, k, l) for h in range(-r, r + 1) for k in range(-r, r + 1) for l in range(-r, r + 1)
                    if (h, k, l) != (0, 0, 0)])
    return np.concatenate([[[0, 0, 0]], hkl[rng.choice(len(hkl), n - 1, replace=False)]])


def spin_summed(er, rdm1):
    from ecw_cc_b200 import utilities
    C = er.mo_coeff_g
    return utilities.convert_g_to_ru_rdm1(C @ rdm1 @ C.T)[0]


# -- the crystal --------------------------------------------------------------------------------------------------------
def test_cell_metric_triclinic():
    """|G_h| = 2 pi / d_h with the textbook triclinic 1/d^2; M has the cell's lengths and angles."""
    from ecw_cc_b200 import molint
    a, b, c, al, be, ga = 7.1, 8.3, 9.2, 81.0, 97.0, 104.0
    cr = molint.Crystal((a, b, c, al, be, ga))
    ca, cb, cg = np.cos(np.deg2rad([al, be, ga]))
    sa, sb, sg = np.sin(np.deg2rad([al, be, ga]))
    hkl = reflections(40, 1)[1:]
    h, k, l = hkl.T
    inv_d2 = (h ** 2 / a ** 2 * sa ** 2 + k ** 2 / b ** 2 * sb ** 2 + l ** 2 / c ** 2 * sg ** 2
              + 2 * k * l / (b * c) * (cb * cg - ca) + 2 * h * l / (a * c) * (cg * ca - cb)
              + 2 * h * k / (a * b) * (ca * cb - cg)) / (1 - ca ** 2 - cb ** 2 - cg ** 2 + 2 * ca * cb * cg)
    G = np.linalg.norm(cr.G(hkl), axis=1) * molint.ANGSTROM
    assert np.abs(G - 2 * np.pi * np.sqrt(inv_d2)).max() < 1e-12 * G.max()
    M = cr.M
    assert np.allclose(np.linalg.norm(M, axis=0), [a, b, c], rtol=0, atol=1e-12)
    cos = lambda u, v: u @ v / np.linalg.norm(u) / np.linalg.norm(v)
    assert np.allclose([cos(M[:, 1], M[:, 2]), cos(M[:, 0], M[:, 2]), cos(M[:, 0], M[:, 1])], [ca, cb, cg], atol=1e-14)
    assert M[1, 0] == M[2, 0] == M[2, 1] == 0
    assert np.allclose(cr.cartesian([[1, 0, 0], [0.5, 0.5, 0.5]]), [M[:, 0], 0.5 * M.sum(1)], atol=1e-14)
    assert abs(cr.volume - abs(np.linalg.det(M))) < 1e-10
    # G_h . (M x) = 2 pi h . x for fractional x
    x = np.array([0.3, -0.2, 0.7])
    assert np.allclose(cr.G(hkl) @ (M @ x) * molint.ANGSTROM, 2 * np.pi * hkl @ x, atol=1e-12)


def test_three_length_cell_gives_the_G_of_F(water):
    from ecw_cc_b200 import exp_pot, molint
    mol, er = water
    cell = (8.0, 9.0, 10.0)
    hkl = reflections(30, 2)
    vx = exp_pot.Exp(0.1, [[['F', np.ones(len(hkl)), hkl, cell]]], mol, er.mo_coeff_g)
    assert np.array_equal(molint.Crystal(cell).G(hkl), vx.sf[0, 0]["G"])
    assert np.array_equal(molint.Crystal(cell + (90.0, 90.0, 90.0)).G(hkl), vx.sf[0, 0]["G"])


def test_symop_parser():
    from ecw_cc_b200 import molint
    for s in ['x,y,z', '-x,y+1/2,-z+1/2', 'x-y,x,z+1/6', '-y,x-y,z+1/3', 'x+1/2,y+1/2,z', '-x,-y,-z', 'y,x,-z+3/4',
              'x+1/4,-z+3/4,y+1/4']:
        R, t = molint.parse_symop(s)
        assert molint.symop_string(R, t) == s
        R2, t2 = molint.parse_symop(molint.symop_string(R, t))
        assert np.array_equal(R, R2) and np.array_equal(t, t2)
    R, t = molint.parse_symop(' -X , Y+1/2 , -Z+0.5 ')
    assert np.array_equal(R, np.diag([-1, 1, -1])) and np.allclose(t, [0, 0.5, 0.5])
    R, t = molint.parse_symop((np.diag([1, -1, 1]), (0.0, 0.5, 0.5)))
    assert molint.symop_string(R, t) == 'x,-y+1/2,z+1/2'
    for bad in ['x,y', 'x,y,w', 'x,y,z,x', 'x,,z', '1/2x,y,z', '0.5x,y,z', 'x,x,z', 'x+y,x+y,z', 'x,y,z+',
                (np.eye(3) * 0.5, (0, 0, 0)), (np.zeros((3, 3)), (0, 0, 0)), (np.eye(2), (0, 0)), 'x*y,y,z']:
        with pytest.raises(ValueError):
            molint.parse_symop(bad)


def test_crystal_validation():
    from ecw_cc_b200 import molint
    for cell in [(8.0, 9.0), (8.0, -9.0, 10.0), (8.0, 9.0, 10.0, 90.0, 0.0, 90.0), (8.0, 9.0, 10.0, 90.0, 180.0, 90.0),
                 (8.0, 9.0, 10.0, 150.0, 150.0, 150.0), (8.0, np.nan, 10.0)]:
        with pytest.raises(ValueError):
            molint.Crystal(cell)
    with pytest.raises(ValueError):
        molint.Crystal((8.0, 9.0, 10.0), symops=[])
    with pytest.raises(ValueError):
        molint.Crystal((8.0, 9.0, 10.0), adp=[np.array([[0.01, 0.02, 0], [0, 0.01, 0], [0, 0, 0.01]])])   # not symmetric
    with pytest.raises(ValueError):
        molint.Crystal((8.0, 9.0, 10.0), adp=[np.diag([0.01, -0.02, 0.01])])                              # not PSD
    cr = molint.Crystal((8.0, 9.0, 10.0), adp=[None, 0.02, np.diag([0.01, 0.02, 0.03])])
    U = cr.adp_bohr(3)
    assert np.array_equal(U[0], np.zeros((3, 3))) and np.allclose(U[1], 0.02 * molint.ANGSTROM ** 2 * np.eye(3))
    with pytest.raises(ValueError):
        cr.adp_bohr(4)


# -- the planes ---------------------------------------------------------------------------------------------------------
def test_identity_crystal_is_ft_aopair(water):
    from ecw_cc_b200 import molint
    mol, _ = water
    cr = molint.Crystal((8.0, 9.0, 10.0))
    hkl = reflections(20, 3)
    assert np.abs(molint.ft_aopair_cryst(mol, cr, hkl) - molint.ft_aopair(mol, cr.G(hkl))).max() <= 1e-15


def parity(mol, w):
    """+-1 per AO under the diagonal sign matrix diag(w): the parity of its Cartesian components."""
    first = np.searchsorted(mol.ao, np.arange(mol.nao))
    return np.prod(np.asarray(w)[None, :] ** mol.lmn[first], axis=1)


@pytest.mark.parametrize("basis", ["6-31g**", "cc-pvdz"])
def test_symmetry_by_explicit_copies(basis):
    """P2_1/c in a monoclinic cell (beta != 90): every W_s = M R_s M^-1 is a diagonal sign matrix, so the cell's density
    is that of a supermolecule of four copies (atoms at W_s r + M t_s) with densities S_s D S_s (S_s the AO parities).
    sum D B must equal the transform of that supermolecule, with the smearing (T_A' + T_B')/2, U' = W U W^T, applied
    per pair by hand."""
    from ecw_cc_b200 import molint
    cr0 = molint.Crystal(MONO)
    shift = cr0.cartesian([0.21, 0.13, 0.32])
    atoms = [(s, tuple(np.asarray(r) + shift)) for s, r in H2O]
    mol = molint.Molecule(atoms, basis)
    adp = aniso_adp(len(atoms), 4)
    cr = molint.Crystal(MONO, P21C, adp)
    hkl = reflections(16, 5, r=2)
    rng = np.random.default_rng(6)
    X = rng.standard_normal((mol.nao, mol.nao))
    D = X + X.T
    got = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, hkl), D)

    M, Minv = cr.M, np.linalg.inv(cr.M)
    super_atoms, blocks, U_super = [], [], []
    for R, t in cr.ops:
        W = M @ R @ Minv
        assert np.abs(W - np.diag(np.round(np.diag(W)))).max() < 1e-12
        w = np.round(np.diag(W))
        for (s, r), U in zip(atoms, adp):
            super_atoms.append((s, tuple(w * np.asarray(r) + M @ t)))
            U_super.append(np.diag(w) @ U @ np.diag(w))
        S = parity(mol, w)
        blocks.append(S[:, None] * D * S[None, :])
    sup = molint.Molecule(super_atoms, basis)
    nao = mol.nao
    Dsup = np.zeros((4 * nao, 4 * nao))
    for s, b in enumerate(blocks):
        Dsup[s * nao:(s + 1) * nao, s * nao:(s + 1) * nao] = b
    G = cr.G(hkl)
    A = molint.ft_aopair(sup, G)
    U_b = np.array(U_super) * molint.ANGSTROM ** 2
    T = np.exp(-0.5 * np.einsum('hi,aij,hj->ha', G, U_b, G))[:, sup.ao_atom]
    want = np.einsum('hij,ij->h', 0.5 * (T[:, :, None] + T[:, None, :]) * A, Dsup)
    assert np.abs(got - want).max() <= 1e-11 * np.abs(want).max(), np.abs(got - want).max()


def test_electron_count_and_isotropic_smearing(water):
    from ecw_cc_b200 import molint
    mol, er = water
    D = spin_summed(er, np.diag(er.mo_occ))
    hkl = reflections(12, 7)
    static = molint.Crystal(MONO, P21C)
    u = 0.025
    smeared = molint.Crystal(MONO, P21C, [u] * 3)
    Fs = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, static, hkl), D)
    Ft = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, smeared, hkl), D)
    assert abs(Fs[0] - 4 * 10) < 1e-8 and abs(Ft[0] - 4 * 10) < 1e-8
    g2 = (static.G(hkl) ** 2).sum(1)
    assert np.abs(Ft - np.exp(-0.5 * u * molint.ANGSTROM ** 2 * g2) * Fs).max() < 1e-13


# -- the target ---------------------------------------------------------------------------------------------------------
def make_target(water, n=24, seed=8):
    """F_obs from a perturbed density in P2_1/c with ADPs, random sigma."""
    from ecw_cc_b200 import exp_pot, molint
    from oracle.make_golden_solver import target_rdm1
    mol, er = water
    cr = molint.Crystal(MONO, P21C, aniso_adp(3, 9))
    hkl = reflections(n, seed)
    rng = np.random.default_rng(seed)
    probe = exp_pot.Exp(0.0, [[['Fobs', np.ones(n), None, hkl, cr]]], mol, er.mo_coeff_g)
    probe.Vexp_update(target_rdm1(10, 16), target_rdm1(10, 16), (0, 0))
    a = np.abs(probe.prop_calc[0][1])
    sigma = 0.02 + 0.05 * rng.uniform(size=n) * a.mean()
    F_obs = 1.7 * a + sigma * rng.standard_normal(n)
    return np.abs(F_obs), sigma, hkl, cr


def penalty(vx, rdm1):
    vx.Vexp_update(rdm1, rdm1, (0, 0))
    return vx.prop_calc[0][3]


def test_scale_is_the_chi2_minimum(water):
    from ecw_cc_b200 import exp_pot
    from oracle.make_golden_solver import target_rdm1
    mol, er = water
    F_obs, sigma, hkl, cr = make_target(water)
    vx = exp_pot.Exp(0.3, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, er.mo_coeff_g)
    rdm1 = target_rdm1(10, 16) + 0.002 * np.random.default_rng(1).standard_normal((26, 26))
    vx.Vexp_update(rdm1, rdm1, (0, 0))
    name, F_c, k, chi2 = vx.prop_calc[0]
    assert name == 'Fobs' and np.iscomplexobj(F_c) and F_c.shape == (len(hkl),)
    w = 1 / sigma ** 2
    f = lambda s: np.sum(w * (s * np.abs(F_c) - F_obs) ** 2) / (len(hkl) - 1)
    best = minimize_scalar(f, bracket=(0.5 * k, k, 2 * k), tol=1e-12)
    assert abs(best.x - k) < 1e-6 * k and abs(chi2 - f(k)) < 1e-12 * chi2 and f(k) <= best.fun * (1 + 1e-14)
    # fixed scale: k and the N_h denominator as given
    vf = exp_pot.Exp(0.3, [[['Fobs', F_obs, sigma, hkl, cr, 1.5]]], mol, er.mo_coeff_g)
    vf.Vexp_update(rdm1, rdm1, (0, 0))
    assert vf.prop_calc[0][2] == 1.5
    assert abs(vf.prop_calc[0][3] - np.sum(w * (1.5 * np.abs(F_c) - F_obs) ** 2) / len(hkl)) < 1e-12 * chi2


@pytest.mark.parametrize("k_fixed", [None, 1.6])
def test_potential_is_the_penalty_gradient(water, k_fixed):
    """Vexp = -dP/dgamma for P = L chi^2, k re-refined at each displaced point (or fixed): central differences along
    random symmetric directions."""
    from ecw_cc_b200 import exp_pot
    from oracle.make_golden_solver import target_rdm1
    mol, er = water
    F_obs, sigma, hkl, cr = make_target(water)
    L = 0.3
    tgt = ['Fobs', F_obs, sigma, hkl, cr] + ([] if k_fixed is None else [k_fixed])
    vx = exp_pot.Exp(L, [[tgt]], mol, er.mo_coeff_g)
    rng = np.random.default_rng(11)
    rdm1 = target_rdm1(10, 16) + 0.002 * rng.standard_normal((26, 26))
    rdm1 = 0.5 * (rdm1 + rdm1.T)
    vx.Vexp_update(rdm1, rdm1, (0, 0))
    V = vx.Vexp[0, 0].copy()
    assert np.abs(V - V.T).max() < 1e-12
    eps = 1e-5                                                  # |F_c| makes P non-quadratic: O(eps^2) truncation
    for _ in range(3):
        X = rng.standard_normal(rdm1.shape)
        X = 0.5 * (X + X.T)
        fd = L * (penalty(vx, rdm1 + eps * X) - penalty(vx, rdm1 - eps * X)) / (2 * eps)
        an = -np.sum(V * X)
        assert abs(fd - an) <= 1e-7 * abs(an), (fd, an)


def test_extinguished_reflections_do_not_steer_the_fit(water):
    """The HF density of water keeps the molecule's point symmetry, which extinguishes some reflections of this cell:
    their F_c is rounding noise (|F_c| <= 1e-12 max |F_c|), |F| has a cusp there, and they add nothing to the
    potential.  The potential equals that of the target without them (whose chi^2 denominator and scale differ, so
    the comparison uses a fixed scale and rescales L by the degrees of freedom)."""
    from ecw_cc_b200 import exp_pot, molint
    mol, er = water
    cr = molint.Crystal(MONO, P21C, [0.02, 0.03, 0.03])
    hkl = reflections(60, 12, r=4)[1:]
    hf = np.diag(er.mo_occ)
    probe = exp_pot.Exp(0.0, [[['Fobs', np.ones(len(hkl)), None, hkl, cr]]], mol, er.mo_coeff_g)
    probe.Vexp_update(hf, hf, (0, 0))
    a = np.abs(probe.prop_calc[0][1])
    cusp = a <= molint.FOBS_ZERO * a.max()
    assert cusp.any() and (a[cusp] < 1e-14 * a.max()).all() and (a[~cusp] > 1e-6 * a.max()).all()
    F_obs = np.random.default_rng(13).uniform(0.5, 2.0, len(hkl))
    full = exp_pot.Exp(0.3, [[['Fobs', F_obs, None, hkl, cr, 1.3]]], mol, er.mo_coeff_g)
    full.Vexp_update(hf, hf, (0, 0))
    keep = ~cusp
    part = exp_pot.Exp(0.3 * keep.sum() / len(hkl), [[['Fobs', F_obs[keep], None, hkl[keep], cr, 1.3]]], mol,
                       er.mo_coeff_g)
    part.Vexp_update(hf, hf, (0, 0))
    assert np.abs(full.Vexp[0, 0] - part.Vexp[0, 0]).max() <= 1e-12 * np.abs(part.Vexp[0, 0]).max()


def test_statistics(water):
    from ecw_cc_b200 import exp_pot
    from oracle.make_golden_solver import target_rdm1
    mol, er = water
    F_obs, sigma, hkl, cr = make_target(water)
    rdm1 = target_rdm1(10, 16)
    vx = exp_pot.Exp(0.3, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, er.mo_coeff_g)
    Delta, vmax = vx.Vexp_update(rdm1, rdm1, (0, 0))
    _, F_c, k, _ = vx.prop_calc[0]
    assert abs(Delta - np.sum(np.abs(k * np.abs(F_c) - F_obs)) / np.sum(F_obs)) < 1e-14
    assert vmax == np.max(np.abs(vx.Vexp[0, 0]))
    # relative to HF: F_HF complex or as amplitudes, with the HF amplitudes' own refined scale
    hf = np.diag(er.mo_occ)
    vx.Vexp_update(hf, hf, (0, 0))
    F_hf = vx.prop_calc[0][1]
    w = 1 / sigma ** 2
    a_hf = np.abs(F_hf)
    k_hf = np.sum(w * F_obs * a_hf) / np.sum(w * a_hf ** 2)
    for hf_entry in (F_hf, a_hf):
        vh = exp_pot.Exp(0.3, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, er.mo_coeff_g, HF_prop=[[hf_entry]])
        d2, _ = vh.Vexp_update(rdm1, rdm1, (0, 0))
        assert abs(d2 - np.sum(np.abs(k * np.abs(F_c) - F_obs)) / np.sum(np.abs(k_hf * a_hf - F_obs))) < 1e-13
    vk = exp_pot.Exp(0.3, [[['Fobs', F_obs, sigma, hkl, cr, 1.2]]], mol, er.mo_coeff_g, HF_prop=[[F_hf]])
    d3, _ = vk.Vexp_update(rdm1, rdm1, (0, 0))
    assert abs(d3 - np.sum(np.abs(1.2 * np.abs(F_c) - F_obs)) / np.sum(np.abs(1.2 * a_hf - F_obs))) < 1e-13
    # any diagonal state: here an excited state
    ve = exp_pot.Exp(0.3, [[['mat', rdm1]], [['Fobs', F_obs, None, hkl, cr]]], mol, er.mo_coeff_g)
    de, _ = ve.Vexp_update(rdm1, rdm1, (1, 1))
    assert ve.prop_calc[0][0] == 'Fobs' and ve.Vexp[1, 1].shape == rdm1.shape
    ke = ve.prop_calc[0][2]
    assert abs(ke - np.sum(F_obs * np.abs(F_c)) / np.sum(np.abs(F_c) ** 2)) < 1e-13 * ke
    assert abs(de - np.sum(np.abs(ke * np.abs(F_c) - F_obs)) / np.sum(F_obs)) < 1e-14
    assert not ve.device_fobs_ready()


def test_input_validation(water):
    from ecw_cc_b200 import exp_pot, molint
    mol, er = water
    hkl = reflections(4)
    C = er.mo_coeff_g
    cr = molint.Crystal(MONO, P21C)
    one = np.ones(4)
    with pytest.raises(NotImplementedError, match="molint.Molecule"):
        exp_pot.Exp(0.1, [[['Fobs', one, None, hkl, cr]]], None, C)
    bad = [
        ['Fobs', -one, None, hkl, cr],                          # negative amplitude
        ['Fobs', one * (1 + 1j), None, hkl, cr],                # complex
        ['Fobs', [1.0, np.nan, 1.0, 1.0], None, hkl, cr],       # not finite
        ['Fobs', one[:3], None, hkl, cr],                       # length mismatch
        ['Fobs', one, np.zeros(4), hkl, cr],                    # sigma = 0
        ['Fobs', one, -one, hkl, cr],                           # sigma < 0
        ['Fobs', one, one[:3], hkl, cr],                        # sigma length
        ['Fobs', one, None, hkl[:, :2], cr],                    # hkl not (N_h, 3)
        ['Fobs', one, None, hkl + 0.5, cr],                     # hkl not integer
        ['Fobs', one, None, hkl, (8.0, 9.0, 10.0)],             # not a Crystal
        ['Fobs', one, None, hkl, molint.Crystal(MONO, P21C, [0.01] * 4)],      # ADPs for 4 atoms, molecule has 3
        ['Fobs', one, None, hkl, cr, 0.0],                      # fixed scale not positive
        ['Fobs', one, None, hkl, cr, -1.0],
        ['Fobs', one[:1], None, hkl[:1], cr],                   # N_h = 1 with a refined scale
        ['Fobs', one, None, hkl],                               # no crystal
        ['Fobs', one, None, hkl, cr, 1.0, 2.0],                 # too long
    ]
    for target in bad:
        with pytest.raises(ValueError):
            exp_pot.Exp(0.1, [[target]], mol, C)
    for cell in [(8.0, 9.0), (8.0, 9.0, 10.0, 90.0, 200.0, 90.0)]:
        with pytest.raises(ValueError):
            molint.Crystal(cell)
    with pytest.raises(ValueError):
        exp_pot.Exp(0.1, [[['Fobs', one, None, hkl, cr]]], mol, None)
    assert exp_pot.Exp(0.1, [[['Fobs', one[:1], None, hkl[:1], cr, 1.0]]], mol, C).device_fobs_ready()   # fixed k
    vx = exp_pot.Exp(0.1, [[['Fobs', one, None, hkl, cr]]], mol, C)
    assert vx.device_fobs_ready() and not vx.device_sf_ready() and not vx.device_mat_ready()
    assert vx.dip_int is None and vx.Ek_int is None and vx.v1e_int is None
    two = [['Fobs', one, None, hkl, cr], ['Fobs', one, None, hkl, cr]]
    assert not exp_pot.Exp(0.1, [two], mol, C).device_fobs_ready()
    mixed = [['Fobs', one, None, hkl, cr], ['F', one, hkl, (8.0, 9.0, 10.0)]]
    assert not exp_pot.Exp(0.1, [mixed], mol, C).device_fobs_ready()
    assert not exp_pot.Exp(0.1, [[['F', one, hkl, (8.0, 9.0, 10.0)]]], mol, C).device_fobs_ready()


def test_c_entries_without_a_device(built_lib, water):
    import torch
    if torch.cuda.is_available():
        return
    from ecw_cc_b200 import EcwError, exp_pot, molint
    assert built_lib.ecw_ft_aopair_cryst(None, 1, None, None, 1, None, 1, None, None, 1, 1, None, None) != 0
    assert built_lib.ecw_vexp_sfobs(None, 2, None, 1, None, 2, None, None, 0.0, 0.1, None, None, None, None, None,
                                    None, None) != 0
    assert built_lib.ecw_vexp_sfobs_workspace_bytes(26, 13, 24) == built_lib.ecw_vexp_sf_workspace_bytes(26, 13, 24)
    assert built_lib.ecw_vexp_sfobs_workspace_bytes(26, 13, 24) > 8 * (2 * 13 * 26 + 2 * 169 + 48)
    assert built_lib.ecw_vexp_sfobs_workspace_bytes(26, 0, 24) < 0
    mol, _ = water
    with pytest.raises(EcwError, match="no CUDA device"):
        exp_pot.ft_aopair_cryst_device(mol, molint.Crystal(MONO, P21C), np.zeros((1, 3)), "cpu")
