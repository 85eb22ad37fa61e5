"""Density maps on the host: AO values and densities on uniform grids against the overlap matrix and the electron count,
the sign of the Fourier synthesis, the symmetry expansion of `Crystal.expand` against explicit copies and full-sphere
data, Parseval's theorem, systematic absences, group closure, the residual-map coefficients, cube files, and input
validation (and `EcwError` without a device)."""
import ctypes

import numpy as np
import pytest

from helpers import load_golden
from oracle.make_golden_h2o import H2O

P21C = ['x,y,z', '-x,y+1/2,-z+1/2', '-x,-y,-z', 'x,-y+1/2,z+1/2']
MONO = (7.0, 8.0, 9.0, 90.0, 104.0, 90.0)


def uniform_grid(lo, hi, h):
    """Points lo + h (i, j, k) covering [lo, hi] per axis, [P, 3]."""
    axes = [lo[d] + h * np.arange(int(np.ceil((hi[d] - lo[d]) / h)) + 1) for d in range(3)]
    return np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3)


def test_ao_products_integrate_to_the_overlap():
    """Trapezoid rule on a uniform grid for the AOs of H2O/6-31G* whose exponents are all <= 0.8 bohr^-2 (the O d shell,
    the outer O sp shell and the outer H s functions: the O core, the O 2sp shell and the inner H s functions are left
    out).  A product of two such AOs has p <= 1.6 bohr^-2; by Poisson summation the relative error of the trapezoid
    rule with spacing h = 0.3 bohr is of order (pi / (h sqrt(p)))^4 exp(-pi^2 / (p h^2)) = 6e2 x 2e-30 per axis, and
    the box reaches 10 bohr beyond every atom, where the most diffuse product (p = 0.32) has fallen below 1e-13."""
    from ecw_cc_b200 import molint
    mol = molint.Molecule(H2O, "6-31g*")
    first = np.searchsorted(mol.ao, np.arange(mol.nao))
    pmax = np.array([mol.ex[mol.ao == mu].max() for mu in range(mol.nao)])
    keep = np.where(pmax <= 0.8)[0]
    assert any(mol.lmn[first[mu]].sum() == 2 for mu in keep)                # the d shell is in
    assert len(keep) == 11
    h = 0.3
    xyz = mol.atom_coords()
    pts = uniform_grid(xyz.min(0) - 10.0, xyz.max(0) + 10.0, h)
    phi = molint.ao_values(mol, pts)[:, keep]
    S_quad = h ** 3 * phi.T @ phi
    S = mol.intor_symmetric('int1e_ovlp')[np.ix_(keep, keep)]
    assert np.abs(S_quad - S).max() <= 1e-9, np.abs(S_quad - S).max()


def test_ao_values_at_a_point_by_hand():
    from ecw_cc_b200 import molint
    mol = molint.Molecule(H2O, "6-31g*")
    r = np.array([[0.3, -0.7, 1.1]])
    want = np.zeros(mol.nao)
    for q in range(len(mol.ex)):
        d = r[0] - mol.cen[q]
        want[mol.ao[q]] += mol.coef[q] * np.prod(d ** mol.lmn[q]) * np.exp(-mol.ex[q] * d @ d)
    assert np.abs(molint.ao_values(mol, r)[0] - want).max() <= 1e-15 * np.abs(want).max()


def test_h2_density_integrates_to_two_electrons():
    """H2/cc-pVDZ RHF.  The steepest product is p = 2 x 13.01 bohr^-2: spacing h = 0.12 bohr gives a relative trapezoid
    error of about 2 exp(-pi^2 / (p h^2)) = 7e-12 per axis; the box reaches 10 bohr beyond the atoms, where the most
    diffuse product (p = 0.244) is below 3e-11."""
    from ecw_cc_b200 import molint
    mol = molint.Molecule([("H", (0., 0., -0.37)), ("H", (0., 0., 0.37))], "cc-pvdz")
    _, _, C, (S, _, _, _) = molint.rhf(mol)
    D = 2 * C[:, :1] @ C[:, :1].T
    assert abs(np.sum(D * S) - 2) < 1e-12
    h = 0.12
    xyz = mol.atom_coords()
    pts = uniform_grid(xyz.min(0) - 10.0, xyz.max(0) + 10.0, h)
    n = h ** 3 * molint.density_points(mol, D, pts).sum()
    assert abs(n - 2) <= 1e-9, n - 2


# -- Fourier maps -------------------------------------------------------------------------------------------------------
def water_hf():
    """H2O/6-31G at its reference geometry, HF AO density from the stored MOs (a translation leaves them valid)."""
    g = load_golden("h2o_631g.npz")
    C = g["mo_coeff"]
    return 2 * C[:, :5] @ C[:, :5].T


def half_sphere(crystal, s_max):
    """The reflections h > 0 (or h = 0, k > 0, or h = k = 0, l > 0) with sin(theta)/lambda <= s_max (1/Angstrom)."""
    from ecw_cc_b200 import molint
    r = [int(np.ceil(2 * s_max * np.linalg.norm(crystal.M[:, d]))) + 1 for d in range(3)]
    hkl = np.array([(h, k, l) for h in range(0, r[0] + 1) for k in range(-r[1], r[1] + 1)
                    for l in range(-r[2], r[2] + 1) if h > 0 or k > 0 or (k == 0 and l > 0)])
    s = np.linalg.norm(crystal.G(hkl), axis=1) * molint.ANGSTROM / (4 * np.pi)
    return hkl[s <= s_max]


def test_fourier_map_peaks_at_the_oxygen_not_at_its_inversion():
    """P1 cell, water at a general position, F_calc to sin(theta)/lambda = 1/Angstrom with U_iso = 0.02 A^2: the map
    maximum lies within 0.2 A of O (mod lattice).  With the wrong sign of the synthesis it would lie at -x_O."""
    from ecw_cc_b200 import molint
    cell = (6.0, 7.0, 8.0, 80.0, 95.0, 105.0)
    cr0 = molint.Crystal(cell)
    x_O = np.array([0.31, 0.22, 0.27])
    shift = cr0.cartesian(x_O)
    mol = molint.Molecule([(s, tuple(np.asarray(r) + shift)) for s, r in H2O], "6-31g")
    cr = molint.Crystal(cell, adp=[0.02] * 3)
    hkl = half_sphere(cr, 1.0)
    assert len(hkl) > 3000
    F = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, hkl), water_hf())
    shape = (40, 47, 54)                                            # about 0.15 A apart
    rho = molint.fourier_map(cr, hkl, F, shape)
    peak = np.array(np.unravel_index(np.argmax(rho), shape)) / np.array(shape)

    def dist(x, y):
        d = x - y
        return np.linalg.norm(cr.M @ (d - np.round(d)))
    assert dist(peak, x_O) <= 0.2, dist(peak, x_O)
    assert dist(peak, -x_O) > 1.0


def parity(mol, w):
    """+-1 per AO under the diagonal sign matrix diag(w): the parity of its Cartesian components."""
    first = np.searchsorted(mol.ao, np.arange(mol.nao))
    return np.prod(np.asarray(w)[None, :] ** mol.lmn[first], axis=1)


def unique_set(crystal, hkl):
    """One representative of every orbit of hkl under {R_u^T, -R_u^T}: the lexicographically largest member."""
    keep = []
    for h in hkl:
        orbit = [tuple(s * (R.T @ h)) for R, _ in crystal.ops for s in (1, -1)]
        if tuple(h) == max(orbit):
            keep.append(h)
    return np.array(keep)


@pytest.fixture(scope="module")
def p21c():
    """H2O/6-31G* (with d functions) at a general position of P2_1/c, a random symmetric AO density, all reflections with
    |h_d| <= 3, their unique set and F_calc of both."""
    from ecw_cc_b200 import molint
    cr0 = molint.Crystal(MONO)
    shift = cr0.cartesian([0.21, 0.13, 0.32])
    atoms = [(s, tuple(np.asarray(r) + shift)) for s, r in H2O]
    mol = molint.Molecule(atoms, "6-31g*")
    cr = molint.Crystal(MONO, P21C)
    rng = np.random.default_rng(6)
    X = rng.standard_normal((mol.nao, mol.nao))
    D = X + X.T + 10 * np.eye(mol.nao)
    r = 3
    full = np.array([(h, k, l) for h in range(-r, r + 1) for k in range(-r, r + 1) for l in range(-r, r + 1)])
    uniq = unique_set(cr, full)
    F_full = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, full), D)
    F_uniq = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, uniq), D)
    return {"mol": mol, "atoms": atoms, "cr": cr, "D": D, "full": full, "uniq": uniq, "F_full": F_full,
            "F_uniq": F_uniq}


def test_expansion_matches_explicit_copies_and_full_sphere(p21c):
    """The map of the unique P2_1/c data expanded by `Crystal.expand` equals the map of the full sphere of P2_1/c data
    and that of an explicit four-copy supermolecule in P1 (W_s = M R_s M^-1 is a diagonal sign matrix in this cell, so
    copy s has atoms at W_s r + M t_s and density S_s D S_s, S_s the AO parities)."""
    from ecw_cc_b200 import molint
    cr, D, mol, atoms = p21c["cr"], p21c["D"], p21c["mol"], p21c["atoms"]
    shape = (8, 9, 7)                                               # n_d > 2 max |h_d|
    ref = molint.fourier_map(cr, p21c["uniq"], p21c["F_uniq"], shape)
    assert len(p21c["uniq"]) < len(p21c["full"]) / 3
    full = molint.fourier_map(cr, p21c["full"], p21c["F_full"], shape)

    M, Minv = cr.M, np.linalg.inv(cr.M)
    super_atoms, blocks = [], []
    for R, t in cr.ops:
        w = np.round(np.diag(M @ R @ Minv))
        super_atoms += [(s, tuple(w * np.asarray(r) + M @ t)) for s, r in atoms]
        S = parity(mol, w)
        blocks.append(S[:, None] * D * S[None, :])
    sup = molint.Molecule(super_atoms, "6-31g*")
    Dsup = np.zeros((sup.nao, sup.nao))
    for s, b in enumerate(blocks):
        Dsup[s * mol.nao:(s + 1) * mol.nao, s * mol.nao:(s + 1) * mol.nao] = b
    p1 = molint.Crystal(MONO)
    F_sup = np.einsum('hij,ij->h', molint.ft_aopair_cryst(sup, p1, p21c["full"]), Dsup)
    copies = molint.fourier_map(p1, p21c["full"], F_sup, shape)
    scale = np.abs(ref).max()
    assert np.abs(full - ref).max() <= 1e-12 * scale
    assert np.abs(copies - ref).max() <= 1e-12 * scale


def test_expand_returns_consistent_data_unchanged(p21c):
    cr = p21c["cr"]
    hh, Fh, F000 = cr.expand(p21c["uniq"], p21c["F_uniq"])
    idx = {tuple(h): i for i, h in enumerate(p21c["full"])}
    want = p21c["F_full"][[idx[tuple(h)] for h in hh]]
    assert np.abs(Fh - want).max() <= 1e-12 * np.abs(want).max()
    assert abs(F000 - p21c["F_full"][idx[(0, 0, 0)]].real) <= 1e-14 * F000
    assert len(hh) == (len(p21c["full"]) - 1) // 2
    # unmerged equivalents and Friedel mates with noise are averaged
    rng = np.random.default_rng(3)
    noisy = p21c["F_full"] + 0.01 * (rng.standard_normal(len(p21c["full"])) + 1j * rng.standard_normal(len(p21c["full"])))
    hn, Fn, _ = cr.expand(p21c["full"], noisy)
    assert np.array_equal(hn, hh)
    k = next(i for i, h in enumerate(hn) if tuple(h) == (1, 2, 3))
    contrib = []
    for R, t in cr.ops:
        for h, F in zip(p21c["full"], noisy):
            g = R.T @ h
            ph = np.exp(-2j * np.pi * np.mod(h @ t, 1.0))
            if tuple(g) == (1, 2, 3):
                contrib.append(ph * F)
            if tuple(-g) == (1, 2, 3):
                contrib.append(np.conj(ph * F))
    assert len(contrib) == 8 and abs(Fn[k] - np.mean(contrib)) <= 1e-13 * abs(Fn[k])


def test_parseval_and_mean(p21c):
    """On a grid with n_d > 2 max |h_d| the synthesis is an exact discrete inverse transform."""
    from ecw_cc_b200 import molint
    cr = p21c["cr"]
    hh, Fh, F000 = cr.expand(p21c["uniq"], p21c["F_uniq"])
    V = cr.volume_bohr3
    for shape in [(7, 7, 7), (8, 9, 10)]:
        rho = molint.fourier_map(cr, p21c["uniq"], p21c["F_uniq"], shape)
        ms = (F000 ** 2 + 2 * np.sum(np.abs(Fh) ** 2)) / V ** 2
        assert abs(np.mean(rho ** 2) - ms) <= 1e-12 * ms
        assert abs(np.mean(rho) - F000 / V) <= 1e-12 * F000 / V


def test_systematic_absences_expand_to_zero():
    """P2_1/c: 0k0 with k odd (the screw axis) and h0l with l odd (the glide plane) cancel, whatever F was given."""
    from ecw_cc_b200 import molint
    cr = molint.Crystal(MONO, P21C)
    hkl = np.array([(0, 1, 0), (0, 3, 0), (1, 0, 1), (2, 0, -3), (0, 2, 0), (1, 0, 2), (1, 1, 1)])
    F = np.array([5.0, 2 - 3j, 4j, 1.5, 3.0, 2.0 + 1j, 1.0])
    hh, Fh, _ = cr.expand(hkl, F)
    got = {tuple(h): f for h, f in zip(hh, Fh)}
    for h in [(0, 1, 0), (0, 3, 0), (1, 0, 1), (2, 0, -3)]:
        assert abs(got[h]) <= 1e-15 * 5, (h, got[h])
    for h in [(0, 2, 0), (1, 0, 2), (1, 1, 1)]:
        assert abs(got[h]) > 0.5


def test_closure_is_checked_and_group_repairs_it():
    """Coset representatives of a molecule on an inversion centre of P2_1/c ({1, -1} closed; {1, 2_1, -1} not)."""
    from ecw_cc_b200 import molint
    cr = molint.Crystal(MONO, ['x,y,z', '-x,-y,-z', '-x,y+1/2,-z+1/2'])
    hkl, F = np.array([(1, 2, 3), (0, 1, 1)]), np.array([1.0 + 1j, 2.0])
    with pytest.raises(ValueError, match="group="):
        cr.expand(hkl, F)
    with pytest.raises(ValueError, match="group="):
        molint.fourier_map(cr, hkl, F, (4, 4, 4))
    hh, Fh, _ = cr.expand(hkl, F, group=P21C)
    assert np.array_equal(hh, molint.Crystal(MONO, P21C).expand(hkl, F)[0])
    molint.Crystal(MONO, ['x,y,z', '-x,-y,-z']).expand(hkl, F)                  # closed
    molint.check_group([molint.parse_symop(s) for s in ['x,y,z', 'x+1/2,y+1/2,z']])   # centring: closed mod 1
    with pytest.raises(ValueError):
        molint.check_group([molint.parse_symop(s) for s in ['x,y,z', 'x+1/3,y,z']])


# -- residual map -------------------------------------------------------------------------------------------------------
def fobs_exp(L=0.1):
    """An evaluated 'Fobs' target of H2O/6-31G in P2_1/c: HF density, measured amplitudes of a perturbed density; the
    reflections include 0 0 0 and the absences 0 1 0 and 1 0 1, whose F_calc is rounding noise (FOBS_ZERO)."""
    from ecw_cc_b200 import exp_pot, molint
    from oracle.make_golden_solver import target_rdm1
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    er = molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol)))
    cr = molint.Crystal(MONO, P21C, [0.02, 0.03, 0.03])
    rng = np.random.default_rng(11)
    hkl = np.concatenate([[(0, 0, 0), (0, 1, 0), (1, 0, 1)], rng.integers(-3, 4, (40, 3))])
    probe = exp_pot.Exp(0.0, [[['Fobs', np.ones(len(hkl)), None, hkl, cr]]], mol, er.mo_coeff_g)
    probe.Vexp_update(target_rdm1(10, 16), target_rdm1(10, 16), (0, 0))
    F_obs = 1.7 * np.abs(probe.prop_calc[0][1]) + 0.05 * rng.uniform(size=len(hkl))
    vx = exp_pot.Exp(L, [[['Fobs', F_obs, 0.1 + 0.1 * rng.uniform(size=len(hkl)), hkl, cr]]], mol, er.mo_coeff_g)
    hf = np.diag(er.mo_occ)
    vx.Vexp_update(hf, hf, (0, 0))
    return vx, F_obs, hkl, cr


def test_residual_coefficients_by_hand():
    from ecw_cc_b200 import maps, molint
    vx, F_obs, hkl, cr = fobs_exp()
    _, F_c, k, _ = vx.prop_calc[0]
    a = np.abs(F_c)
    zero = a <= molint.FOBS_ZERO * a.max()
    assert zero[1] and zero[2]
    want = np.where(zero, 0.0, (F_obs / k - a)) * np.where(zero, 0.0, F_c / np.where(zero, 1.0, a))
    h, c, crystal = maps.residual_coefficients(vx)
    assert crystal is cr and np.array_equal(h, hkl[1:])                # 0 0 0 left out: F000 = 0
    assert np.abs(c - want[1:]).max() <= 1e-14 * np.abs(want).max()
    assert c[0] == 0 and c[1] == 0
    h2, c2, _ = maps.residual_coefficients(vx, index=(0, 0))
    assert np.array_equal(c2, c)
    # the host map of these coefficients has no mean (F000 = 0)
    rho = molint.fourier_map(cr, h, c, (8, 8, 8))
    assert abs(rho.mean()) <= 1e-14 * np.abs(rho).max()


def test_residual_map_needs_an_evaluated_fobs_target():
    from ecw_cc_b200 import exp_pot, maps, molint
    vx, F_obs, hkl, cr = fobs_exp()
    with pytest.raises(ValueError):
        maps.residual_coefficients(vx, index=(0, 1))
    fresh = exp_pot.Exp(0.1, vx.exp_data, vx.mol, vx.mo_coeff)
    with pytest.raises(ValueError, match="evaluated"):
        maps.residual_map(fresh, (8, 8, 8), "cpu")
    mat = exp_pot.Exp(0.1, [[['mat', np.eye(26)]]], None, None)
    with pytest.raises(ValueError):
        maps.residual_map(mat, (8, 8, 8), "cpu")
    # what `fobs_update_device` leaves: device tensors, F_calc as [2, N_h] (Re, Im) planes
    import torch
    F = vx.prop_calc[0][1]
    vx.prop_calc = [['Fobs', torch.from_numpy(np.stack([F.real, F.imag])), torch.tensor(1.7), torch.tensor(0.9)]]
    with pytest.raises(ValueError, match="sync_host"):
        maps.residual_coefficients(vx)
    vx.sync_host()
    assert np.array_equal(maps.residual_coefficients(vx)[0], hkl[1:])


# -- cube files ---------------------------------------------------------------------------------------------------------
def test_cube_layout_line_by_line(tmp_path):
    from ecw_cc_b200 import maps, molint
    mol = molint.Molecule(H2O, "6-31g")
    vals = np.arange(2 * 3 * 7, dtype=float).reshape(2, 3, 7) * 0.25 - 3.0
    origin, axes = np.array([-1.0, -2.0, -3.0]), np.array([[0.5, 0, 0], [0, 0.25, 0], [0.1, 0, 0.2]])
    p = tmp_path / "t.cube"
    maps.write_cube(str(p), mol, origin, axes, vals, comment="test map")
    lines = p.read_text().split("\n")
    assert lines[0] == "test map" and lines[1]
    assert lines[2] == "%5d%12.6f%12.6f%12.6f" % (3, -1.0, -2.0, -3.0)
    assert lines[3] == "    2    0.500000    0.000000    0.000000"
    assert lines[4] == "    3    0.000000    0.250000    0.000000"
    assert lines[5] == "    7    0.100000    0.000000    0.200000"
    xyz = mol.atom_coords()
    assert lines[6] == "    8    8.000000%12.6f%12.6f%12.6f" % tuple(xyz[0])
    assert lines[7].startswith("    1    1.000000") and lines[8].startswith("    1    1.000000")
    body = lines[9:]
    assert body[-1] == "" and len(body) == 2 * 3 * 2 + 1               # two lines per k-row (6 + 1), final newline
    for n, row in enumerate(vals.reshape(-1, 7)):
        assert body[2 * n] == "".join("%13.5E" % x for x in row[:6])
        assert body[2 * n + 1] == "%13.5E" % row[6]
    assert all(len(line) == 13 * 6 for line in body[0:-1:2])


def test_cube_round_trip(tmp_path):
    from ecw_cc_b200 import maps, molint
    mol = molint.Molecule(H2O, "6-31g")
    origin, axes, shape = maps.box(mol, 9, 10, 11)
    pts = (origin + np.stack(np.meshgrid(*[np.arange(n) for n in shape], indexing="ij"), -1) @ axes).reshape(-1, 3)
    rho = molint.density_points(mol, water_hf(), pts).reshape(shape)
    p = str(tmp_path / "rho.cube")
    maps.write_cube(p, mol, origin, axes, rho)
    c = maps.read_cube(p)
    assert c["values"].shape == shape
    assert np.all(np.abs(c["values"] - rho) <= 1e-5 * np.abs(rho))
    assert np.abs(c["origin"] - origin).max() <= 1e-6 and np.abs(c["axes"] - axes).max() <= 1e-6
    assert np.array_equal(c["Z"], [8, 1, 1]) and np.abs(c["coords"] - mol.atom_coords()).max() <= 1e-6


def test_box_is_the_cubegen_box():
    from ecw_cc_b200 import maps, molint
    mol = molint.Molecule(H2O, "6-31g")
    origin, axes, shape = maps.box(mol)
    xyz = mol.atom_coords()
    assert shape == (80, 80, 80)
    assert np.allclose(origin, xyz.min(0) - 3.0, rtol=0, atol=1e-15)
    assert np.allclose(origin + 79 * np.diag(axes), xyz.max(0) + 3.0, rtol=0, atol=1e-13)
    assert np.count_nonzero(axes - np.diag(np.diag(axes))) == 0
    cr = molint.Crystal(MONO)
    ax = maps.cell_axes(cr, (10, 20, 30))
    assert np.allclose(ax * np.array([[10], [20], [30]]), (cr.M * molint.ANGSTROM).T, rtol=0, atol=1e-13)


# -- validation ---------------------------------------------------------------------------------------------------------
def test_input_validation():
    from ecw_cc_b200 import maps, molint
    mol = molint.Molecule(H2O, "6-31g")
    cr = molint.Crystal(MONO, P21C)
    D = np.eye(mol.nao)
    o, a = np.zeros(3), np.eye(3)
    for args in [(np.eye(3), o, a, (2, 2, 2)), (D, o, a, (2, 0, 2)), (D, o, a, (2, 2)), (D, np.zeros(2), a, (2, 2, 2)),
                 (D, o, np.eye(2), (2, 2, 2)), (np.full_like(D, np.nan), o, a, (2, 2, 2)),
                 (D, np.full(3, np.inf), a, (2, 2, 2))]:
        with pytest.raises(ValueError):
            maps.density_grid(mol, *args, device="cpu")
    hkl = np.array([(1, 0, 0), (0, 2, 1)])
    for h, F, shape in [(hkl, np.ones(3), (4, 4, 4)), (hkl + 0.5, np.ones(2), (4, 4, 4)), (hkl[:, :2], np.ones(2), (4, 4, 4)),
                        (hkl, np.array([1.0, np.nan]), (4, 4, 4)), (hkl, np.ones(2), (4, 4, 0)),
                        (hkl, np.ones(2), (4, 4, 513))]:
        with pytest.raises(ValueError):
            maps.fourier_map(cr, h, F, shape, "cpu")
    with pytest.raises(ValueError):
        molint.fourier_map(cr, hkl, np.ones(2), (4, 0, 4))
    with pytest.raises(ValueError):
        maps.box(mol, 1, 10, 10)
    with pytest.raises(ValueError):
        molint.density_points(mol, np.eye(3), np.zeros((2, 3)))
    with pytest.raises(ValueError):
        molint.ao_values(mol, np.zeros((2, 2)))


def test_no_device_raises_ecw_error(built_lib, tmp_path):
    import torch
    from ecw_cc_b200 import EcwError, maps, molint
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    mol = molint.Molecule(H2O, "6-31g")
    cr = molint.Crystal(MONO, P21C)
    with pytest.raises(EcwError):
        maps.density_grid(mol, np.eye(mol.nao), np.zeros(3), np.eye(3), (2, 2, 2), "cpu")
    with pytest.raises(EcwError):
        maps.fourier_map(cr, np.array([(1, 0, 0)]), np.ones(1), (4, 4, 4), "cpu")
    with pytest.raises(EcwError):
        maps.density(mol, str(tmp_path / "x.cube"), np.eye(mol.nao), 4, 4, 4)
    vx = fobs_exp()[0]
    with pytest.raises(EcwError):
        maps.residual_map(vx, (4, 4, 4), "cpu")
    box = (ctypes.c_double * 12)(*([0.0] * 3 + list(np.eye(3).ravel())))
    assert built_lib.ecw_density_grid(None, 1, None, 1, None, box, 1, 1, 1, None, None, None) != 0
    assert built_lib.ecw_fourier_map(None, None, 0, 0.0, 1.0, 1, 1, 1, None, None) != 0
    assert built_lib.ecw_density_grid_workspace_bytes(0, 10) == -1
    assert built_lib.ecw_density_grid_workspace_bytes(10, 100000) == 8 * 2 * 32768 * 10
