"""Density maps on the GPU: `ecw_density_grid` against `molint.density_points`, `ecw_fourier_map` against
`molint.fourier_map` and Parseval, the two kernels against each other through the structure-factor convention (H2 in a
P1 cell), and the maps of a fitted 'Fobs' state from `Solver_CCSD`."""
import numpy as np
import pytest

from helpers import load_golden
from oracle.make_golden_c2h2 import C2H2
from oracle.make_golden_h2o import H2O
from oracle.make_golden_solver import target_rdm1

pytestmark = pytest.mark.gpu
P21C = ['x,y,z', '-x,y+1/2,-z+1/2', '-x,-y,-z', 'x,-y+1/2,z+1/2']
MONO = (7.0, 8.0, 9.0, 90.0, 104.0, 90.0)
GROUPS = {                                                      # operations and a cell of their system
    "P-1": (['x,y,z', '-x,-y,-z'], (5.1, 6.2, 7.3, 78.0, 95.0, 107.0)),
    "P2_1/c": (P21C, (5.5, 6.5, 7.5, 90.0, 103.0, 90.0)),
    "P2_12_12_1": (['x,y,z', '-x+1/2,-y,z+1/2', '-x,y+1/2,-z+1/2', 'x+1/2,-y+1/2,-z'], (5.0, 6.0, 7.0)),
}


def water():
    from ecw_cc_b200 import molint
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    return mol, molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol))), g


def reflections(crystal, n, s_max, seed):
    """(0, 0, 0), the reflection of largest sin(theta)/lambda <= s_max, and n - 2 random others below s_max."""
    from ecw_cc_b200 import molint
    r = [int(np.ceil(2 * s_max * np.linalg.norm(crystal.M[:, d]))) + 1 for d in range(3)]
    hkl = np.array([(h, k, l) for h in range(-r[0], r[0] + 1) for k in range(-r[1], r[1] + 1)
                    for l in range(-r[2], r[2] + 1)])
    s = np.linalg.norm(crystal.G(hkl), axis=1) * molint.ANGSTROM / (4 * np.pi)
    ok = np.where((s <= s_max) & (s > 0))[0]
    top = ok[np.argmax(s[ok])]
    rest = np.random.default_rng(seed).choice(np.setdiff1d(ok, [top]), n - 2, replace=False)
    return np.concatenate([[[0, 0, 0]], hkl[[top]], hkl[rest]]), s[top]


def fobs_data(mol, er, n, seed, s_max=0.6):
    """Amplitudes of a perturbed density in P2_1/c with ADPs (systematic absences left out), random sigma."""
    from ecw_cc_b200 import exp_pot, molint
    cr = molint.Crystal(MONO, P21C, [0.02, 0.03, 0.03])
    hkl, _ = reflections(cr, 3 * n, s_max, seed)
    probe = exp_pot.Exp(0.0, [[['Fobs', np.ones(len(hkl)), None, hkl, cr]]], mol, er.mo_coeff_g)
    probe.Vexp_update(target_rdm1(10, 16), target_rdm1(10, 16), (0, 0))
    a = np.abs(probe.prop_calc[0][1])
    keep = np.where(a > 1e-6 * a.max())[0][:n]
    rng = np.random.default_rng(seed)
    a, hkl = a[keep], hkl[keep]
    sigma = 0.05 * a.mean() * (0.5 + rng.uniform(size=len(a)))
    return np.abs(2.0 * a + 0.3 * sigma * rng.standard_normal(len(a))), sigma, hkl, cr


def grid_points(origin, axes, shape):
    """origin + i a1 + j a2 + k a3 in the order of the device kernel, [n1 n2 n3, 3]."""
    i, j, k = (x.reshape(-1, 1).astype(float) for x in np.meshgrid(*[np.arange(n) for n in shape], indexing="ij"))
    return ((origin + i * axes[0]) + j * axes[1]) + k * axes[2]


# -- the density kernel -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("atoms,basis", [(H2O, "6-31++g**"), (C2H2, "cc-pvdz")])
def test_density_kernel_matches_host(built_lib, atoms, basis):
    import torch
    from ecw_cc_b200 import maps, molint
    mol = molint.Molecule(atoms, basis)
    assert mol.lmax == 2
    rng = np.random.default_rng(1)
    X = rng.standard_normal((mol.nao, mol.nao))
    D = X @ X.T / mol.nao + 0.05 * rng.standard_normal((mol.nao, mol.nao))      # not symmetric
    dev = torch.device("cuda", 0)
    origin, axes, _ = maps.box(mol, 10, 10, 10, margin=2.0)
    axes = axes + np.array([[0.0, 0.03, -0.02], [0.05, 0.0, 0.01], [-0.04, 0.02, 0.0]])   # not cubic, not orthogonal
    for shape in [(1, 1, 1), (3, 5, 7), (9, 1, 4), (33, 32, 32)]:           # the last is larger than one chunk
        got = maps.density_grid(mol, D, origin, axes, shape, dev)
        again = maps.density_grid(mol, D, origin, axes, shape, dev)
        assert torch.equal(got, again)
        want = molint.density_points(mol, D, grid_points(origin, axes, shape)).reshape(shape)
        err = np.abs(got.cpu().numpy() - want) / np.maximum(1.0, np.abs(want))
        assert err.max() <= 1e-12, (shape, err.max())


def test_density_cube_writer(built_lib, tmp_path):
    from ecw_cc_b200 import maps, molint
    mol, er, g = water()
    C = g["mo_coeff"]
    D = 2 * C[:, :5] @ C[:, :5].T
    rho = maps.density(mol, str(tmp_path / "w.cube"), D, 12, 11, 10)
    c = maps.read_cube(str(tmp_path / "w.cube"))
    origin, axes, shape = maps.box(mol, 12, 11, 10)
    want = molint.density_points(mol, D, grid_points(origin, axes, shape)).reshape(shape)
    assert np.abs(rho - want).max() <= 1e-12 * np.abs(want).max()
    assert np.all(np.abs(c["values"] - rho) <= 1e-5 * np.abs(rho))


# -- the Fourier kernel -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("group", sorted(GROUPS))
def test_fourier_kernel_matches_host(built_lib, group):
    import torch
    from ecw_cc_b200 import maps, molint
    ops, cell = GROUPS[group]
    cr0 = molint.Crystal(cell)
    mol = molint.Molecule([(s, tuple(np.asarray(r) + cr0.cartesian([0.21, 0.13, 0.32]))) for s, r in H2O], "6-31g*")
    cr = molint.Crystal(cell, ops, [0.02, 0.03, 0.03])
    hkl, _ = reflections(cr, 150, 1.0, 2)
    rng = np.random.default_rng(3)
    X = rng.standard_normal((mol.nao, mol.nao))
    F = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, hkl), X + X.T + 5 * np.eye(mol.nao))
    hh, Fh, F000 = cr.expand(hkl, F)
    bound = (abs(F000) + 2 * np.abs(Fh).sum()) / cr.volume_bohr3
    dev = torch.device("cuda", 0)
    for shape in [(9, 10, 11), (16, 15, 8), (1, 1, 1)]:
        got = maps.fourier_map(cr, hkl, F, shape, dev)
        again = maps.fourier_map(cr, hkl, F, shape, dev)
        assert torch.equal(got, again)
        want = molint.fourier_map(cr, hkl, F, shape)
        assert np.abs(got.cpu().numpy() - want).max() <= 1e-12 * bound, shape
    # Parseval on the device output: exact when n_d > 2 max |h_d|
    hkl, _ = reflections(cr, 60, 0.4, 4)
    F = np.einsum('hij,ij->h', molint.ft_aopair_cryst(mol, cr, hkl), X + X.T + 5 * np.eye(mol.nao))
    hh, Fh, F000 = cr.expand(hkl, F)
    shape = tuple(2 * int(np.abs(hh[:, d]).max()) + 1 + d for d in range(3))
    rho = maps.fourier_map(cr, hkl, F, shape, dev).cpu().numpy()
    V = cr.volume_bohr3
    ms = (F000 ** 2 + 2 * np.sum(np.abs(Fh) ** 2)) / V ** 2
    assert abs(np.mean(rho ** 2) - ms) <= 1e-12 * ms
    assert abs(np.mean(rho) - F000 / V) <= 1e-12 * abs(F000) / V


def test_real_space_matches_reciprocal_space(built_lib):
    """H2/cc-pVDZ (RHF) in a 6 A cubic P1 cell, no ADPs.  The synthesis of F_calc (device planes of
    `ft_aopair_cryst_device`) over every reflection with exp(-|G|^2 / 4 p_max) >= 1e-10 (p_max = 26 bohr^-2, twice the
    steepest H exponent: |G| <= 49.1 bohr^-1, 1.4e6 reflections in the half set) equals the lattice sum of
    `density_grid` over the 27 nearest images.  The omitted reflections carry about 1e-8 e/bohr^3 (the tail of the
    steepest primitive products), the images beyond the first shell less than 1e-20: tolerance 1e-7 e/bohr^3, at grid
    points more than 0.5 bohr from a nucleus."""
    import torch
    from ecw_cc_b200 import exp_pot, maps, molint
    a = 6.0
    cr = molint.Crystal((a, a, a))
    mol = molint.Molecule([("H", (2.63, 3.1, 2.9)), ("H", (3.37, 3.0, 3.05))], "cc-pvdz")
    _, _, C, _ = molint.rhf(mol)
    D = 2 * C[:, :1] @ C[:, :1].T
    g_max = np.sqrt(4 * 26.0 * np.log(1e10))
    r = int(np.ceil(g_max * a * molint.ANGSTROM / (2 * np.pi)))
    h, k, l = (x.ravel() for x in np.meshgrid(*[np.arange(-r, r + 1)] * 3, indexing="ij"))
    hkl = np.stack([h, k, l], axis=1)
    half = (h > 0) | ((h == 0) & (k > 0)) | ((h == 0) & (k == 0) & (l > 0))
    hkl = hkl[half & (np.linalg.norm(cr.G(hkl), axis=1) <= g_max)]
    assert len(hkl) > 1.3e6
    dev = torch.device("cuda", 0)
    Dt = torch.from_numpy(D.ravel()).to(dev)
    F = np.empty(len(hkl), dtype=np.complex128)
    for c0 in range(0, len(hkl), 200000):
        planes = exp_pot.ft_aopair_cryst_device(mol, cr, hkl[c0:c0 + 200000], dev)
        f = (planes.reshape(2, -1, mol.nao ** 2) @ Dt).cpu().numpy()
        F[c0:c0 + 200000] = f[0] + 1j * f[1]
        del planes
    F000 = float(np.sum(D * mol.intor_symmetric('int1e_ovlp')))
    shape = (12, 13, 14)
    recip = maps.synthesis(hkl, F, F000, cr.volume_bohr3, shape, dev).cpu().numpy()
    axes = maps.cell_axes(cr, shape)
    M = cr.M * molint.ANGSTROM
    real = np.zeros(shape)
    for n in np.ndindex(3, 3, 3):
        real += maps.density_grid(mol, D, M @ (np.array(n) - 1), axes, shape, dev).cpu().numpy()
    pts = grid_points(np.zeros(3), axes, shape)
    d = pts[:, None, :] - mol.atom_coords()[None]
    frac = d @ np.linalg.inv(M).T
    dist = np.linalg.norm((frac - np.round(frac)) @ M.T, axis=2).min(1).reshape(shape)
    off = dist > 0.5
    assert off.sum() > 0.9 * off.size and real.max() > 0.1
    assert np.abs(recip - real)[off].max() <= 1e-7, np.abs(recip - real)[off].max()


# -- maps of a fitted state ---------------------------------------------------------------------------------------------
def test_fitted_state_maps(built_lib):
    """`Solver_CCSD` with one 'Fobs' target on the device route: the residual map equals the host synthesis of the same
    coefficients, its RMS falls as chi^2 falls, and the density cube of the fitted state integrates to tr(D S)."""
    import torch
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import exp_pot, maps, molint, utilities
    mol, er, g = water()
    F_obs, sigma, hkl, cr = fobs_data(mol, er, 40, 4, s_max=0.35)
    dev = torch.device("cuda", 0)
    shape = (14, 16, 18)
    S = mol.intor_symmetric('int1e_ovlp')
    C = er.mo_coeff_g
    D_hf = utilities.convert_g_to_ru_rdm1(C @ np.diag(er.mo_occ) @ C.T)[0]
    origin, axes, fine = maps.box(mol, 300, 300, 300, margin=6.0)
    h3 = abs(np.linalg.det(axes))
    n_hf = h3 * maps.density_grid(mol, D_hf, origin, axes, fine, dev).sum().item()
    chi2, rms = [], []
    for L in (0.005, 0.02):
        vx = exp_pot.Exp(L, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, C)
        out = ecw.Solver_CCSD(ecw.GCC(er), vx, conv="tl", conv_thres=float(g["conv_thres"]), maxiter=60).SCF(L)
        assert hasattr(vx, "_fobs_dev") and out[0].startswith("Convergence reached")
        got = maps.residual_map(vx, shape, dev).cpu().numpy()            # the solver leaves host copies
        h, c, _ = maps.residual_coefficients(vx)
        want = molint.fourier_map(cr, h, c, shape)
        hh, ch, _ = cr.expand(h, c)
        assert np.abs(got - want).max() <= 1e-12 * 2 * np.abs(ch).sum() / cr.volume_bohr3
        chi2.append(vx.prop_calc[0][3])
        rms.append(np.sqrt(np.mean(got ** 2)))
        # the density of the fitted state on a fine box (spacing 0.05 bohr): the O 1s primitives (exponents up to 5484
        # bohr^-2) are not resolved at that spacing (about 1e-4 of the count for the HF density); the deformation
        # density has almost no core part and integrates to tr((D - D_HF) S) to about 1e-6 electrons
        D = utilities.convert_g_to_ru_rdm1(C @ out[4] @ C.T)[0]
        n = h3 * maps.density_grid(mol, D, origin, axes, fine, dev).sum().item()
        assert abs(n - np.sum(D * S)) <= 2e-3 * np.sum(D * S), (n, np.sum(D * S))
        assert abs((n - n_hf) - np.sum((D - D_hf) * S)) <= 1e-5, (n - n_hf, np.sum((D - D_hf) * S))
    assert chi2[1] < chi2[0] and rms[1] < rms[0], (chi2, rms)
    # one device evaluation leaves device tensors in prop_calc: the map asks for sync_host()
    rdm1 = torch.from_numpy(out[4]).to(dev)
    vx.fobs_update_device(rdm1, torch.from_numpy(er.fock).to(dev))
    with pytest.raises(ValueError, match="sync_host"):
        maps.residual_map(vx, shape, dev)
    vx.sync_host()
    assert np.abs(maps.residual_map(vx, shape, dev).cpu().numpy() - got).max() <= 1e-12 * np.abs(got).max()
