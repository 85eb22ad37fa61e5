"""Amplitude target ('Fobs') on the GPU: `ecw_ft_aopair_cryst` against `molint.ft_aopair_cryst`, the device potential
`ecw_vexp_sfobs` against the host branch of `exp_pot.Exp.Vexp_update`, and `Solver_CCSD` through the device route
against the host route, under every GEMM engine."""
import numpy as np
import pytest

from helpers import load_golden
from oracle.make_golden_c2h2 import C2H2
from oracle.make_golden_h2o import H2O
from oracle.make_golden_solver import target_rdm1

pytestmark = pytest.mark.gpu
TOL = 1e-10
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


def aniso_adp(natom, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(natom):
        x = 0.03 * rng.standard_normal((3, 3))
        out.append(0.01 * np.eye(3) + x @ x.T)
    return out


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


@pytest.mark.parametrize("group", sorted(GROUPS))
@pytest.mark.parametrize("atoms,basis", [(H2O, "6-31++g**"), (C2H2, "cc-pvdz")])
def test_ft_aopair_cryst_kernel_matches_numpy(built_lib, atoms, basis, group):
    import torch
    from ecw_cc_b200 import exp_pot, molint
    mol = molint.Molecule(atoms, basis)
    ops, cell = GROUPS[group]
    cr = molint.Crystal(cell, ops, aniso_adp(len(atoms), 2))
    hkl, s_top = reflections(cr, 200, 1.2, 1)
    assert s_top > 1.15
    want = molint.ft_aopair_cryst(mol, cr, hkl)
    dev = torch.device("cuda", 0)
    got = exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
    again = exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
    assert torch.equal(got, again)                             # fixed summation order: identical bits
    got = got.cpu().numpy()
    err = max(np.abs(got[0] - want.real).max(), np.abs(got[1] - want.imag).max())
    assert err <= 1e-12 * cr.nsym, err


def test_identity_crystal_matches_ft_aopair_planes(built_lib):
    import torch
    from ecw_cc_b200 import exp_pot, molint
    mol = molint.Molecule(C2H2, "cc-pvdz")
    cr = molint.Crystal((5.0, 6.0, 7.0))
    hkl, _ = reflections(cr, 150, 1.0, 3)
    dev = torch.device("cuda", 0)
    a = exp_pot.ft_aopair_device(mol, cr.G(hkl), dev)
    b = exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
    assert (a - b).abs().max().item() <= 1e-14


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


def test_device_potential_matches_host_branch(built_lib):
    import torch
    from ecw_cc_b200 import exp_pot
    mol, er, _ = water()
    F_obs, sigma, hkl, cr = fobs_data(mol, er, 60, 2)
    rng = np.random.default_rng(5)
    rdm1 = target_rdm1(10, 16) + 0.003 * rng.standard_normal((26, 26))      # not symmetric: the CC rdm1 is not
    fock = er.fock + 0.01 * rng.standard_normal((26, 26))
    hf = np.diag(er.mo_occ)
    probe = exp_pot.Exp(0.0, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, er.mo_coeff_g)
    probe.Vexp_update(hf, hf, (0, 0))
    F_hf = probe.prop_calc[0][1]
    close = lambda x, y: abs(x - y) <= 1e-12 * max(1.0, abs(y))
    cases = [(extra, hf_prop, rdm1) for extra in ([], [1.7]) for hf_prop in (False, [[F_hf]])]   # refined / fixed k
    cases.append(([], False, hf))          # the HF density: reflections its point symmetry extinguishes (|F| cusp)
    for extra, hf_prop, rdm1 in cases:
        tgt = ['Fobs', F_obs, sigma, hkl, cr] + extra
        host = exp_pot.Exp(0.3, [[tgt]], mol, er.mo_coeff_g, HF_prop=hf_prop)
        devp = exp_pot.Exp(0.3, [[tgt]], mol, er.mo_coeff_g, HF_prop=hf_prop)
        d_h, vmax_h = host.Vexp_update(rdm1, rdm1, (0, 0), L=0.7)
        d_d, vmax_d, fsp = devp.fobs_update_device(torch.from_numpy(rdm1).cuda(), torch.from_numpy(fock).cuda(),
                                                   L=0.7)
        assert close(d_d, d_h) and close(vmax_d, vmax_h), (d_d, d_h, vmax_d, vmax_h)
        assert np.abs(fsp.cpu().numpy() - (fock - host.Vexp[0, 0])).max() <= 1e-12
        devp.sync_host()
        assert isinstance(devp.Vexp[0, 0], np.ndarray) and np.abs(devp.Vexp[0, 0] - host.Vexp[0, 0]).max() <= 1e-12
        name, F_c, k, chi2 = devp.prop_calc[0]
        assert name == 'Fobs' and np.abs(F_c - host.prop_calc[0][1]).max() <= 1e-12
        assert isinstance(k, float) and isinstance(chi2, float)
        assert close(k, host.prop_calc[0][2]) and close(chi2, host.prop_calc[0][3])
        if extra:
            assert k == 1.7


def test_solver_device_route_matches_host_route(built_lib, engine):
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import exp_pot

    class HostRouteExp(exp_pot.Exp):                           # the same target, forced onto the host route
        def device_fobs_ready(self):
            return False

    mol, er, g = water()
    F_obs, sigma, hkl, cr = fobs_data(mol, er, 40, 4, s_max=0.35)
    chi2 = []
    for L in (0.005, 0.01, 0.02):                               # L = 0.05 diverges for these data
        runs = []
        for make in (exp_pot.Exp, HostRouteExp):
            vx = make(L, [[['Fobs', F_obs, sigma, hkl, cr]]], mol, er.mo_coeff_g)
            out = ecw.Solver_CCSD(ecw.GCC(er), vx, conv="tl", conv_thres=float(g["conv_thres"]), maxiter=60).SCF(L)
            runs.append((out, vx))
        (a, va), (b, vb) = runs
        assert hasattr(va, "_fobs_dev") and not hasattr(vb, "_fobs_dev")   # the two routes were taken
        assert a[0] == b[0] and a[0].startswith("Convergence reached") and len(a[1]) == len(b[1]), (a[0], b[0])
        assert np.abs(a[1] - b[1]).max() < TOL and np.abs(a[2] - b[2]).max() < TOL
        assert np.abs(a[4] - b[4]).max() < TOL
        for x, y in zip(a[5], b[5]):
            assert np.abs(x - y).max() < TOL
        assert np.abs(va.prop_calc[0][1] - vb.prop_calc[0][1]).max() < TOL
        assert abs(va.prop_calc[0][2] - vb.prop_calc[0][2]) < TOL and abs(va.prop_calc[0][3] - vb.prop_calc[0][3]) < TOL
        chi2.append(va.prop_calc[0][3])
    assert chi2[0] > chi2[1] > chi2[2], chi2
