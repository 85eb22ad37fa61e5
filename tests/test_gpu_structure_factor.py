"""Structure-factor ('F') target on the GPU: `ecw_ft_aopair` against `molint.ft_aopair`, the device potential
`ecw_vexp_sf` against the host branch of `exp_pot.Exp.Vexp_update`, and `Solver_CCSD` through the device route against
the host route, under every GEMM engine."""
import numpy as np
import pytest

from helpers import load_golden
from oracle.make_golden_c2h2 import C2H2
from oracle.make_golden_h2o import H2O
from oracle.make_golden_solver import target_rdm1

pytestmark = pytest.mark.gpu
TOL = 1e-10
CELL = (8.0, 9.0, 10.0)


def water():
    from ecw_cc_b200 import molint
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    return mol, molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol))), g


def reflections(cell, n, s_max, seed):
    """(0, 0, 0), the reflection of largest sin(theta)/lambda <= s_max, and n - 2 random others below s_max."""
    a, b, c = cell
    r = [int(np.ceil(2 * s_max * x)) for x in cell]
    hkl = np.array([(h, k, l) for h in range(-r[0], r[0] + 1) for k in range(-r[1], r[1] + 1)
                    for l in range(-r[2], r[2] + 1)])
    s = 0.5 * np.sqrt((hkl[:, 0] / a) ** 2 + (hkl[:, 1] / b) ** 2 + (hkl[:, 2] / c) ** 2)
    ok = np.where((s <= s_max) & (s > 0))[0]
    top = ok[np.argmax(s[ok])]
    rest = np.random.default_rng(seed).choice(np.setdiff1d(ok, [top]), n - 2, replace=False)
    return np.concatenate([[[0, 0, 0]], hkl[[top]], hkl[rest]]), s[top]


@pytest.mark.parametrize("atoms,basis", [(H2O, "6-31++g**"), (C2H2, "cc-pvdz")])
def test_ft_aopair_kernel_matches_numpy(built_lib, atoms, basis):
    import torch
    from ecw_cc_b200 import exp_pot, molint
    mol = molint.Molecule(atoms, basis)
    cell = (5.0, 6.0, 7.0)
    hkl, s_top = reflections(cell, 300, 1.2, 1)
    assert s_top > 1.15
    G = 2 * np.pi * hkl / np.array(cell) / molint.ANGSTROM
    want = molint.ft_aopair(mol, G)
    dev = torch.device("cuda", 0)
    got = exp_pot.ft_aopair_device(mol, G, dev)
    again = exp_pot.ft_aopair_device(mol, G, dev)
    assert torch.equal(got, again)                             # fixed summation order: identical bits
    got = got.cpu().numpy()
    err = max(np.abs(got[0] - want.real).max(), np.abs(got[1] - want.imag).max())
    assert err <= 1e-12, err


def test_device_potential_matches_host_branch(built_lib):
    import torch
    from ecw_cc_b200 import exp_pot
    mol, er, _ = water()
    hkl, _ = reflections(CELL, 60, 0.6, 2)
    rng = np.random.default_rng(5)
    F_exp = (2 + rng.standard_normal(len(hkl))) * np.exp(1j * rng.uniform(0, 2 * np.pi, len(hkl)))
    rdm1 = target_rdm1(10, 16) + 0.003 * rng.standard_normal((26, 26))      # not symmetric: the CC rdm1 is not
    fock = er.fock + 0.01 * rng.standard_normal((26, 26))
    hf = np.diag(er.mo_occ)
    probe = exp_pot.Exp(0.0, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g)
    probe.Vexp_update(hf, hf, (0, 0))
    F_hf = probe.prop_calc[0][1]
    for hf_prop in (False, [[F_hf]]):
        host = exp_pot.Exp(0.3, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g, HF_prop=hf_prop)
        devp = exp_pot.Exp(0.3, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g, HF_prop=hf_prop)
        d_h, vmax_h = host.Vexp_update(rdm1, rdm1, (0, 0), L=0.7)
        d_d, vmax_d, fsp = devp.sf_update_device(torch.from_numpy(rdm1).cuda(), torch.from_numpy(fock).cuda(), L=0.7)
        assert abs(d_h - d_d) <= 1e-12 and abs(vmax_h - vmax_d) <= 1e-12
        assert np.abs(fsp.cpu().numpy() - (fock - host.Vexp[0, 0])).max() <= 1e-12
        devp.sync_host()
        assert isinstance(devp.Vexp[0, 0], np.ndarray) and np.abs(devp.Vexp[0, 0] - host.Vexp[0, 0]).max() <= 1e-12
        assert devp.prop_calc[0][0] == 'F' and np.abs(devp.prop_calc[0][1] - host.prop_calc[0][1]).max() <= 1e-12


def test_solver_device_route_matches_host_route(built_lib, engine):
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import exp_pot

    class HostRouteExp(exp_pot.Exp):                           # the same target, forced onto the host route
        def device_sf_ready(self):
            return False

    mol, er, g = water()
    hkl = np.array([(h, k, l) for h in range(0, 3) for k in range(-2, 3) for l in range(-2, 3)
                    if (h, k, l) != (0, 0, 0)][:40])
    probe = exp_pot.Exp(0.0, [[['F', np.zeros(len(hkl)), hkl, CELL]]], mol, er.mo_coeff_g)
    probe.Vexp_update(target_rdm1(10, 16), target_rdm1(10, 16), (0, 0))
    F_exp = probe.prop_calc[0][1]
    resid = []
    for L in (0.01, 0.02, 0.05):
        runs = []
        for make in (exp_pot.Exp, HostRouteExp):
            vx = make(L, [[['F', F_exp, hkl, CELL]]], mol, er.mo_coeff_g)
            out = ecw.Solver_CCSD(ecw.GCC(er), vx, conv="tl", conv_thres=float(g["conv_thres"]), maxiter=60).SCF(L)
            runs.append((out, vx))
        (a, va), (b, vb) = runs
        assert hasattr(va, "_sf_dev") and not hasattr(vb, "_sf_dev")       # the two routes were taken
        assert a[0] == b[0] and a[0].startswith("Convergence reached") and len(a[1]) == len(b[1]), (a[0], b[0])
        assert np.abs(a[1] - b[1]).max() < TOL and np.abs(a[2] - b[2]).max() < TOL
        assert np.abs(a[4] - b[4]).max() < TOL
        for x, y in zip(a[5], b[5]):
            assert np.abs(x - y).max() < TOL
        assert np.abs(va.prop_calc[0][1] - vb.prop_calc[0][1]).max() < TOL
        resid.append(np.sum(np.abs(F_exp - va.prop_calc[0][1])))
    assert resid[0] > resid[1] > resid[2], resid
