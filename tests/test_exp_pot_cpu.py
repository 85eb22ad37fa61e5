"""`ecw_cc_b200.exp_pot.Exp` for every target kind it provides ('mat' GS/ES, 'Ek', 'v1e', 'dip', 'DEk', 'trdip') against
the UNMODIFIED reference class on the same H2O/6-31G inputs (tests/golden/exp_pot_h2o.npz, oracle/make_golden_exp.py);
plus the dipole integrals of the PySCF-free source."""
import numpy as np
import pytest

from helpers import load_golden
from oracle.make_golden_exp import CALLS, run
from oracle.make_golden_h2o import H2O


@pytest.fixture(scope="module")
def water():
    from ecw_cc_b200 import molint
    g = load_golden("h2o_631g.npz")
    mol = molint.Molecule(H2O, "6-31g")
    return mol, molint.geris(mol, (float(g["EHF"]), g["mo_energy"], g["mo_coeff"], molint.integrals(mol)))


def test_dipole_integrals(water):
    from ecw_cc_b200 import molint, utilities
    mol, er = water
    S = mol.intor_symmetric("int1e_ovlp")
    d0 = molint.dipole_integrals(mol)
    c = np.array([0.3, -0.2, 0.5])
    with mol.with_common_orig(c):
        dc = mol.intor_symmetric("int1e_r", comp=3)
    assert np.abs(dc - (d0 - c[:, None, None] * S[None])).max() < 1e-14      # origin shift
    assert np.abs(d0 - d0.transpose(0, 2, 1)).max() < 1e-14
    hf = np.diag(er.mo_occ)
    kw = dict(aobasis=False, mo_coeff=er.mo_coeff_g)
    # RHF/6-31G water: dipole 2.63 D along the C2 axis, virial ratio ~ 1, trace of the rdm1 = 10 electrons
    mu = -utilities.dipole(mol, hf, **kw) + (mol.Z[:, None] * (mol.R - (mol.Z @ mol.R) / mol.Z.sum())).sum(0)
    assert abs(np.linalg.norm(mu) * 2.541746 - 2.632) < 2e-3 and abs(mu[0]) < 1e-10 and abs(mu[1]) < 1e-10
    ek, vne = utilities.Ekin(mol, hf, **kw), utilities.v1e(mol, hf, **kw)
    assert abs(ek / -er.EHF - 1) < 2e-3 and -200 < vne < -198


def test_exp_matches_reference_for_every_target(water):
    from ecw_cc_b200 import exp_pot, utilities
    mol, er = water
    g = load_golden("exp_pot_h2o.npz")
    out = run(exp_pot.Exp, mol, er.mo_coeff_g, utilities)
    assert sorted(out) == sorted(g)
    for k in g:
        want, got = np.asarray(g[k], dtype=float), np.asarray(out[k], dtype=float)
        assert want.shape == got.shape, k
        assert np.abs(want - got).max() <= 1e-11 * max(1.0, np.abs(want).max()), k
    assert len(CALLS) == 7 and float(g["w_11_Delta"]) > 0


def test_errors():
    from ecw_cc_b200 import exp_pot
    with pytest.raises(NotImplementedError):
        exp_pot.Exp(0.1, [[['F', [1.0], [[1, 0, 0]], [10., 10., 10.]]]], None, None)
    with pytest.raises(ValueError):
        exp_pot.Exp(0.1, [[['Ek', 76.0]]], None, None)
    with pytest.raises(SyntaxError):
        exp_pot.Exp([[0.1], [0.2]], [[['mat', np.eye(4)]]], None, None)
