"""Pins of the solver-loop restatement (oracle/solver_np.py) and of the converged-state fixtures against
tests/golden/solver_ccsd_*.npz (made by oracle/make_golden_solver.py from the unmodified reference solver + CCSD.GCC +
exp_pot.Exp)."""
import numpy as np
import pytest

from helpers import load_golden
from oracle import synth
from oracle.ccsd_np import OracleGCC
from oracle.make_golden_solver import CASES, target_rdm1
from oracle.solver_np import ExpMat, scf_loop


def test_expmat_matches_product_exp_pot():
    """The oracle's 'mat' target against the product's ecw_cc_b200.exp_pot.Exp (same constructor as the reference's
    exp_pot.Exp, pinned to the reference's outputs by tests/test_exp_pot_cpu.py)."""
    import ecw_cc_b200.exp_pot as exp_pot
    rng = np.random.default_rng(3)
    n = 10
    target = rng.standard_normal((n, n))
    for L in (0.0, 0.05, 3.0):
        ref, mine = exp_pot.Exp(L, [[["mat", target]]], None, None), ExpMat(L, target)
        rdm1 = rng.standard_normal((n, n))
        a, b = ref.Vexp_update(rdm1, rdm1, (0, 0), L=L), mine.Vexp_update(rdm1, rdm1, (0, 0), L=L)
        assert a == b and np.array_equal(ref.Vexp[0, 0], mine.Vexp[0, 0])
        # with the Hartree-Fock property given (Delta is then relative to target - HF), and with L changed by the call
        for hf in (False, [[0.5 * target]]):
            r2, m2 = exp_pot.Exp(L, [[["mat", target]]], None, None, HF_prop=hf), ExpMat(L, target)
            scale = np.sum(abs(target)) / np.sum(abs(target - hf[0][0])) if hf else 1.0
            for Lc in (None, 2 * L + 0.1):
                (d, vmax), (d0, vmax0) = r2.Vexp_update(rdm1, rdm1, (0, 0), L=Lc), m2.Vexp_update(rdm1, rdm1, (0, 0), L=Lc)
                assert vmax == vmax0 and (d == d0 if not hf else abs(d - d0 * scale) <= 1e-15 * d)
                assert np.array_equal(r2.Vexp[0, 0], m2.Vexp[0, 0]) and r2.L == [[L]]


@pytest.mark.parametrize("name", ["solver_ccsd_o4v6.npz", "solver_ccsd_o8v16.npz"])
def test_oracle_solver_loop_reproduces_reference_runs(name):
    g = load_golden(name)
    o, v = int(g["nocc"]), int(g["nvir"])
    if o * v > 200:
        pytest.skip("kept for the GPU test; the numpy loop at this size takes minutes")
    er = synth.SynthEris(o, v)
    for tag, L, alpha, maxiter in CASES:
        out = scf_loop(OracleGCC(er), ExpMat(L, target_rdm1(o, v)), L, alpha=alpha, conv_thres=float(g["conv_thres"]),
                       maxiter=maxiter)
        assert out[0] == str(g[tag + "_text"])
        assert np.abs(out[1] - g[tag + "_Ep"]).max() < 1e-12
        assert np.abs(out[2] - g[tag + "_Delta"]).max() < 1e-12
        assert np.allclose(out[3], g[tag + "_conv"], rtol=1e-6, atol=1e-13)
        assert np.abs(out[4] - g[tag + "_rdm1"]).max() < 1e-12
        for k, a in zip(("ts", "ls", "td", "ld"), out[5]):
            assert np.abs(a - g[tag + "_" + k]).max() < 1e-12, (tag, k)
