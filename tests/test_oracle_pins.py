"""Pin the CPU oracle against the golden vectors produced by the unmodified reference
(oracle/make_golden.py), including its raw-equation second implementation."""
import numpy as np
import pytest

from helpers import load_golden, MODES
from oracle import synth
from oracle.ccsd_np import OracleGCC, soft_threshold
from oracle import refactored_np as R

TOL = 1e-13


def _assert_matches_golden(cc, g):
    """tupdate / lupdate in every mode with both Fock matrices, energy and rdm1 of `cc` against the golden `g`."""
    o, v = int(g["nocc"]), int(g["nvir"])
    t1, t2, l1, l2 = synth.amplitudes(o, v)
    for fname, fsp in (("sym", synth.fsp(o, v)), ("ns", g["fsp_ns"])):
        for tag, alpha, eq in MODES:
            a, b = cc.tupdate(t1, t2, fsp=fsp, alpha=alpha, equation=eq)
            assert np.abs(a - g["T1_%s_%s" % (fname, tag)]).max() < TOL
            assert np.abs(b - g["T2_%s_%s" % (fname, tag)]).max() < TOL
            a, b = cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq)
            assert np.abs(a - g["L1_%s_%s" % (fname, tag)]).max() < TOL
            assert np.abs(b - g["L2_%s_%s" % (fname, tag)]).max() < TOL
        assert abs(cc.energy(t1, t2, fsp) - float(g["E_%s" % fname])) < TOL
    assert np.abs(cc.gamma(t1, t2, l1, l2) - g["gamma"]).max() < TOL


@pytest.mark.parametrize("name", ["ccsd_o4v6.npz", "ccsd_o5v8.npz"])
def test_oracle_matches_golden(name):
    g = load_golden(name)
    o, v = int(g["nocc"]), int(g["nvir"])
    t1, t2, l1, l2 = synth.amplitudes(o, v)
    cc = OracleGCC(synth.SynthEris(o, v))
    _assert_matches_golden(cc, g)
    # identity the reference itself checks (CCSD.py:675-699): factorised == raw equations
    a, b = cc.tupdate(t1, t2, equation=True)
    assert np.abs(a - g["rawT1"]).max() < 1e-12 and np.abs(b - g["rawT2"]).max() < 1e-12
    a, b = cc.lupdate(t1, t2, l1, l2, equation=True)
    assert np.abs(a - g["rawL1"]).max() < 1e-12 and np.abs(b - g["rawL2"]).max() < 1e-12


@pytest.mark.parametrize("name", ["ccsd_o4v6.npz", "ccsd_o5v8.npz"])
def test_refactored_spec_matches_golden(name):
    """The refactored algorithm (what the device executes) equals the reference."""
    g = load_golden(name)
    o, v = int(g["nocc"]), int(g["nvir"])
    er = synth.SynthEris(o, v)
    E = R.DeviceErisSpec(er)
    t1, t2, l1, l2 = synth.amplitudes(o, v)
    for fname, fsp in (("sym", synth.fsp(o, v)), ("ns", g["fsp_ns"])):
        for tag, alpha, eq in MODES:
            a, b = R.tupdate(E, er.fock, t1, t2, fsp=fsp, alpha=alpha, equation=eq)
            assert np.abs(a - g["T1_%s_%s" % (fname, tag)]).max() < TOL
            assert np.abs(b - g["T2_%s_%s" % (fname, tag)]).max() < TOL
            a, b = R.lupdate(E, er.fock, t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq)
            assert np.abs(a - g["L1_%s_%s" % (fname, tag)]).max() < TOL
            assert np.abs(b - g["L2_%s_%s" % (fname, tag)]).max() < TOL
    assert np.abs(R.gamma(t1, t2, l1, l2) - g["gamma"]).max() < TOL


def test_quirks():
    """Q1: v<0 behaves like v==0; Q2: lupdate(alpha=0) != lupdate(alpha=None)."""
    e = np.array([0.5, -0.5, 0.05, 0.5, -0.5, 0.05, 0.5, -0.05])
    v = np.array([1.0, 1.0, 1.0, -1.0, -1.0, -1.0, 0.0, 0.0])
    w = soft_threshold(e, v, 0.1)
    assert np.allclose(w, [0.6, -0.4, 0.15, 0.4, -0.4, 0.0, 0.4, 0.0])
    with pytest.raises(ValueError):
        soft_threshold(np.zeros(3), np.zeros(4), 0.1)
    o, v_ = 4, 6
    er = synth.SynthEris(o, v_)
    t1, t2, l1, l2 = synth.amplitudes(o, v_)
    cc = OracleGCC(er)
    a0 = cc.lupdate(t1, t2, l1, l2, alpha=0.0)
    an = cc.lupdate(t1, t2, l1, l2, alpha=None)
    assert np.abs(a0[1] - an[1]).max() > 1e-6
    b0 = cc.tupdate(t1, t2, alpha=0.0)
    bn = cc.tupdate(t1, t2, alpha=None)
    assert np.abs(b0[1] - bn[1]).max() < 1e-14
    g = cc.gamma(t1, t2, l1, l2)
    assert abs(np.trace(g) - o) < 1e-12 and np.abs(g - g.T).max() < 1e-15


@pytest.mark.parametrize("name", ["ccsd_o4v6.npz", "ccsd_o5v8.npz"])
def test_faithful_oracle_matches_golden(name):
    """The oracle with the reference's own einsum routing (`faithful=True`, what bench.py's CPU leg times)."""
    g = load_golden(name)
    _assert_matches_golden(OracleGCC(synth.SynthEris(int(g["nocc"]), int(g["nvir"])), faithful=True), g)
