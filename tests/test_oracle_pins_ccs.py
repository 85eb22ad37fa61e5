"""Pin the CCS oracle (oracle/ccs_np.py) to reference-generated vectors."""
import types

import numpy as np
import pytest

from helpers import load_golden
from oracle import synth, ccs_np
from oracle.make_golden import ccs_calls, ccs_inputs

TOL = 1e-13
_MOD = types.SimpleNamespace(gamma_CCS=ccs_np.gamma_CCS, gamma_unsym_CCS=ccs_np.gamma_unsym_CCS,
                             gamma_es_CCS=ccs_np.gamma_es_CCS, gamma_tr_CCS=ccs_np.gamma_tr_CCS)


def inputs_from_golden(g):
    d = {k[3:]: g[k] for k in g if k.startswith("in_")}
    for k in ("r0", "l0", "Em"):
        d[k] = float(d[k])
    return d


@pytest.mark.parametrize("name", ["ccs_o4v6.npz", "ccs_o6v9.npz"])
def test_ccs_oracle_matches_golden(name):
    g = load_golden(name)
    o, v = int(g["nocc"]), int(g["nvir"])
    out = ccs_calls(ccs_np.OracleGccs(synth.SynthEris(o, v)), _MOD, inputs_from_golden(g))
    assert len(out) > 60
    for k, val in out.items():
        assert np.abs(val - g[k]).max() < TOL, k


def test_inplace_shift_quirk():
    """Q6: tsupdate/lsupdate/rsupdate/es_lsupdate shift the passed intermediates in place."""
    o, v = 4, 6
    cc = ccs_np.OracleGccs(synth.SynthEris(o, v))
    d = ccs_inputs(o, v)
    inter = cc.T1inter(d["ts"], d["fsp"])
    before = inter[0].copy()
    cc.tsupdate(d["ts"], inter)
    assert np.abs(np.diagonal(inter[0] - before) + np.diagonal(cc.fock)[o:]).max() < 1e-14
    new = cc.rsupdate(d["rs"], 0.3, cc.R1inter(d["ts"], d["fsp"], d["vm"]), 0.7)
    assert np.all(new[0::2] == 0.0) and np.any(new[1::2] != 0.0)      # Q9 force_alpha


def test_l0_fromE_energy_argument_quirk():
    """Q12 (CCS.py:1488-1490): l0_fromE lowers an ndarray energy argument in place by 1/2 t1 t1 <jk||bc>."""
    from oracle import synth
    from oracle.ccs_np import OracleGccs
    o, v = 4, 6
    er = synth.SynthEris(o, v)
    rng = np.random.default_rng(2)
    ts, ls = 0.1 * rng.standard_normal((o, v)), 0.1 * rng.standard_normal((o, v))
    cc = OracleGccs(er)
    shift = 0.5 * np.einsum('jb,kc,jkbc', ts, ts, er.oovv)
    en = np.array([0.3])
    l0 = cc.l0_fromE(en, ts, ls, None)
    assert abs(en[0] - (0.3 - shift)) < 1e-15 and abs(float(np.ravel(l0)[0]) - float(cc.l0_fromE(0.3, ts, ls, None))) < 1e-14


def test_extract_r0_oracle_matches_reference_fixture():
    """`Gccs.Extract_r0` (CCS.py:1036-1079): the oracle against outputs of the unmodified reference
    (tests/golden/ccs_extract_r0.npz, oracle/make_golden_ccs_r0.py), both root branches and the ValueError."""
    from oracle import ccs_np, synth
    from oracle.make_golden import ccs_inputs
    from oracle.make_golden_ccs_r0 import SIZES, call, r1_variants
    g = load_golden("ccs_extract_r0.npz")
    for o, v in SIZES:
        cc = ccs_np.OracleGccs(synth.SynthEris(o, v))
        d = ccs_inputs(o, v)
        got = [call(cc, r1, d, vm) for vm in (d["vm"], d["vm2"]) for r1 in r1_variants(d)]
        got.append(call(cc, d["rs"], dict(d, fsp=None), d["vm"]))
        want, stat = g["r0_o%dv%d" % (o, v)], g["status_o%dv%d" % (o, v)]
        assert [s for _, s in got] == list(stat) and 0 in stat and 1 in stat
        for (x, s), w in zip(got, want):
            assert s == 1 or abs(x - w) < 1e-10 * max(1.0, abs(w))
