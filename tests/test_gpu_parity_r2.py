"""Round-2 parity pins on the GPU (all through the C ABI):

* the BENCHMARK shape (nocc, nvir) = (40, 400) with the default engine against independent arithmetic — the
  sampled-element oracle (oracle/ccsd_columns.py: reference formulas on function-defined integrals, pinned to the full
  oracle in tests/test_oracle_columns_cpu.py) for all of T1, columns of T2 / L1 / L2, the rdm1 and the energy;
* the SURVEY §8(d) parity sizes (10,48), (16,96) and (20,160) against the full oracle with the ROUTING of the benchmark
  shape (ladders, rings, R4/R6/R9 on the INT8 pipe — asserted on the plan dump — the small products on DMMA);
* the sharded code paths on one GPU through virtual ranks (tests/virtual_ranks.py);
* the run-time accuracy guard of the INT8 route (adversarial operands, non-finite operands).
Tolerance 1e-10 absolute (BASELINE.json north_star)."""
import json

import numpy as np
import pytest

from helpers import MODES

pytestmark = pytest.mark.gpu
TOL = 1e-10


@pytest.fixture(scope="module")
def ecw(built_lib):
    import ecw_cc_b200
    return ecw_cc_b200


# ---------------------------------------------------------------------------------------- (a) the benchmark shape
PAIRS_40_400 = [(3, 250), (250, 399), (399, 3), (250, 250)]       # a < b, a > b, a == b; three distinct virtuals


def test_benchmark_shape_against_sampled_oracle(ecw, monkeypatch):
    import torch
    from oracle import synth, synth_fast
    from oracle.ccsd_columns import ColumnOracle
    from oracle.ccsd_np import OracleGCC
    if torch.cuda.get_device_properties(0).total_memory < 150e9:
        pytest.skip("needs a 180 GB GPU")
    monkeypatch.setenv("ECW_GEMM", "int8")
    monkeypatch.setenv("ECW_INT8_MIN_FLOPS", "2e10")
    o, v = 40, 400
    de = ecw.DeviceEris.synthetic(o, v)                    # product default: 6 digits, vvvv / ovvv_p as planes only
    cc = ecw.GCC(de)
    n = o + v
    d_t1, d_t2 = de.synth_tensor("t1", (o, v)), de.synth_tensor("t2", (o, o, v, v))
    d_l1, d_l2 = de.synth_tensor("l1", (o, v)), de.synth_tensor("l2", (o, o, v, v))
    d_f = de.synth_tensor("fsp", (n, n))
    # the default plans of this shape do run the heavy products on the INT8 pipe
    for fn in ("tupdate", "lupdate"):
        ops = json.loads(cc.plan_json(fn))["ops"]
        notes = [op["note"] for op in ops if op["kind"] == "oz_gemm"]
        for want in (("K1 pp ladder", "R1 Wovvo", "R2 ring", "R9 Y") if fn == "tupdate" else
                     ("K2 pp ladder", "R3 v4", "R7 ring", "R8 l2.t2", "R4 wovoo", "R6 ovvv")):
            assert any(want in s for s in notes), (fn, want)
    pairs = PAIRS_40_400
    got = {}
    modes = (("upd", None),)           # the mode the benchmark runs; the L1 modes are element-wise on top of it
    for tag, alpha in modes:
        a1, a2 = cc.tupdate(d_t1, d_t2, fsp=d_f, alpha=alpha)
        got["T1" + tag] = a1.cpu().numpy()
        got["T2" + tag] = np.stack([a2[:, :, a, b].cpu().numpy() for a, b in pairs])
        del a1, a2
        b1, b2 = cc.lupdate(d_t1, d_t2, d_l1, d_l2, fsp=d_f, alpha=alpha)
        got["L1" + tag] = b1.cpu().numpy()
        got["L2" + tag] = np.stack([b2[:, :, a, b].cpu().numpy() for a, b in pairs])
        del b1, b2
    got["gamma"] = cc.gamma(d_t1, d_t2, d_l1, d_l2).cpu().numpy()
    got["E"] = float(cc.energy(d_t1, d_t2, d_f))
    assert de.guard_trips == 0 and 0.0 < de.max_bound < de.int8_tol
    bound = de.max_bound
    del cc, de, d_t2, d_l2
    torch.cuda.empty_cache()
    # ---- independent arithmetic on the host
    prov = synth_fast.SynthProvider(o, v)
    t1, t2, l1, l2 = synth_fast.amplitudes(o, v)
    fsp = synth.fsp(o, v)
    col = ColumnOracle(prov, pairs)
    worst = {}
    for tag, alpha in modes:
        r1, r2 = col.tupdate(t1, t2, fsp=fsp, alpha=alpha)
        worst["T1" + tag] = np.abs(got["T1" + tag] - r1).max()
        worst["T2" + tag] = np.abs(got["T2" + tag] - r2).max()
        q1, q2 = col.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha)
        worst["L1" + tag] = np.abs(got["L1" + tag][:, col.xs] - q1).max()
        worst["L2" + tag] = np.abs(got["L2" + tag] - q2).max()
        assert np.abs(r2).max() > 1e-3 and np.abs(q2).max() > 1e-3          # the columns are not trivially zero
    class _E:                                                                # rdm1 / energy need amplitudes + oovv only
        nocc, fock, oovv = o, prov.fock, prov.oovv
    orc = OracleGCC(_E)
    worst["gamma"] = np.abs(got["gamma"] - orc.gamma(t1, t2, l1, l2)).max()
    worst["E"] = abs(got["E"] - orc.energy(t1, t2, fsp))
    print("(40,400) default engine vs sampled oracle (INT8 worst-case bound %.1e): " % bound
          + ", ".join("%s %.1e" % kv for kv in sorted(worst.items())))
    assert max(worst.values()) < TOL, worst


# ---------------------------------------------------------------------------------------- (b) SURVEY parity sizes
def _routing_threshold(o, v):
    """2e10 flop at (40,400), scaled like an o^3 v^3 product."""
    return 2e10 * (o / 40.0) ** 3 * (v / 400.0) ** 3


@pytest.mark.parametrize("ov", [(10, 48), (16, 96), (20, 160)])
def test_survey_sizes_with_benchmark_routing(ecw, ov):
    import psutil
    import torch
    from oracle import synth, synth_fast
    from oracle.ccsd_np import OracleGCC
    o, v = ov
    if 8.0 * v ** 4 * 6 > psutil.virtual_memory().available:
        pytest.skip("the full oracle needs %d GB of host memory here" % (8.0 * v ** 4 * 6 / 1e9))
    er = synth_fast.FastSynthEris(o, v)
    t1, t2, l1, l2 = synth_fast.amplitudes(o, v)
    fsp = synth.fsp(o, v)
    de = ecw.DeviceEris.from_geris(er, gemm="int8", int8_digits=6, int8_min_flops=-_routing_threshold(o, v))
    cc = ecw.GCC(de)
    for fn in ("tupdate", "lupdate"):
        ops = json.loads(cc.plan_json(fn))["ops"]
        oz = [op["note"] for op in ops if op["kind"] == "oz_gemm"]
        dm = [op for op in ops if op["kind"] == "gemm"]
        for want in (("K1 pp ladder", "R1 Wovvo", "R2 ring", "R9 Y") if fn == "tupdate" else
                     ("K2 pp ladder", "R3 v4", "R7 ring", "R8 l2.t2", "R4 wovoo", "R6 ovvv")):
            assert any(want in s for s in oz), (fn, want, oz)
        assert len(dm) >= 10                                   # the small products stay on the FP64 DMMA kernels
    orc = OracleGCC(er)
    worst = 0.0
    for tag, alpha, eq in (MODES if v < 100 else MODES[:1] + MODES[2:3]):
        a, b = cc.tupdate(t1, t2, fsp=fsp, alpha=alpha, equation=eq)
        c, d = orc.tupdate(t1, t2, fsp=fsp, alpha=alpha, equation=eq)
        worst = max(worst, np.abs(a - c).max(), np.abs(b - d).max())
        a, b = cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq)
        c, d = orc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq)
        worst = max(worst, np.abs(a - c).max(), np.abs(b - d).max())
    worst = max(worst, np.abs(cc.gamma(t1, t2, l1, l2) - orc.gamma(t1, t2, l1, l2)).max())
    worst = max(worst, abs(cc.energy(t1, t2, fsp) - orc.energy(t1, t2, fsp)))
    print("(%d,%d) benchmark routing vs full oracle: %.2e (INT8 worst-case bound %.1e)" % (o, v, worst, de.max_bound))
    assert worst < TOL and de.guard_trips == 0
    del cc, de
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------- (c) virtual ranks
@pytest.mark.parametrize("world,ov,antisym", [(2, (8, 16), True), (2, (8, 16), False), (3, (5, 9), True), (4, (6, 14), False)])
def test_sharded_paths_on_one_gpu(ecw, world, ov, antisym, engine):
    """Every rank's sharded plan (vvvv row shard, owner-computes GEMMs, split contractions, all-gathers) executed
    concurrently on one device; all ranks must reproduce the unsharded oracle."""
    from oracle import synth
    from oracle.ccsd_np import OracleGCC
    from virtual_ranks import run_ranks
    o, v = ov
    er = synth.SynthEris(o, v)
    fsp = synth.fsp(o, v)
    if antisym:
        t1, t2, l1, l2 = synth.amplitudes(o, v)
    else:
        rng = np.random.default_rng(5)
        t1, l1 = 0.05 * rng.standard_normal((o, v)), 0.05 * rng.standard_normal((o, v))
        t2, l2 = 0.02 * rng.standard_normal((o, o, v, v)), 0.02 * rng.standard_normal((o, o, v, v))

    def body(rank, comm):
        cc = ecw.GCC(er, rank=rank, world=world)
        cc.eris.comm = comm
        assert cc.eris.world == world and cc.eris.buf["vvvv_p"].numel() <= (v * (v - 1) // 2 // world + 1) * (v * (v - 1) // 2)
        res = []
        for alpha, eq in ((None, False), (1e-3, False), (None, True)):
            res += list(cc.tupdate(t1, t2, fsp=fsp, alpha=alpha, equation=eq))
            res += list(cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq))
        res.append(cc.gamma(t1, t2, l1, l2))
        res.append(np.array(cc.energy(t1, t2, fsp)))
        return res

    outs, comm = run_ranks(world, body)
    assert comm.gathers >= 30                                  # the distributed contractions did go through the exchange
    orc = OracleGCC(er)
    ref = []
    for alpha, eq in ((None, False), (1e-3, False), (None, True)):
        ref += list(orc.tupdate(t1, t2, fsp=fsp, alpha=alpha, equation=eq))
        ref += list(orc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha, equation=eq))
    ref.append(orc.gamma(t1, t2, l1, l2))
    ref.append(np.array(orc.energy(t1, t2, fsp)))
    for r, res in enumerate(outs):
        for k, (x, y) in enumerate(zip(res, ref)):
            assert np.abs(x - y).max() < TOL, (r, k)
        for x, y in zip(res, outs[0]):
            assert np.array_equal(x, y), "ranks hold bit-identical replicas"


# ---------------------------------------------------------------------------------------- (e) accuracy guard
def test_int8_guard_adversarial_operands(ecw):
    """Amplitudes 1e4 times the usual size push the worst-case INT8 bound over the tolerance: a container with the
    FP64 layouts repeats the call on the DMMA kernels (result at FP64 accuracy), a planes-only container refuses."""
    from oracle import synth
    from oracle.ccsd_np import OracleGCC
    o, v = 8, 16
    er = synth.SynthEris(o, v)
    t1, t2, l1, l2 = synth.amplitudes(o, v)
    fsp = synth.fsp(o, v)
    orc = OracleGCC(er)
    de = ecw.DeviceEris.from_geris(er, gemm="int8", int8_digits=6, int8_min_flops=-1)
    cc = ecw.GCC(de)
    cc.tupdate(t1, t2, fsp=fsp, equation=True)
    usual = de.last_bound
    assert de.guard_trips == 0 and 0.0 < usual < 1e-12
    big = 1e4 * t2
    a, b = cc.tupdate(t1, big, fsp=fsp, equation=True)
    assert de.guard_trips == 1 and de.last_bound > de.int8_tol
    c, d = orc.tupdate(t1, big, fsp=fsp, equation=True)
    scale = np.abs(d).max()
    assert scale > 1e3 and np.abs(b - d).max() < 1e-13 * scale and np.abs(a - c).max() < 1e-13 * scale
    # the bound is the advertised formula on the actual row scales: quadratic terms scale like 1e8
    assert 1e3 * usual < de.last_bound < 1e9 * usual
    # a looser tolerance keeps the INT8 route; the guard can be switched off
    de2 = ecw.DeviceEris.from_geris(er, gemm="int8", int8_digits=6, int8_min_flops=-1, int8_tol=0.0)
    ecw.GCC(de2).tupdate(t1, big, fsp=fsp, equation=True)
    assert de2.guard_trips == 0
    # planes only: nothing to fall back to
    ds = ecw.DeviceEris.synthetic(o, v, gemm="int8", int8_digits=6, int8_min_flops=-1)
    cs = ecw.GCC(ds)
    cs.tupdate(t1, t2, fsp=fsp, equation=True)
    with pytest.raises(ecw.EcwError, match="cannot guarantee"):
        cs.tupdate(t1, big, fsp=fsp, equation=True)


def test_non_finite_amplitudes_propagate(ecw, engine):
    """A NaN / Inf in an amplitude must come out as NaN (reference: numpy propagates it), not as finite garbage from
    the digit cut."""
    from oracle import synth
    o, v = 8, 16
    er = synth.SynthEris(o, v)
    t1, t2, l1, l2 = synth.amplitudes(o, v)
    fsp = synth.fsp(o, v)
    cc = ecw.GCC(er)
    for bad in (np.nan, np.inf):
        x = t2.copy()
        x[1, 2, 3, 4] = bad
        x[2, 1, 3, 4] = -bad
        x[1, 2, 4, 3] = -bad
        x[2, 1, 4, 3] = bad
        a, b = cc.tupdate(t1, x, fsp=fsp, equation=True)
        assert not np.isfinite(b[1, 2, 3, 4]) and np.isnan(b).sum() > o * o       # the ladder spreads it over (i,j)
        a, b = cc.lupdate(t1, x, l1, l2, fsp=fsp, equation=True)
        assert np.isnan(b).any() and np.isnan(a).any()
        assert np.isnan(cc.gamma(t1, x, l1, l2)).any()

