"""Host logic of bench.py that can be checked without a GPU."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def test_parts_breakdown_shape():
    import bench

    class FakeCC(object):
        def __init__(self):
            self.calls = []

        def gamma(self, *a):
            self.calls.append(("gamma", None))
            return 0

        def energy(self, *a):
            self.calls.append(("energy", None))
            return 0.0

        def tupdate(self, t1, t2, fsp=None, alpha=None):
            self.calls.append(("tupdate", alpha))
            return 1, 2

        def lupdate(self, t1, t2, l1, l2, fsp=None, alpha=None):
            self.calls.append(("lupdate", alpha))
            return 1, 2

    def timed(fn, steps, warmup):
        for _ in range(steps + warmup):
            out = fn()
        return 10.0 * steps, out

    import torch
    cc = FakeCC()
    t2 = torch.zeros(2, 2, 3, 4, dtype=torch.float64)
    parts = bench.time_parts(cc, timed, 1, t2, 3, t2.clone(), 5, reps=2, alpha=1e-3)
    assert set(parts) == {"alpha", "reps", "note", "gamma_ms", "energy_ms", "tupdate_ms", "lupdate_ms",
                          "tupdate_alpha_ms", "lupdate_alpha_ms", "tupdate_general_alpha_ms",
                          "lupdate_general_alpha_ms"}
    assert all(parts[k] == 10.0 for k in parts if k.endswith("_ms"))
    assert cc.calls.count(("tupdate", None)) == 3 and cc.calls.count(("lupdate", 1e-3)) == 6
    assert float(t2.abs().max()) == 0.0                      # the general-path amplitudes are copies


def test_ncu_traffic_only_for_a_matching_capture(tmp_path, monkeypatch):
    import json
    import bench
    (tmp_path / "profiles").mkdir()
    rec = {"nocc": 40, "nvir": 400, "n_gpus": 1, "dram_bytes_read": 5e10, "dram_bytes_write": 1e9,
           "algorithmic_bytes": 3.9e10, "source": "test"}
    (tmp_path / "profiles" / "r2_ladder_ncu.json").write_text(json.dumps(rec))
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    t = bench.ncu_traffic(40, 400, 1)
    assert t["bytes_per_launch"] == 5.1e10 and t["algorithmic_bytes_per_launch"] == 3.9e10
    assert bench.ncu_traffic(40, 400, 8) is None and bench.ncu_traffic(16, 96, 1) is None


def test_cpu_leg_is_a_measurement_with_the_extrapolation_labelled(monkeypatch):
    """cpu_baseline.value is what was measured at (16,96); the bench-shape figure lives under extrapolated_* only."""
    import bench
    monkeypatch.setattr(bench, "cpu_measure", lambda: {(10, 48): 0.5, (16, 96): 20.0})
    cb = bench.cpu_baseline(40, 400, {(16, 96): {"dev": 100.0, "e2e": 50.0}, (10, 48): {"dev": 300.0, "e2e": 150.0}})
    assert cb["value"] == 1.0 / 20.0 and cb["sample_shape"] == [16, 96] and cb["kind"] == "port"
    ss = cb["same_shape"]
    assert ss["shape"] == [16, 96] and ss["cpu_evals_s"] == 0.05 and ss["gpu_e2e_evals_s"] == 50.0 and ss["ratio"] == 1000.0
    assert cb["extrapolated_evals_per_sec_at_bench_shape"] < 1e-3 * cb["value"] and "NOT a measurement" in cb["extrapolation"]
    assert [x["shape"] for x in cb["same_shape_all"]] == [[10, 48], [16, 96]]


def test_dump_outputs_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: small outputs whole, large ones as the same seeded sample every run, float64 .npy files."""
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 100)
    big = torch.arange(1000, dtype=torch.float64).reshape(10, 10, 10)
    outs = {"gamma": torch.ones(5, 5, dtype=torch.float64), "energy": torch.tensor(-1.5, dtype=torch.float64), "t2": big}
    bench.dump_outputs(str(tmp_path / "a"), outs)
    bench.dump_outputs(str(tmp_path / "b"), outs)
    for name in outs:
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, b)
    t2 = np.load(tmp_path / "a" / "t2.npy")
    assert t2.shape == (100,) and np.all(np.diff(t2) > 0)          # distinct sorted flat indices of arange
    assert np.load(tmp_path / "a" / "energy.npy") == -1.5 and np.load(tmp_path / "a" / "gamma.npy").shape == (5, 5)
