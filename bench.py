#!/usr/bin/env python
"""bench.py — CCSD T+Lambda residual evaluations per second on B200.

One *step* = the work of one `Solver_CCSD.SCF` iteration body (Solver_GS.py:683-705):
`gamma` + `energy` + `tupdate` + `lupdate` on the synthetic spin-orbital workload
(nocc, nvir) = (40, 400), FP64 (BASELINE.json configs[3]).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                 # also write the last timed step's results to DIR/*.npy

Prints ONE JSON line.  `value` = steps/s with everything resident in HBM; `e2e` = the same through
the reference-facing API (`GCC.gamma/energy/tupdate/lupdate`) with HOST (pinned numpy) buffers,
host<->device copies inside the timed region.  `roofline` is for the dominant launch (the packed
particle-particle ladder GEMM), timed live with CUDA events on the launching stream.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ccsd_t_lambda_residual_evals_per_sec"
UNIT = "evals/s"
NOMINAL_FP64_TFLOPS = 37.0     # B200 datasheet FP64 / FP64-tensor (context only)


def f_alg(o, v):
    """Algorithmic flops per evaluation (SURVEY.md §8(d))."""
    po, pv = o * (o - 1) // 2, v * (v - 1) // 2
    return 4.0 * po * pv * pv + 18.0 * o ** 3 * v ** 3 + 14.0 * o ** 4 * v ** 2


def f_ref(o, v):
    """Dense flops the reference factorisation executes (K1-K5, R1-R7, o^4v^2 terms; SURVEY §2.2)."""
    return 8.0 * o ** 2 * v ** 4 + 2.0 * o * v ** 4 + 14.0 * o ** 3 * v ** 3 + 14.0 * o ** 4 * v ** 2


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                               "--format=csv,noheader,nounits"], timeout=5).decode()
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for nm, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ----------------------------------------------------------------------------- CPU (reference algorithm)
CPU_SHAPES = [(10, 48), (16, 96)]          # BASELINE.md section 3 / SURVEY 8(d): the sizes the reference's CPU path is timed at


def use_all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs use every host core (and say how many)."""
    n = os.cpu_count() or 1
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(n)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=n)
    except Exception:
        pass
    return n


def cpu_eval_time(o, v, reps=1, warm=0):
    """Seconds per evaluation (gamma + energy + tupdate + lupdate) of the reference algorithm: the numpy port
    oracle/ccsd_np.py with the reference's own einsum routing (pyscf.lib.einsum -> BLAS, plain np.einsum -> C loops),
    pinned to the unmodified reference in tests/test_oracle_pins.py."""
    from oracle import synth, synth_fast
    from oracle.ccsd_np import OracleGCC
    er = synth_fast.FastSynthEris(o, v)
    t1, t2, l1, l2 = synth_fast.amplitudes(o, v)
    fsp = synth.fsp(o, v)
    cc = OracleGCC(er, faithful=True)

    def one():
        cc.gamma(t1, t2, l1, l2)
        cc.energy(t1, t2, fsp)
        cc.tupdate(t1, t2, fsp=fsp)
        cc.lupdate(t1, t2, l1, l2, fsp=fsp)

    for _ in range(warm):
        one()
    best = 1e99
    for _ in range(reps):
        t0 = time.perf_counter()
        one()
        best = min(best, time.perf_counter() - t0)
    return best


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else (os.cpu_count() or 1)
    except Exception:
        return os.cpu_count() or 1


def cpu_measure():
    """{shape: seconds per eval} at CPU_SHAPES: 3 evals (best) at (10,48), one at (16,96) — 30-60 s of CPU work."""
    use_all_host_cores()
    return {(10, 48): cpu_eval_time(10, 48, reps=3, warm=1), (16, 96): cpu_eval_time(16, 96, reps=1, warm=0)}


def cpu_baseline(o, v, gpu_same_shape):
    """Measured CPU numbers at the shapes the reference can run, beside THIS RUN's GPU numbers at the same shapes; the
    (nocc, nvir) of the bench line itself is out of the reference's reach (three v^4 arrays: ~600 GB at (40,400)), so
    the figure for it is an extrapolation and is labelled as one."""
    sec = cpu_measure()
    so, sv = CPU_SHAPES[-1]
    same = []
    for (a, b) in CPU_SHAPES:
        g = gpu_same_shape.get((a, b), {})
        cpu = 1.0 / sec[(a, b)]
        same.append({"shape": [a, b], "cpu_evals_s": cpu, "cpu_s_per_eval": sec[(a, b)],
                     "gpu_evals_s": g.get("dev"), "gpu_e2e_evals_s": g.get("e2e"),
                     "ratio": (g.get("e2e") / cpu) if g.get("e2e") else None,
                     "ratio_device_resident": (g.get("dev") / cpu) if g.get("dev") else None})
    factor = f_ref(so, sv) / f_ref(o, v)
    return {"value": 1.0 / sec[(so, sv)], "unit": UNIT, "cores": blas_threads(), "kind": "port",
            "sample": "MEASURED at (nocc,nvir)=(%d,%d), the largest SURVEY 8(d) CPU size: reference algorithm "
                      "(oracle/ccsd_np.py, reference's einsum routing), %d BLAS threads, %.2f s per eval; the bench "
                      "shape (%d,%d) cannot be run by the reference (~600 GB of v^4 intermediates)"
                      % (so, sv, blas_threads(), sec[(so, sv)], o, v),
            "sample_shape": [so, sv],
            "same_shape": same[-1], "same_shape_all": same,
            "extrapolated_evals_per_sec_at_bench_shape": (1.0 / sec[(so, sv)]) * factor,
            "extrapolation": "NOT a measurement: the (%d,%d) rate times the ratio of the reference's dense flop "
                             "counts f_ref(%d,%d)/f_ref(%d,%d) = %.3g" % (so, sv, so, sv, o, v, factor)}


def run_reference(args):
    """The reference arm: the reference algorithm on the host cores.  It cannot execute the bench shape, so every
    number printed here is MEASURED at the CPU shapes of BASELINE.md section 3 and the line says so in `config`; the
    flop-count extrapolation to the bench shape sits under an `extrapolated_*` key only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = use_all_host_cores()
    o, v = args.nocc, args.nvir
    so, sv = CPU_SHAPES[-1]
    for _ in range(min(args.warmup, 1)):
        cpu_eval_time(10, 48)
    small = [cpu_eval_time(10, 48) for _ in range(max(1, min(args.steps, 20)))]
    t0 = time.perf_counter()
    big = []
    while len(big) < args.steps and (not big or time.perf_counter() - t0 + big[-1] < 100.0):
        big.append(cpu_eval_time(so, sv))                       # bounded: as many (16,96) evals as fit ~100 s
    sec = sum(big) / len(big)
    val = 1.0 / sec
    factor = f_ref(so, sv) / f_ref(o, v)
    cb = {"value": val, "unit": UNIT, "cores": blas_threads(), "kind": "port",
          "sample": "reference algorithm (oracle port, reference's einsum routing) MEASURED at (%d,%d): %d evals, "
                    "%.2f s each, %d host threads; (10,48): %d evals, %.3f s each"
                    % (so, sv, len(big), sec, ncores, len(small), sum(small) / len(small)),
          "sample_shape": [so, sv], "evals_per_sec_10_48": len(small) / sum(small),
          "extrapolated_evals_per_sec_at_bench_shape": val * factor,
          "extrapolation": "NOT a measurement: x f_ref(%d,%d)/f_ref(%d,%d) = %.3g" % (so, sv, o, v, factor)}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "steps_timed": len(big), "warmup": args.warmup, "ms_per_step": 1e3 * sec,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "synthetic spin-orbital CCSD T+Lambda residual (gamma+energy+tupdate+lupdate), "
                                   "nocc=%d nvir=%d FP64 - the largest shape of SURVEY 8(d) the reference's CPU path "
                                   "runs; the bench shape nocc=%d nvir=%d needs ~600 GB there.  Same-shape GPU numbers: "
                                   "cpu_baseline.same_shape of the other arm's line" % (so, sv, o, v),
                       "nocc": so, "nvir": sv, "bench_shape": [o, v]},
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- ours
def measure_fp64_peak(torch, n=8192, reps=5):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    c = torch.empty(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 1e99
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.matmul(a, b, out=c)
        e.record()
        e.synchronize()
        best = min(best, s.elapsed_time(e))
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / best / 1e9


def measure_int8_peak(torch, n=8192, burst_reps=10, sustain_s=4.0):
    """Dense INT8 tensor-core rate of this GPU, TOP/s: torch._int_mm (cuBLASLt int8 -> int32) 8192^3, best of 10
    (burst) and back to back for ~4 s (sustained) — the same protocol as MEASURED_PEAKS.json's bf16 figures."""
    a = torch.randint(-128, 127, (n, n), dtype=torch.int8, device="cuda")
    b = torch.randint(-128, 127, (n, n), dtype=torch.int8, device="cuda")
    for _ in range(3):
        torch._int_mm(a, b)
    torch.cuda.synchronize()
    ops = 2.0 * n ** 3
    best = 1e99
    for _ in range(burst_reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch._int_mm(a, b)
        e.record()
        e.synchronize()
        best = min(best, s.elapsed_time(e))
    reps = max(10, int(sustain_s * 1e3 / best))
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        torch._int_mm(a, b)
    e.record()
    e.synchronize()
    sustained = ops * reps / s.elapsed_time(e) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return {"burst_tops": ops / best / 1e9, "sustained_tops": sustained, "reps_sustained": reps,
            "how": "torch._int_mm int8 %d^3: best of %d (burst); %d back-to-back launches (sustained)" % (n, burst_reps, reps)}


def ncu_traffic(o, v, world):
    """dram bytes read+written by the dominant launch from the committed `ncu --set full` capture of THIS shape and
    GPU count (profiles/r2_ladder_ncu.json); None when there is no capture that matches."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_ladder_ncu.json")))
        if [o, v, world] != [d["nocc"], d["nvir"], d["n_gpus"]]:
            return None
        return {"bytes_per_launch": d["dram_bytes_read"] + d["dram_bytes_write"],
                "algorithmic_bytes_per_launch": d["algorithmic_bytes"], "source": d["source"]}
    except Exception:
        return None


def same_shape_gpu(ecw, torch, shapes, reps=5):
    """evals/s of this repo's path at the shapes the CPU leg is measured at: device resident and through the numpy API
    (host arrays in, host arrays out)."""
    from oracle import synth, synth_fast
    out = {}
    for (o, v) in shapes:
        er = synth_fast.FastSynthEris(o, v)
        t1, t2, l1, l2 = synth_fast.amplitudes(o, v)
        fsp = synth.fsp(o, v)
        cc = ecw.GCC(er)
        dev = [torch.from_numpy(x).cuda() for x in (t1, t2, l1, l2, fsp)]

        def step(a):
            cc.gamma(a[0], a[1], a[2], a[3])
            cc.energy(a[0], a[1], a[4])
            cc.tupdate(a[0], a[1], fsp=a[4])
            cc.lupdate(a[0], a[1], a[2], a[3], fsp=a[4])

        res = {}
        for tag, args_ in (("dev", dev), ("e2e", [t1, t2, l1, l2, fsp])):
            step(args_)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                step(args_)
            torch.cuda.synchronize()
            res[tag] = reps / (time.perf_counter() - t0)
        out[(o, v)] = res
        del cc, dev
        torch.cuda.empty_cache()
    return out


def time_parts(cc, timed, t1, t2, l1, l2, fsp, reps=2, alpha=1e-3):
    """ms per call of the four functions of one evaluation, and of the two updates with the L1 term (SURVEY §8d:
    "report also tupdate and lupdate separately, and with/without alpha").  `timed(fn, steps, warmup) -> (ms, out)`."""
    calls = [("gamma", lambda: cc.gamma(t1, t2, l1, l2)),
             ("energy", lambda: cc.energy(t1, t2, fsp)),
             ("tupdate", lambda: cc.tupdate(t1, t2, fsp=fsp, alpha=None)),
             ("lupdate", lambda: cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=None)),
             ("tupdate_alpha", lambda: cc.tupdate(t1, t2, fsp=fsp, alpha=alpha)),
             ("lupdate_alpha", lambda: cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha))]
    # the path every L1-regularised iteration after the first runs: amplitudes without antisymmetry (Q11)
    g2, gl2 = t2.clone(), l2.clone()
    g2[0, 1, 2, 3] += 1e-3
    gl2[0, 1, 2, 3] += 1e-3
    calls += [("tupdate_general_alpha", lambda: cc.tupdate(t1, g2, fsp=fsp, alpha=alpha)),
              ("lupdate_general_alpha", lambda: cc.lupdate(t1, g2, l1, gl2, fsp=fsp, alpha=alpha))]
    out = {"alpha": alpha, "reps": reps,
           "note": "*_general_*: doubles amplitudes without antisymmetry (what the reference's L1 update leaves, "
                   "utilities.py:59-67): the general plans, dense (ij) ladder rows"}
    for name, fn in calls:
        ms, res = timed(fn, reps, 1)
        del res
        out[name + "_ms"] = ms / reps
    return out


def time_ccs(ecw, torch, o=24, v=240, reps=5):
    """ms per iteration body of the ECW-CCS solvers at a synthetic (nocc, nvir): the ground-state body of
    Solver_CCS.SCF (Solver_GS.py:166-204: T1inter, tsupdate, L1inter, lsupdate, gamma, energy_ccs) and the per-state
    right + left body of Solver_ES.SCF (Solver_ES.py:258-368: R1inter, Extract_Em_r, rsupdate, R0inter, r0update,
    es_L1inter, Extract_Em_l, es_lsupdate, L0inter, l0update), through the numpy API of ecw_cc_b200.Gccs."""
    import numpy as np
    de = ecw.DeviceEris.synthetic(o, v, gemm="int8", keep_fp64_vvvv=True)
    cc = ecw.Gccs(de)
    n = o + v
    rng = np.random.default_rng(3)
    ts, ls, rs, rl = (0.05 * rng.standard_normal((o, v)) for _ in range(4))
    fsp = de.fock + 0.02 * rng.standard_normal((n, n))
    vm = 0.02 * rng.standard_normal((n, n))

    def gs():
        t = cc.tsupdate(ts, cc.T1inter(ts, fsp))
        l = cc.lsupdate(t, ls, cc.L1inter(t, fsp))
        cc.gamma(t, l)
        cc.energy_ccs(t, fsp)

    def es():
        ri = cc.R1inter(ts, fsp, vm)
        em, _, _ = cc.Extract_Em_r(rs, 0.3, ri)
        cc.rsupdate(rs, 0.3, ri, em)
        cc.r0update(rs, 0.3, em, cc.R0inter(ts, fsp, vm))
        li = cc.es_L1inter(ts, fsp, vm)
        el, _, _ = cc.Extract_Em_l(rl, 0.2, li)
        cc.es_lsupdate(rl, 0.2, el, li)
        cc.l0update(rl, 0.2, el, cc.L0inter(ts, fsp, vm))

    out = {"nocc": o, "nvir": v, "reps": reps}
    for name, fn in (("ccs_gs_iteration_ms", gs), ("ccs_es_state_iteration_ms", es)):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        out[name] = 1e3 * (time.perf_counter() - t0) / reps
    del cc, de
    torch.cuda.empty_cache()
    return out


def config5_ladder(ecw, torch, dist, rank, world, reps=3):
    """BASELINE.json configs[4] — "nocc=60 nvir=800, vvvv ladder sharded at 2/4/8 B200": the packed particle-particle
    ladder (CCSD.py:305) R[ij_p, ab_p] = sum_{cd_p} tau_p[ij_p, cd_p] vvvv_p[ab_p, cd_p] at (60, 800) with the digit planes
    of vvvv_p (613 GB) row-sharded over the packed virtual pair index, through the same C entry points the residual
    plans use (ecw_eris_vvvv_planes, ecw_ozaki_split, ecw_ozaki_gemm) plus an NCCL all-gather of the result.  The whole
    residual at this shape does not fit 8 x 180 GB with the current lowering (DESIGN.md section 7); this is the sharded
    ladder on its own.  Returns a dict (extra key `config5` of the bench line); never raises."""
    from ecw_cc_b200 import lib
    from ecw_cc_b200.eris import SYNTH_KIND
    o, v, ns = 60, 800, 6
    if os.environ.get("ECW_CONFIG5_SHAPE"):                     # smoke runs of this leg on a small shape
        o, v = (int(x) for x in os.environ["ECW_CONFIG5_SHAPE"].split(","))
    po, pv = o * (o - 1) // 2, v * (v - 1) // 2
    nshmax = (pv + world - 1) // world
    out = {"nocc": o, "nvir": v, "n_gpus": world, "what": "packed pp-ladder (CCSD.py:305) with vvvv planes row-sharded"}
    try:
        torch.cuda.empty_cache()
        free, total = torch.cuda.mem_get_info()
        need = ns * nshmax * pv * 1.01 + 8.0 * po * pv * 2.8 + 8.0 * po * nshmax * (world + 1) + 2.5e9
        out["per_rank_gb"] = {"vvvv_planes": ns * nshmax * pv / 1e9, "tau_fp64_and_planes": 8.0 * po * pv * 1.75 / 1e9,
                              "result_shard_gathered_full": 8.0 * po * (nshmax * (world + 1) + pv) / 1e9,
                              "needed": need / 1e9, "free": free / 1e9}
        if need > 0.95 * free:
            out["skipped"] = "needs %.0f GB per rank, %.0f GB free" % (need / 1e9, free / 1e9)
            return out
        t0 = time.perf_counter()
        de = ecw.DeviceEris(o, v, rank=rank, world=world, gemm="int8", int8_digits=ns)
        n0, nsh = de._shard_rows()
        chunk_rows = max(128, min(4096, (1 << 28) // pv // 128 * 128))
        tmp = torch.empty(chunk_rows * pv, dtype=torch.float64, device="cuda")

        def rows(r0, nr):
            if lib.ecw_synth_tensor(SYNTH_KIND["vvvv_p"], tmp.data_ptr(), o, v, n0 + r0, nr, 0.01, de.stream()) != 0:
                raise RuntimeError("ecw_synth_tensor(vvvv_p rows) failed")
            return tmp
        de._cut_vvvv_planes(rows, chunk_rows)
        torch.cuda.synchronize()
        out["setup_s"] = time.perf_counter() - t0
        st = de.stream()
        g = torch.Generator(device="cuda").manual_seed(20260)          # the same operand on every rank
        tau = (torch.rand((po, pv), generator=g, dtype=torch.float64, device="cuda") - 0.5) * 0.04
        pb = torch.empty(int(lib.ecw_ozaki_plane_bytes(po, pv, ns)), dtype=torch.int8, device="cuda")
        sb = torch.empty(int(lib.ecw_ozaki_stat_elems(po)), dtype=torch.float64, device="cuda")
        cr = torch.zeros((po, nshmax), dtype=torch.float64, device="cuda")
        full = torch.empty((world, po, nshmax), dtype=torch.float64, device="cuda")
        res = torch.empty((po, pv), dtype=torch.float64, device="cuda")
        pa, sa = de.buf["vvvv_oz"], de.buf["vvvv_ozs"]

        def gemm():
            if lib.ecw_ozaki_gemm(pa.data_ptr(), sa.data_ptr(), pb.data_ptr(), sb.data_ptr(), nsh, po, pv, cr.data_ptr(),
                                  1, nshmax, 1.0, 0.0, ns, st) != 0:
                raise RuntimeError("ecw_ozaki_gemm failed")

        def step():
            if lib.ecw_ozaki_split(tau.data_ptr(), po, pv, pv, 1, ns, pb.data_ptr(), sb.data_ptr(), st) != 0:
                raise RuntimeError("ecw_ozaki_split failed")
            gemm()
            if world > 1:
                dist.all_gather_into_tensor(full, cr)
                res.copy_(full.permute(1, 0, 2).reshape(po, world * nshmax)[:, :pv])
            else:
                res.copy_(cr[:, :pv])

        step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gemm()
        g1.record()
        torch.cuda.synchronize()
        gemm_ms = g0.elapsed_time(g1)
        # spot check against FP64 arithmetic: three columns of this rank's shard from regenerated FP64 vvvv rows
        worst = 0.0
        row = torch.empty(pv, dtype=torch.float64, device="cuda")
        for m in (0, nsh // 2, nsh - 1):
            if lib.ecw_synth_tensor(SYNTH_KIND["vvvv_p"], row.data_ptr(), o, v, n0 + m, 1, 0.01, st) != 0:
                raise RuntimeError("ecw_synth_tensor failed")
            ref = tau @ row
            worst = max(worst, float((res[:, n0 + m] - ref).abs().max()))
        if world > 1:
            t = torch.tensor([ms, gemm_ms, worst], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, gemm_ms, worst = float(t[0]), float(t[1]), float(t[2])
        flops = 2.0 * po * pv * float(pv)
        out.update({"ladder_ms": ms, "ladder_gemm_ms": gemm_ms, "ladders_per_sec": 1e3 / ms,
                    "fp64_equivalent_tflops_all_gpus": flops / ms / 1e9,
                    "fp64_equivalent_tflops_per_gpu_gemm_only": flops * (nsh / float(pv)) / gemm_ms / 1e9,
                    "launch": "%dx%dx%d per rank (M = vvvv rows of the shard, N = P_o, K = P_v)" % (nsh, po, pv),
                    "max_abs_err_vs_fp64_3_columns_per_rank": worst,
                    "timed": "digit cut of tau_p + INT8 product on the shard + ncclAllGather of the result + layout copy, "
                             "%d repetitions, max over ranks" % reps})
        del de, tmp, tau, pb, sb, cr, full, res, pa, sa
        torch.cuda.empty_cache()
    except Exception as exc:                                    # never lose the bench line over this extra key
        out["error"] = repr(exc)[:300]
        try:
            torch.cuda.empty_cache()
        except Exception:
            pass
    return out


def np_copy(x):
    import numpy as np
    return np.array(x, copy=True)


DUMP_SAMPLE = 1 << 21          # elements kept of an output larger than this: 16 MB in float64
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 20261020


def dump_outputs(path, outs):
    """Write {name: device tensor} as path/<name>.npy in float64.  An output with more than DUMP_SAMPLE elements is
    stored as the flat elements at a fixed, seeded set of sorted indices (the same for every run at the same shape),
    so that two builds can be compared output for output; smaller ones are stored whole, in their own shape."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in outs.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(t.numel(), size=DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy().astype(np.float64)
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise RuntimeError("--dump-outputs: more than %d bytes" % DUMP_MAX_BYTES)
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import lib

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries ONE JSON line: whatever libraries print to file descriptor 1 during the run (NCCL's version banner at
    # NCCL_DEBUG >= VERSION, ...) is sent to stderr; the line itself goes to the saved descriptor
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    o, v = args.nocc, args.nvir
    n = o + v

    de = ecw.DeviceEris.synthetic(o, v, rank=rank, world=world, gemm=args.gemm, int8_digits=args.int8_digits)
    cc = ecw.GCC(de)
    ns = de.int8_digits
    t1, t2 = de.synth_tensor("t1", (o, v)), de.synth_tensor("t2", (o, o, v, v))
    l1, l2 = de.synth_tensor("l1", (o, v)), de.synth_tensor("l2", (o, o, v, v))
    fsp = de.synth_tensor("fsp", (n, n))
    alpha = args.alpha

    def step_dev():
        g = cc.gamma(t1, t2, l1, l2)
        e = cc.energy(t1, t2, fsp)
        a, b = cc.tupdate(t1, t2, fsp=fsp, alpha=alpha)
        c, d = cc.lupdate(t1, t2, l1, l2, fsp=fsp, alpha=alpha)
        return g, e, a, b, c, d

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        out = None
        for _ in range(warmup):
            out = fn()          # results are held over the next call, as in the timed loop (and in a solver loop): the
        barrier()               # pinned result blocks of both generations exist before the clock starts
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            out = fn()
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, out

    # ---- device-resident leg (value) with clocks sampled during the timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.ecw_profile_enable(de._h, 0)
    ms_dev, last = timed(step_dev, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("gamma", "energy", "tupdate_t1", "tupdate_t2", "lupdate_l1",
                                                  "lupdate_l2"), last)))
    del last

    # ---- the functions of one evaluation on their own, and the updates with the L1 term (extra key "parts")
    try:
        parts = time_parts(cc, timed, t1, t2, l1, l2, fsp)
    except Exception as exc:                                   # never lose the bench line over the breakdown
        parts = {"error": repr(exc)[:200]}

    # ---- dominant launch, timed live with CUDA events on the launching stream
    lib.ecw_profile_enable(de._h, 1)
    ladder_ms = []
    for _ in range(min(args.steps, 3)):
        cc.tupdate(t1, t2, fsp=fsp, alpha=alpha)
        buf = ctypes.create_string_buffer(1 << 22)
        lib.ecw_profile_dump(de._h, buf, 1 << 22)
        ops = json.loads(buf.value.decode())
        ladder_ms += [x["ms"] for x in ops if x["kind"] in ("gemm", "oz_gemm") and "K1 pp ladder" in x["note"]]
    lib.ecw_profile_enable(de._h, 0)
    ladder = [x for x in ops if x["kind"] in ("gemm", "oz_gemm") and "K1 pp ladder" in x["note"]][0]
    ladder_flops = 2.0 * ladder["M"] * ladder["N"] * ladder["K"]
    ladder_ms = sum(ladder_ms) / len(ladder_ms)
    t_ms = sum(x["ms"] for x in ops)
    gemm_ms = sum(x["ms"] for x in ops if x["kind"] in ("gemm", "oz_gemm", "oz_split"))
    int8_ms = sum(x["ms"] for x in ops if x["kind"] in ("oz_gemm", "oz_split"))

    # ---- end-to-end leg: host (pinned numpy) buffers through the reference-facing API.  As in the solver loop
    # (Solver_GS.py:683-705) the amplitudes a step receives are arrays the class itself handed out earlier, so their
    # device copies are reused (GCC._to_dev); fsp — rebuilt on the host from the rdm1 every iteration — and the singles
    # are uploaded every step, every result is downloaded every step.
    h = {k: cc.to_numpy(x) for k, x in (("t1", t1), ("t2", t2), ("l1", l1), ("l2", l2))}
    h["t1"], h["l1"] = h["t1"].copy(), h["l1"].copy()          # small: plain host arrays, uploaded per call
    h["fsp"] = fsp.cpu().numpy()

    def step_host():
        g = cc.gamma(h["t1"], h["t2"], h["l1"], h["l2"])
        e = cc.energy(h["t1"], h["t2"], h["fsp"])
        a, b = cc.tupdate(h["t1"], h["t2"], fsp=h["fsp"], alpha=alpha)
        c, d = cc.lupdate(h["t1"], h["t2"], h["l1"], h["l2"], fsp=h["fsp"], alpha=alpha)
        return g, e, a, b, c, d

    e2e_steps = max(1, min(args.steps, 5))
    keep = step_host()
    keep = step_host()          # two generations of pinned result blocks exist from here on (cudaHostAlloc: ~1 s per 2 GB)
    del keep                    # ... and are back in the object's pool: the timed loop allocates nothing
    cc.h2d_bytes = cc.d2h_bytes = cc.h2d_reused = 0
    cc.host_seconds = {k: 0.0 for k in cc.host_seconds}
    ms_e2e, _ = timed(step_host, e2e_steps, 1)
    host_ms = {k: 1e3 * val / (e2e_steps + 1) for k, val in cc.host_seconds.items()}
    h2d = cc.h2d_bytes // (e2e_steps + 1)
    d2h = cc.d2h_bytes // (e2e_steps + 1)
    h2d_reused = cc.h2d_reused // (e2e_steps + 1)
    # the same with every input uploaded (arrays the class has never seen): the round-1 protocol, kept for comparison
    cold = {k: np_copy(x) for k, x in h.items()}

    def step_cold():
        cc.gamma(cold["t1"], cold["t2"], cold["l1"], cold["l2"])
        cc.energy(cold["t1"], cold["t2"], cold["fsp"])
        cc.tupdate(cold["t1"], cold["t2"], fsp=cold["fsp"], alpha=alpha)
        cc.lupdate(cold["t1"], cold["t2"], cold["l1"], cold["l2"], fsp=cold["fsp"], alpha=alpha)

    ms_cold, _ = timed(step_cold, 1, 1)
    del cold

    # ---- the solver loop itself, device resident (ecw_cc_b200.Solver_CCSD mirrors Solver_GS.Solver_CCSD.SCF): per
    # iteration gamma -> Vexp('mat') on the host (n x n) -> energy -> tupdate -> lupdate -> convergence vector
    import numpy as np
    from ecw_cc_b200.exp_pot import Exp
    rng = np.random.default_rng(7)
    pert = 0.02 * rng.standard_normal((n, n))
    target = np.diag(np.concatenate([np.ones(o), np.zeros(v)])) + 0.5 * (pert + pert.T)
    # One iteration per SCF call (maxiter=0) from the synthetic amplitudes: the random integrals of this size are far
    # from a perturbative system (E_MP2 = -361), so the reference's quasi-Newton iteration blows up after an update and
    # would leave the antisymmetric (packed) path the value/e2e legs are measured on.
    solver = ecw.Solver_CCSD(cc, Exp(0.05, [[["mat", target]]]), conv_thres=0.0, maxiter=0,
                             tsini=t1, lsini=l1, tdini=t2, ldini=l2)
    solver_calls = max(1, min(args.steps, 3))

    def solver_run():
        return solver.SCF(0.05, alpha=alpha, return_device=True)

    ms_solver, sout = timed(solver_run, solver_calls, 1)
    solver_iters = solver_calls

    per_step = 0
    if world > 1 and de.own_nccl:
        # collectives per step: count them over one more step
        before = lib.ecw_ctx_nccl_ops(de._h)
        step_dev()
        torch.cuda.synchronize()
        per_step = lib.ecw_ctx_nccl_ops(de._h) - before
    # what the line needs from the container (cheap; before it may be dropped)
    gh, gc = ctypes.c_int64(0), ctypes.c_int64(0)
    lib.ecw_ctx_graph_stats(de._h, ctypes.byref(gh), ctypes.byref(gc))
    graph_stats = {"replays": gh.value, "captures": gc.value,
                   "note": "one GPU: a call whose plan and pointer arguments were seen before is one cudaGraphLaunch of the "
                           "same kernels (include/ecw_b200.h, ecw_ctx_set_graphs); gpu_launches counts the kernels"}
    anti = alpha is None
    launches = sum(cc.plan_launches(f, alpha, False, anti) for f in ("tupdate", "lupdate"))
    launches += cc.plan_launches("gamma") + cc.plan_launches("energy") + 3   # + antisymmetry checks
    exec_flops = (cc.plan_flops("tupdate", alpha, False, anti) + cc.plan_flops("lupdate", alpha, False, anti)
                  + cc.plan_flops("gamma") + cc.plan_flops("energy"))
    own_nccl = de.own_nccl
    # BASELINE.json configs[4] beside the 8-GPU line (or on request): the sharded vvvv ladder at (60, 800).  Every
    # measurement of the line itself is done: the (40,400) container and amplitudes go first (the ladder's shard of the
    # vvvv planes alone is 77 GB per rank at 8 GPUs).
    c5 = None
    if args.config5 or (world == 8 and (o, v) == (40, 400)):
        import gc as _gc
        solver = sout = cc = de = t1 = t2 = l1 = l2 = fsp = h = None
        _gc.collect()
        torch.cuda.empty_cache()
        c5 = config5_ladder(ecw, torch, dist, rank, world)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak = measure_fp64_peak(torch)
    evals_per_s = args.steps * world / (ms_dev / 1e3) if world == 1 else args.steps / (ms_dev / 1e3)
    e2e_per_s = e2e_steps / (ms_e2e / 1e3)
    fp64_equiv = ladder_flops / ladder_ms / 1e9
    if ladder["kind"] == "oz_gemm":
        # the dominant launch runs on the INT8 tensor pipe: ns(ns+1)/2 int8 products per FP64 product
        nprod = ns * (ns + 1) // 2
        mp = {}
        try:
            mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        traffic = ncu_traffic(o, v, world)      # only a capture of this shape and GPU count counts
        # the ladder is timed inside the step (per-op events between back-to-back launches): the SUSTAINED figure is the
        # denominator the measurement rules name for that; the burst-based fraction is reported next to it.  The INT8
        # rate itself is MEASURED in this run (cuBLASLt int8 GEMM), not derived from the bf16 figure.
        bf16_burst = float(mp.get("bf16_tflops", 0.0))
        bf16 = float(mp.get("bf16_tflops_sustained", 0.0)) or bf16_burst
        i8 = measure_int8_peak(torch)
        int8_peak = i8["burst_tops"]       # the conservative denominator: this kernel beats cuBLASLt's sustained rate
        roofline = {"bound": "tensor",
                    "kernel": "ecw::ozaki_gemm_kernel<%d> (tcgen05.mma kind::i8, TMEM accumulators), launch = packed "
                              "pp-ladder %dx%dx%d (CCSD.py:305)" % (ns, ladder["M"], ladder["N"], ladder["K"]),
                    "achieved": fp64_equiv * nprod, "peak": int8_peak, "unit": "TOP/s",
                    "unit_note": "dense int8 tensor ops (2 per multiply-add): the TFLOP/s of a kernel whose operands "
                                 "are int8 digits; the FP64-equivalent rate is in fp64_equivalent_tflops",
                    "frac": fp64_equiv * nprod / int8_peak,
                    "traffic": (traffic or {}).get("bytes_per_launch"), "traffic_detail": traffic,
                    "frac_vs_sustained_peak": fp64_equiv * nprod / i8["sustained_tops"],
                    "peak_source": "INT8 dense GEMM rate of this GPU measured in this run with cuBLASLt (%s): burst "
                                   "%.0f TOP/s (the peak used here), sustained %.0f TOP/s (the launch is timed inside a "
                                   "long power-capped step, where it runs faster than cuBLASLt's own sustained rate); "
                                   "for comparison 2 x MEASURED_PEAKS.json bf16 = %.0f (sustained) / %.0f (burst), "
                                   "nominal 4500" % (i8["how"], i8["burst_tops"], i8["sustained_tops"], 2.0 * bf16,
                                                     2.0 * bf16_burst),
                    "int8_peak_measured": i8,
                    "int8_products_per_fp64_product": nprod,
                    "fp64_equivalent_tflops": fp64_equiv, "cublas_dgemm_tflops_measured": peak,
                    "fp64_equivalent_over_fp64_tensor_peak": fp64_equiv / peak,
                    "launch_ms": ladder_ms, "launch_flops": ladder_flops,
                    "gemm_share_of_tupdate": gemm_ms / t_ms, "int8_share_of_tupdate": int8_ms / t_ms}
    else:
        roofline = {"bound": "tensor",
                    "kernel": "ecw::dgemm_tma_kernel (FP64 DMMA), launch = packed pp-ladder %dx%dx%d (CCSD.py:305)"
                              % (ladder["M"], ladder["N"], ladder["K"]),
                    "achieved": fp64_equiv, "peak": peak, "unit": "TFLOP/s",
                    "frac": fp64_equiv / peak, "traffic": None,
                    "peak_source": "cuBLAS DGEMM 8192^3 (torch.matmul fp64) measured in this run, burst; "
                                   "MEASURED_PEAKS.json has no FP64 entry; nominal FP64 tensor peak %.0f TFLOP/s"
                                   % NOMINAL_FP64_TFLOPS,
                    "launch_ms": ladder_ms, "launch_flops": ladder_flops,
                    "gemm_share_of_tupdate": gemm_ms / t_ms}
    line = {
        "metric": METRIC, "value": evals_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "synthetic spin-orbital CCSD T+Lambda residual (gamma+energy+tupdate+lupdate), "
                               "nocc=%d nvir=%d FP64" % (o, v),
                   "nocc": o, "nvir": v, "alpha": alpha, "parallelism": "1 GPU" if world == 1 else "vshard%d" % world,
                   "collectives": None if world == 1 else (
                       ("ncclAllGather / grouped ncclSend+ncclRecv enqueued by the library's executor on its own "
                        "communicator, %d per step" % per_step) if own_nccl else "torch.distributed (host-driven)"),
                   "gemm_engine": ("int8 tcgen05 (%d digits) for the large GEMMs, FP64 DMMA for the rest" % ns) if ns
                   else "FP64 DMMA",
                   "l2_policy": "inputs larger than L2 (the packed vvvv, %.1f GB, is streamed every step)"
                                % ((ns if ns else 8) * (v * (v - 1) // 2) ** 2 / 1e9),
                   "fp64_tensor_peak_measured_tflops": peak,
                   "tflops_alg_over_fp64_tensor_peak": f_alg(o, v) * evals_per_s / 1e12 / peak,
                   "f_alg_flops_per_eval": f_alg(o, v), "executed_gemm_flops_per_eval": exec_flops,
                   "tflops_alg": f_alg(o, v) * evals_per_s / 1e12, "tflops_executed": exec_flops * evals_per_s / 1e12},
        "clocks": clocks,
        "e2e": {"value": e2e_per_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "h2d_bytes_reused_per_step": int(h2d_reused), "download_ms_per_step": host_ms,
                "protocol": "GCC.gamma/energy/tupdate/lupdate with numpy arrays in and out; the doubles amplitudes are "
                            "arrays the class handed out (as in Solver_CCSD.SCF, where each step's amplitudes are the "
                            "previous step's results), so their device copies are reused; fsp, t1, l1 are uploaded and "
                            "all results downloaded every step",
                "all_inputs_uploaded": {"value": 1e3 / ms_cold, "h2d_bytes_per_step": int(6 * 8 * o * o * v * v),
                                        "note": "every amplitude a fresh host array (round-1 protocol), 1 step"}},
        "solver_loop": {"value": solver_iters / (ms_solver / 1e3), "unit": "iterations/s",
                        "h2d_bytes_per_iteration": 0, "d2h_bytes_per_iteration": 32,
                        "what": "ecw_cc_b200.Solver_CCSD.SCF (mirror of Solver_GS.Solver_CCSD.SCF) with "
                                "ecw_cc_b200.exp_pot.Exp ('mat' target): the same iteration with the amplitudes, the "
                                "rdm1, the experimental potential and the dressed Fock resident on the GPU; only "
                                "Delta, vmax, the energy and the convergence distance (4 doubles) cross PCIe"},
        "parts": parts,
        "cuda_graphs": graph_stats,
        "gpu_launches": int(launches * args.steps),
        "roofline": roofline,
    }
    if c5 is not None:
        line["config5"] = c5
    if world == 1:
        try:
            line["parts_ccs"] = time_ccs(ecw, torch)
        except Exception as exc:
            line["parts_ccs"] = {"error": repr(exc)[:200]}
    if not args.no_cpu and world == 1:
        # this repo's path at the CPU shapes first (GPU still warm), then the CPU leg itself on the host cores
        line["cpu_baseline"] = cpu_baseline(o, v, same_shape_gpu(ecw, torch, CPU_SHAPES))
    sys.stdout.flush()
    os.write(out_fd, (json.dumps(line) + "\n").encode())
    os.close(out_fd)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nocc", type=int, default=40)
    ap.add_argument("--nvir", type=int, default=400)
    ap.add_argument("--alpha", type=float, default=None, help="L1 coefficient (default: none, as Main.CCSD_GS)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config5", action="store_true", help="add the sharded (60,800) vvvv ladder as extra key config5 (default: at 8 GPUs)")
    ap.add_argument("--gemm", default=None, choices=["int8", "dmma"], help="GEMM engine (default: int8)")
    ap.add_argument("--int8-digits", type=int, default=None, help="base-256 digits of the INT8 engine (default: from the integral magnitudes, 6 for the benchmark)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rdm1, energy, T1/T2 and L1/L2 updates) as DIR/<name>.npy, "
                         "float64; outputs above %d elements as a fixed seeded sample of it (64 MB at most in all)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps this repo's path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
