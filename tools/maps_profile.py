"""Timing of the density maps on one GPU: `ecw_density_grid` (AO values, one FP64 GEMM and a row-dot per chunk of
points) and `ecw_fourier_map` (direct Fourier synthesis), with CUDA events after warm-up.

Shapes: decane/cc-pVDZ (nao = 250, the molecule of tools/sf_profile.py) with a random symmetric AO density on the
default 80^3 box of `maps.box` and on a 160^3 box; Fourier maps of N_h = 1000 / 5000 unique reflections (the lowest-angle
orbits that are not systematically absent, in the monoclinic 20 x 12 x 10 Angstrom cell of tools/sfobs_profile.py)
expanded with nsym = 4 (P2_1/c) and 8 (C2/c) on a 96^3 cell grid; each unique reflection of these groups gives two
reflections of the half set.  Algorithmic work: the density needs 2 nao^2 + 2 nao flops per point (X = Phi D and the
row-dot) plus one exp per primitive and point; the synthesis 16 flops per (reflection of the half set, grid point)
(two complex products of the per-axis phase factors and the two-term update).  Also checks that two calls give
identical bits.  The timed calls are the C entry points on device-resident inputs; the host expansion of the unique
data (`Crystal.expand`) is timed separately with the host clock.

Usage: python tools/maps_profile.py [--reps 5] [--out FILE]   (needs a CUDA device)"""
import argparse
import ctypes
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np

from sf_profile import decane, gpu_info
from sfobs_profile import CELL, OPS


def unique_reflections(crystal, n, s_max=0.9):
    """The n lowest-angle orbits of reflections under {+-R_u^T} that are not systematically absent, one
    representative (the lexicographically largest member) each, and the sin(theta)/lambda of the last."""
    from ecw_cc_b200 import molint
    r = [int(np.ceil(2 * s_max * np.linalg.norm(crystal.M[:, d]))) + 1 for d in range(3)]
    hkl = np.stack([x.ravel() for x in np.meshgrid(*[np.arange(-m, m + 1) for m in r], indexing="ij")], axis=1)
    s = np.linalg.norm(crystal.G(hkl), axis=1) * molint.ANGSTROM / (4 * np.pi)
    order = np.argsort(s, kind="stable")
    reps, seen = [], set()
    for i in order[1:]:
        rep = max(tuple(int(x) for x in sg * (R.T @ hkl[i])) for R, _ in crystal.ops for sg in (1, -1))
        if rep not in seen:
            seen.add(rep)
            reps.append((rep, s[i]))
    hh, Fh, _ = crystal.expand(np.array([h for h, _ in reps]), np.ones(len(reps)))
    present = {tuple(h) for h, f in zip(hh, Fh) if abs(f) > 1e-9}
    reps = [(h, x) for h, x in reps if h in present][:n]
    assert len(reps) == n and reps[-1][1] < s_max
    return np.array([h for h, _ in reps]), float(reps[-1][1])


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import maps, molint
    if not torch.cuda.is_available():
        raise SystemExit("maps_profile.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    mol = molint.Molecule(decane(), "cc-pvdz")
    nao = mol.nao
    header = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": gpu_info(), "molecule": "C10H22/cc-pVDZ",
              "nao": nao, "nprim": len(mol.ex)}
    print(json.dumps(header), flush=True)
    results = [header]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            ev[0].record()
            for _ in range(reps):
                fn()
            ev[1].record()
            torch.cuda.synchronize()
            ts.append(ev[0].elapsed_time(ev[1]) / reps)
        return sorted(ts)[1], ts

    rng = np.random.default_rng(0)
    X = rng.standard_normal((nao, nao))
    D = (X + X.T) / nao
    prim, ao_first = maps._prim_table(mol)
    t_prim, t_first, t_dm = (torch.from_numpy(x).to(dev) for x in (prim, ao_first, D))
    for n in (80, 160):
        origin, axes, shape = maps.box(mol, n, n, n)
        npts = n ** 3
        out = torch.empty(shape, dtype=torch.float64, device=dev)
        ws = ecw.lib.ecw_density_grid_workspace_bytes(nao, npts)
        work = torch.empty((ws + 7) // 8, dtype=torch.float64, device=dev)
        box = (ctypes.c_double * 12)(*np.concatenate([origin, axes.ravel()]))

        def one(dst=out):
            rc = ecw.lib.ecw_density_grid(t_prim.data_ptr(), len(prim), t_first.data_ptr(), nao, t_dm.data_ptr(), box,
                                          n, n, n, dst.data_ptr(), work.data_ptr(), stream)
            if rc != 0:
                raise RuntimeError("ecw_density_grid failed")
        ms, all_ms = timed(one, args.reps)
        again = torch.empty_like(out)
        one(again)
        torch.cuda.synchronize()
        flops = npts * (2.0 * nao * nao + 2.0 * nao)
        r = {"kind": "density_grid", "shape": shape, "points": npts, "workspace_bytes": ws, "ms": ms, "ms_all": all_ms,
             "flops": flops, "TFLOPs": flops / (ms * 1e-3) / 1e12, "exp_per_s": npts * len(prim) / (ms * 1e-3),
             "bit_identical": bool(torch.equal(out, again))}
        print(json.dumps(r), flush=True)
        results.append(r)
        del out, again, work
        torch.cuda.empty_cache()

    shape = (96, 96, 96)
    npts = int(np.prod(shape))
    for nh in (1000, 5000):
        for nsym in (4, 8):
            cr = molint.Crystal(CELL, OPS[nsym])
            hkl, s_max = unique_reflections(cr, nh)
            F = rng.standard_normal(nh) + 1j * rng.standard_normal(nh)
            t0 = time.perf_counter()
            hh, Fh, F000 = cr.expand(hkl, F)
            t_expand = (time.perf_counter() - t0) * 1e3
            t_h = torch.from_numpy(np.ascontiguousarray(hh)).to(dev)
            t_c = torch.from_numpy(np.ascontiguousarray(np.stack([Fh.real, Fh.imag]))).to(dev)
            out = torch.empty(shape, dtype=torch.float64, device=dev)

            def one(dst=out):
                rc = ecw.lib.ecw_fourier_map(t_h.data_ptr(), t_c.data_ptr(), len(hh), F000, cr.volume_bohr3, *shape,
                                             dst.data_ptr(), stream)
                if rc != 0:
                    raise RuntimeError("ecw_fourier_map failed")
            ms, all_ms = timed(one, args.reps)
            again = torch.empty_like(out)
            one(again)
            torch.cuda.synchronize()
            terms = float(len(hh)) * npts
            r = {"kind": "fourier_map", "n_h_unique": nh, "nsym": nsym, "max_sin_theta_over_lambda": round(s_max, 4),
                 "n_half": len(hh), "shape": shape, "ms": ms, "ms_all": all_ms, "terms": terms,
                 "terms_per_s": terms / (ms * 1e-3), "flops": 16 * terms, "TFLOPs": 16 * terms / (ms * 1e-3) / 1e12,
                 "bit_identical": bool(torch.equal(out, again)), "host_expand_ms": t_expand}
            print(json.dumps(r), flush=True)
            results.append(r)
            del out, again
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
