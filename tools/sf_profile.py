"""Timing of the structure-factor ('F') target on one GPU: the build of the Fourier-transformed AO-pair planes
(`ecw_ft_aopair`) and one iteration of the device potential (`ecw_vexp_sf`), with CUDA events after warm-up.

Shape: decane (C10H22, all-trans, idealised geometry) in cc-pVDZ, nao = 250, with random orthonormal MOs (the timing
does not depend on them, and RHF at that size is not needed), at N_h = 1000 and 5000 reflections (the lowest-angle
reflections of a 20 x 12 x 10 Angstrom orthorhombic cell).  The planes are 2 N_h nao^2 doubles and one iteration reads
them twice (F_calc, then the potential); their size exceeds the 126 MB L2 at both N_h, so every pass reads HBM.

Usage: python tools/sf_profile.py [--nh 1000 5000] [--reps 20] [--out FILE]   (needs a CUDA device)"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def decane():
    """All-trans C10H22: C-C 1.54, C-H 1.09 Angstrom, tetrahedral angles."""
    cc, ch = 1.54, 1.09
    half = np.deg2rad(109.47 / 2)
    dx, dy = cc * np.sin(half), cc * np.cos(half) / 2
    atoms = []
    carbons = [np.array([i * dx, dy if i % 2 else -dy, 0.0]) for i in range(10)]
    for i, c in enumerate(carbons):
        atoms.append(("C", tuple(c)))
        out = np.array([0.0, 1.0 if i % 2 else -1.0, 0.0])     # the side away from the chain
        hs = [out * np.cos(np.deg2rad(54.75)) + s * np.array([0, 0, np.sin(np.deg2rad(54.75))]) for s in (1, -1)]
        if i in (0, 9):
            hs.append(np.array([-1.0 if i == 0 else 1.0, 0.0, 0.0]))
        for h in hs:
            atoms.append(("H", tuple(c + ch * h / np.linalg.norm(h))))
    return atoms


def lowest_reflections(cell, n):
    a, b, c = cell
    r = 16
    hkl = np.array([(h, k, l) for h in range(-r, r + 1) for k in range(-r, r + 1) for l in range(-r, r + 1)])
    s = 0.5 * np.sqrt((hkl[:, 0] / a) ** 2 + (hkl[:, 1] / b) ** 2 + (hkl[:, 2] / c) ** 2)
    order = np.argsort(s, kind="stable")
    return hkl[order[:n]], float(s[order[n - 1]])


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--nh", type=int, nargs="+", default=[1000, 5000])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import exp_pot, molint
    if not torch.cuda.is_available():
        raise SystemExit("sf_profile.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    mol = molint.Molecule(decane(), "cc-pvdz")
    nao = mol.nao
    rng = np.random.default_rng(0)
    q, _ = np.linalg.qr(rng.standard_normal((nao, nao)))
    C = np.zeros((2 * nao, 2 * nao))                             # G format: alpha rows / even columns, beta / odd
    C[:nao, 0::2], C[nao:, 1::2] = q, q
    n = 2 * nao
    x = 0.01 * rng.standard_normal((n, n))
    rdm1 = torch.from_numpy(np.diag((np.arange(n) < 2 * 41).astype(float)) + x + x.T).to(dev)
    fock = torch.from_numpy(np.diag(np.sort(rng.standard_normal(n)))).to(dev)
    cell = (20.0, 12.0, 10.0)
    header = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": gpu_info(), "molecule": "C10H22/cc-pVDZ",
              "nao": nao, "nprim": len(mol.ex), "n_spin_orbitals": n}
    print(json.dumps(header), flush=True)
    results = [header]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for nh in args.nh:
        hkl, s_max = lowest_reflections(cell, nh)
        G = 2 * np.pi * hkl / np.array(cell) / molint.ANGSTROM
        F_exp = rng.standard_normal(nh) * np.exp(1j * rng.uniform(0, 2 * np.pi, nh))
        plane_bytes = 2 * nh * nao * nao * 8
        # build of the planes: warm-up, then timed calls (each includes the upload of the 8 KB-sized primitive table)
        exp_pot.ft_aopair_device(mol, G, dev)
        torch.cuda.synchronize()
        t_build = []
        for _ in range(3):
            ev[0].record()
            ft = exp_pot.ft_aopair_device(mol, G, dev)
            ev[1].record()
            torch.cuda.synchronize()
            t_build.append(ev[0].elapsed_time(ev[1]))
        again = exp_pot.ft_aopair_device(mol, G, dev)
        identical = bool(torch.equal(ft, again))
        del again
        # one iteration of the potential: the first sf_update_device builds and keeps the planes, then raw calls
        vx = exp_pot.Exp(0.1, [[['F', F_exp, hkl, cell]]], mol, C)
        vx.sf_update_device(rdm1, fock)
        st = vx._sf_dev
        fsp = torch.empty_like(rdm1)
        stream = torch.cuda.current_stream(dev).cuda_stream

        def one():
            rc = ecw.lib.ecw_vexp_sf(rdm1.data_ptr(), n, st["C"].data_ptr(), nao, st["ft"].data_ptr(), nh,
                                     st["F_exp"].data_ptr(), 0.1, fock.data_ptr(), st["vexp"].data_ptr(),
                                     fsp.data_ptr(), st["F_calc"].data_ptr(), st["stats"].data_ptr(),
                                     st["ws"].data_ptr(), stream)
            if rc != 0:
                raise RuntimeError("ecw_vexp_sf failed")
        for _ in range(3):
            one()
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(args.reps):
            one()
        ev[1].record()
        torch.cuda.synchronize()
        t_iter = ev[0].elapsed_time(ev[1]) / args.reps
        # the same through the Python method (adds the 16-byte stats copy and its synchronisation)
        t0 = time.perf_counter()
        for _ in range(args.reps):
            vx.sf_update_device(rdm1, fock)
        torch.cuda.synchronize()
        t_py = (time.perf_counter() - t0) * 1e3 / args.reps
        r = {"n_h": nh, "max_sin_theta_over_lambda": round(s_max, 4), "plane_bytes": plane_bytes,
             "ft_build_ms": sorted(t_build)[1], "ft_build_ms_all": t_build, "ft_bit_identical": identical,
             "vexp_sf_ms": t_iter, "vexp_sf_bytes_read": 2 * plane_bytes,
             "vexp_sf_plane_GBps": 2 * plane_bytes / (t_iter * 1e-3) / 1e9, "sf_update_device_ms": t_py}
        print(json.dumps(r), flush=True)
        results.append(r)
        del vx, st, ft
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
