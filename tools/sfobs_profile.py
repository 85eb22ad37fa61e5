"""Timing of the amplitude target ('Fobs') on one GPU: the build of the symmetrised, smeared AO-pair planes
(`ecw_ft_aopair_cryst`) and one iteration of the device potential (`ecw_vexp_sfobs`), with CUDA events after warm-up.

Shape: decane/cc-pVDZ (nao = 250, the molecule of tools/sf_profile.py) with random orthonormal MOs, anisotropic ADPs on
every atom, in a monoclinic 20 x 12 x 10 Angstrom cell (beta = 105 degrees) at N_h = 1000 and 5000 (the lowest-angle
reflections) and nsym = 1 (P1), 4 (P2_1/c) and 8 (C2/c).  The planes have the layout of 'F', 2 N_h nao^2 doubles, so the
per-iteration cost should not depend on nsym; the build should cost about nsym times the single-operation build.
Also checks that two builds give identical bits, and times `ecw_vexp_sf` on the same planes for comparison.

Usage: python tools/sfobs_profile.py [--nh 1000 5000] [--nsym 1 4 8] [--reps 20] [--out FILE]   (needs a CUDA device)"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np

from sf_profile import decane, gpu_info

CELL = (20.0, 12.0, 10.0, 90.0, 105.0, 90.0)
P21C = ['x,y,z', '-x,y+1/2,-z+1/2', '-x,-y,-z', 'x,-y+1/2,z+1/2']
C2C = ['x,y,z', '-x,y,-z+1/2', '-x,-y,-z', 'x,-y,z+1/2']
OPS = {1: ['x,y,z'], 4: P21C,
       8: C2C + ['x+1/2,y+1/2,z', '-x+1/2,y+1/2,-z+1/2', '-x+1/2,-y+1/2,-z', 'x+1/2,-y+1/2,z+1/2']}


def lowest_reflections(crystal, n):
    r = 16
    hkl = np.array([(h, k, l) for h in range(-r, r + 1) for k in range(-r, r + 1) for l in range(-r, r + 1)])
    s = np.linalg.norm(crystal.G(hkl), axis=1)
    order = np.argsort(s, kind="stable")
    from ecw_cc_b200 import molint
    return hkl[order[:n]], float(s[order[n - 1]] * molint.ANGSTROM / (4 * np.pi))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--nh", type=int, nargs="+", default=[1000, 5000])
    ap.add_argument("--nsym", type=int, nargs="+", default=[1, 4, 8])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import ecw_cc_b200 as ecw
    from ecw_cc_b200 import exp_pot, molint
    if not torch.cuda.is_available():
        raise SystemExit("sfobs_profile.py measures on the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    atoms = decane()
    mol = molint.Molecule(atoms, "cc-pvdz")
    nao = mol.nao
    rng = np.random.default_rng(0)
    q, _ = np.linalg.qr(rng.standard_normal((nao, nao)))
    C = np.zeros((2 * nao, 2 * nao))                             # G format: alpha rows / even columns, beta / odd
    C[:nao, 0::2], C[nao:, 1::2] = q, q
    n = 2 * nao
    x = 0.01 * rng.standard_normal((n, n))
    rdm1 = torch.from_numpy(np.diag((np.arange(n) < 2 * 41).astype(float)) + x + x.T).to(dev)
    fock = torch.from_numpy(np.diag(np.sort(rng.standard_normal(n)))).to(dev)
    adp = []
    for _ in atoms:
        y = 0.05 * rng.standard_normal((3, 3))
        adp.append(0.01 * np.eye(3) + y @ y.T)
    header = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": gpu_info(), "molecule": "C10H22/cc-pVDZ",
              "nao": nao, "nprim": len(mol.ex), "n_spin_orbitals": n, "cell": CELL, "adp": "anisotropic, every atom"}
    print(json.dumps(header), flush=True)
    results = [header]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    stream = torch.cuda.current_stream(dev).cuda_stream

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(reps):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / reps

    for nh in args.nh:
        for nsym in args.nsym:
            cr = molint.Crystal(CELL, OPS[nsym], adp)
            hkl, s_max = lowest_reflections(cr, nh)
            a = np.abs(rng.standard_normal(nh)) + 0.1
            sigma = 0.05 + 0.05 * rng.uniform(size=nh)
            plane_bytes = 2 * nh * nao * nao * 8
            # build: warm-up, then timed calls (each includes the host tables and their upload)
            exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
            torch.cuda.synchronize()
            t_build = []
            for _ in range(3):
                ev[0].record()
                ft = exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
                ev[1].record()
                torch.cuda.synchronize()
                t_build.append(ev[0].elapsed_time(ev[1]))
            again = exp_pot.ft_aopair_cryst_device(mol, cr, hkl, dev)
            identical = bool(torch.equal(ft, again))
            del again, ft
            # one iteration: the first fobs_update_device builds and keeps the planes, then raw calls
            vx = exp_pot.Exp(0.1, [[['Fobs', a, sigma, hkl, cr]]], mol, C)
            vx.fobs_update_device(rdm1, fock)
            st = vx._fobs_dev
            fsp = torch.empty_like(rdm1)

            def one_obs():
                rc = ecw.lib.ecw_vexp_sfobs(rdm1.data_ptr(), n, st["C"].data_ptr(), nao, st["ft"].data_ptr(), nh,
                                            st["F_obs"].data_ptr(), st["w"].data_ptr(), 0.0, 0.1, fock.data_ptr(),
                                            st["vexp"].data_ptr(), fsp.data_ptr(), st["F_calc"].data_ptr(),
                                            st["stats"].data_ptr(), st["ws"].data_ptr(), stream)
                if rc != 0:
                    raise RuntimeError("ecw_vexp_sfobs failed")
            F_exp = torch.zeros((2, nh), dtype=torch.float64, device=dev)
            stats2 = torch.zeros(2, dtype=torch.float64, device=dev)

            def one_sf():                                   # ecw_vexp_sf on the same planes and workspace
                rc = ecw.lib.ecw_vexp_sf(rdm1.data_ptr(), n, st["C"].data_ptr(), nao, st["ft"].data_ptr(), nh,
                                         F_exp.data_ptr(), 0.1, fock.data_ptr(), st["vexp"].data_ptr(), fsp.data_ptr(),
                                         st["F_calc"].data_ptr(), stats2.data_ptr(), st["ws"].data_ptr(), stream)
                if rc != 0:
                    raise RuntimeError("ecw_vexp_sf failed")
            t_obs, t_sf = [], []
            for _ in range(3):                              # alternate the two calls
                t_obs.append(timed(one_obs, args.reps))
                t_sf.append(timed(one_sf, args.reps))
            r = {"n_h": nh, "nsym": nsym, "max_sin_theta_over_lambda": round(s_max, 4), "plane_bytes": plane_bytes,
                 "ft_cryst_build_ms": sorted(t_build)[1], "ft_cryst_build_ms_all": t_build,
                 "ft_cryst_bit_identical": identical, "vexp_sfobs_ms": sorted(t_obs)[1], "vexp_sfobs_ms_all": t_obs,
                 "vexp_sf_same_planes_ms": sorted(t_sf)[1], "vexp_sf_same_planes_ms_all": t_sf,
                 "vexp_sfobs_plane_GBps": 2 * plane_bytes / (sorted(t_obs)[1] * 1e-3) / 1e9,
                 "k": float(st["stats"][2]), "chi2": float(st["stats"][3])}
            print(json.dumps(r), flush=True)
            results.append(r)
            del vx, st
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
