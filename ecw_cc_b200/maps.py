"""Electron-density maps of a fitted state: density cubes and Fourier (residual) maps on the GPU.

- `density_grid`: rho(r) = sum_mu,nu D_mu,nu phi_mu(r) phi_nu(r) (e/bohr^3) on the box grid r_ijk = origin + i a1 +
  j a2 + k a3 (bohr), stored [n1, n2, n3] with k fastest, the cube-file order (`ecw_density_grid`).  For a fitted state
  D = `utilities.convert_g_to_ru_rdm1(C_g @ rdm1 @ C_g.T)[0]`, the AO density of `exp_pot.Exp`.
- `fourier_map`: rho(x) = (1/V) sum_h F(h) exp(-2 pi i h.x) on the fractional grid x_ijk = (i/n1, j/n2, k/n3) of a
  `molint.Crystal`, from unique data expanded to the full sphere by `Crystal.expand` (`ecw_fourier_map`).
- `residual_map`: the Fourier synthesis of (|F_obs|/k - |F_calc|) F_calc/|F_calc| of a fitted 'Fobs' target, F000 = 0.
- `box` / `density`: the default box and the cube writer of PySCF's `cubegen.density`, for a `molint.Molecule`.
- `write_cube` / `read_cube`: Gaussian cube files.

The device functions raise `EcwError` without a CUDA device; there is no CPU fallback.  `molint.density_points` and
`molint.fourier_map` are the host references, for small grids.
"""
import ctypes

import numpy as np

from . import molint


def _shape3(shape):
    try:
        shape = tuple(int(n) for n in shape)
    except (TypeError, ValueError):
        raise ValueError("shape must be three positive grid dimensions")
    if len(shape) != 3 or min(shape) < 1:
        raise ValueError("shape must be three positive grid dimensions")
    return shape


def _prim_table(mol):
    """The primitive table of `ecw_ft_aopair` ([nprim, 8] = centre, exponent, coefficient, l) and ao_first [nao + 1]."""
    ao = np.asarray(mol.ao)
    if np.any(np.diff(ao) < 0) or ao[0] != 0 or ao[-1] != mol.nao - 1:
        raise ValueError("the primitives of each AO must be contiguous (molint.Molecule.ao non-decreasing)")
    if np.any(mol.lmn > 2) or np.any(mol.lmn < 0):
        raise ValueError("ecw_density_grid takes Cartesian powers up to 2 per direction (s, p, d)")
    prim = np.ascontiguousarray(np.concatenate([mol.cen, mol.ex[:, None], mol.coef[:, None], mol.lmn], axis=1),
                                dtype=np.float64)
    return prim, np.searchsorted(ao, np.arange(mol.nao + 1)).astype(np.int64)


def box(mol, nx=80, ny=80, nz=80, margin=3.0):
    """The box of `cubegen.density`: origin = min(atom coords) - margin, extent = max - min + 2 margin and step =
    extent / (n - 1) along each Cartesian axis (bohr).  Returns (origin [3], axes [3, 3] (rows a1, a2, a3), shape)."""
    shape = _shape3((nx, ny, nz))
    if min(shape) < 2:
        raise ValueError("a box needs at least two points per axis")
    if not np.isfinite(margin) or margin < 0:
        raise ValueError("margin must be a non-negative length in bohr")
    xyz = mol.atom_coords()
    origin = xyz.min(0) - margin
    extent = xyz.max(0) - xyz.min(0) + 2 * margin
    return origin, np.diag(extent / (np.array(shape) - 1.0)), shape


def cell_axes(crystal, shape):
    """Step vectors of the fractional grid of `crystal` in bohr, [3, 3]: row d is column d of M (bohr) / n_d."""
    shape = _shape3(shape)
    return (crystal.M * molint.ANGSTROM).T / np.array(shape, dtype=np.float64)[:, None]


def density_grid(mol, dm, origin, axes, shape, device):
    """rho on the box grid origin + i a1 + j a2 + k a3 (bohr; axes rows a1, a2, a3) as a float64 tensor [n1, n2, n3] on
    `device`, for the AO density dm [nao, nao] of the `molint.Molecule` mol (`ecw_density_grid`)."""
    import torch
    from ._lib import lib, EcwError
    shape = _shape3(shape)
    dm = np.ascontiguousarray(dm, dtype=np.float64)
    if dm.shape != (mol.nao, mol.nao) or not np.all(np.isfinite(dm)):
        raise ValueError("dm must be a finite (nao, nao) AO density matrix")
    b = np.concatenate([np.asarray(origin, dtype=np.float64).reshape(-1), np.asarray(axes, dtype=np.float64).reshape(-1)])
    if b.shape != (12,) or not np.all(np.isfinite(b)):
        raise ValueError("origin must be 3 and axes 3 x 3 finite values (bohr)")
    prim, ao_first = _prim_table(mol)
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: ecw_density_grid has no CPU implementation (molint.density_points is the "
                       "host reference)")
    npts = shape[0] * shape[1] * shape[2]
    ws = lib.ecw_density_grid_workspace_bytes(mol.nao, npts)
    if ws < 0:
        raise EcwError("ecw_density_grid_workspace_bytes failed")
    t_prim, t_first, t_dm = (torch.from_numpy(x).to(device) for x in (prim, ao_first, dm))
    out = torch.empty(shape, dtype=torch.float64, device=device)
    work = torch.empty((ws + 7) // 8, dtype=torch.float64, device=device)
    rc = lib.ecw_density_grid(t_prim.data_ptr(), len(prim), t_first.data_ptr(), mol.nao, t_dm.data_ptr(),
                              (ctypes.c_double * 12)(*b), shape[0], shape[1], shape[2], out.data_ptr(),
                              work.data_ptr(), torch.cuda.current_stream(out.device).cuda_stream)
    if rc != 0:
        raise EcwError("ecw_density_grid failed")
    return out


def synthesis(hkl_half, F_half, F000, volume_bohr3, shape, device):
    """`molint.fourier_synthesis` on the GPU (`ecw_fourier_map`): a float64 tensor [n1, n2, n3]."""
    import torch
    from ._lib import lib, EcwError
    shape = _shape3(shape)
    if max(shape) > 512:
        raise ValueError("ecw_fourier_map takes 1 to 512 grid points per axis")
    h = np.ascontiguousarray(np.asarray(hkl_half, dtype=np.int64).reshape(-1, 3))
    F = np.asarray(F_half, dtype=np.complex128).reshape(-1)
    if len(F) != len(h):
        raise ValueError("one coefficient per reflection of the half set")
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: ecw_fourier_map has no CPU implementation (molint.fourier_map is the host "
                       "reference)")
    out = torch.empty(shape, dtype=torch.float64, device=device)
    t_h = torch.from_numpy(h).to(device)
    t_c = torch.from_numpy(np.ascontiguousarray(np.stack([F.real, F.imag]))).to(device)
    rc = lib.ecw_fourier_map(t_h.data_ptr(), t_c.data_ptr(), len(h), float(F000), float(volume_bohr3), shape[0],
                             shape[1], shape[2], out.data_ptr(), torch.cuda.current_stream(out.device).cuda_stream)
    if rc != 0:
        raise EcwError("ecw_fourier_map failed")
    return out


def fourier_map(crystal, hkl, F, shape, device, group=None):
    """Fourier map (1/V) sum_h F(h) exp(-2 pi i h.x) in e/bohr^3 on the [n1, n2, n3] fractional grid of `crystal`, as
    a float64 tensor on `device`.  F: structure factors of the reflections hkl, expanded to the full sphere by
    `crystal.expand(hkl, F, group)` (equivalents and Friedel mates averaged; pass the full space group as `group` when
    the crystal lists only coset representatives).  F at (0, 0, 0), if given, is F000."""
    shape = _shape3(shape)
    if max(shape) > 512:
        raise ValueError("ecw_fourier_map takes 1 to 512 grid points per axis")
    hh, Fh, F000 = crystal.expand(hkl, F, group)
    return synthesis(hh, Fh, F000, crystal.volume_bohr3, shape, device)


def residual_coefficients(vexp, index=None):
    """(hkl, coefficients, crystal) of the residual map of an evaluated 'Fobs' target of the `exp_pot.Exp` vexp:
    c_h = (|F_obs|/k - |F_calc|) F_calc/|F_calc| from `prop_calc` (F_calc unscaled, k), c_h = 0 where |F_calc| <=
    `molint.FOBS_ZERO` max |F_calc| (the phase is undefined there), and (0, 0, 0) left out (F000 = 0).
    index: (state, target position) of the target; None takes the only 'Fobs' target."""
    keys = sorted(k for k, sf in vexp.sf.items() if "F_obs" in sf)
    if index is None:
        if len(keys) != 1:
            raise ValueError("residual_map: %d 'Fobs' targets; pass index=(state, target position)" % len(keys))
        index = keys[0]
    index = tuple(index)
    if index not in keys:
        raise ValueError("residual_map: exp_data[%d][%d] is not an 'Fobs' target" % index)
    st, i = index
    rank = [name for name in vexp.prop_names[st][:i]].count('Fobs')       # its place among the 'Fobs' results
    got = [pc for pc in vexp.prop_calc if pc[0] == 'Fobs']
    sf = vexp.sf[index]
    if len(got) <= rank:
        raise ValueError("residual_map: the 'Fobs' target has not been evaluated (run Vexp_update or a solver first)")
    pc = got[rank]
    if not isinstance(pc[1], np.ndarray) or not isinstance(pc[2], float):
        raise ValueError("residual_map: prop_calc holds device results; call vexp.sync_host() first")
    if pc[1].shape != sf["F_obs"].shape:
        raise ValueError("residual_map: the 'Fobs' target has not been evaluated (run Vexp_update or a solver first)")
    F_c, k = pc[1], pc[2]
    a = np.abs(F_c)
    unit = np.divide(F_c, a, out=np.zeros_like(F_c), where=a > molint.FOBS_ZERO * a.max())
    coef = (sf["F_obs"] / k - a) * unit
    keep = np.any(sf["hkl"] != 0, axis=1)
    return sf["hkl"][keep], coef[keep], sf["crystal"]


def residual_map(vexp, shape, device, index=None, group=None):
    """Residual density Delta rho = Fourier synthesis of (|F_obs|/k - |F_calc|) exp(i phi_calc) with F000 = 0, in
    e/bohr^3 on the [n1, n2, n3] fractional grid of the target's crystal, as a float64 tensor on `device`: the check
    that a fit has used up the signal in the data.  vexp: an `exp_pot.Exp` whose 'Fobs' target `Vexp_update` or a solver
    has evaluated (after `fobs_update_device`, call `vexp.sync_host()` first; `Solver_CCSD` does so when it finishes);
    index / group as for `residual_coefficients`
    and `fourier_map`.  Raises ValueError when there is no evaluated 'Fobs' target."""
    hkl, coef, crystal = residual_coefficients(vexp, index)
    return fourier_map(crystal, hkl, coef, shape, device, group)


def density(mol, outfile, dm, nx=80, ny=80, nz=80, margin=3.0):
    """Write the density of the AO density dm to the cube file outfile on the box of `cubegen.density` (same
    signature and box, computed on the current CUDA device).  Returns the values [nx, ny, nz]."""
    import torch
    from ._lib import EcwError
    origin, axes, shape = box(mol, nx, ny, nz, margin)
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: ecw_density_grid has no CPU implementation")
    rho = density_grid(mol, dm, origin, axes, shape, torch.device("cuda", torch.cuda.current_device())).cpu().numpy()
    write_cube(outfile, mol, origin, axes, rho, "Electron density in real space (e/Bohr^3)")
    return rho


def write_cube(path, mol, origin, axes, values, comment=''):
    """Gaussian cube file: two comment lines; natoms and the origin; per axis the count and the step vector (positive
    count: bohr); per atom Z, nuclear charge and position (bohr); the values '%13.5E', six per line and a line break
    after each k-row.  For a map of a unit cell pass origin 0 and `cell_axes(crystal, shape)`."""
    values = np.asarray(values, dtype=np.float64)
    origin = np.asarray(origin, dtype=np.float64).reshape(3)
    axes = np.asarray(axes, dtype=np.float64).reshape(3, 3)
    if values.ndim != 3:
        raise ValueError("values must be an [n1, n2, n3] grid")
    Z, xyz = mol.atom_charges(), mol.atom_coords()
    lines = [(comment.splitlines() or ["ecw_cc_b200 map"])[0],
             "values in e/bohr^3, lengths in bohr",
             "%5d%12.6f%12.6f%12.6f" % ((len(Z),) + tuple(origin))]
    lines += ["%5d%12.6f%12.6f%12.6f" % ((n,) + tuple(a)) for n, a in zip(values.shape, axes)]
    lines += ["%5d%12.6f%12.6f%12.6f%12.6f" % ((int(z), float(z)) + tuple(r)) for z, r in zip(Z, xyz)]
    n3 = values.shape[2]
    rows = values.reshape(-1, n3)
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
        for row in rows:
            for c0 in range(0, n3, 6):
                f.write("".join("%13.5E" % x for x in row[c0:c0 + 6]) + "\n")


def read_cube(path):
    """Read a Gaussian cube file.  Returns a dict: comment (two lines), origin [3] and axes [3, 3] in bohr, Z [natom],
    charge [natom], coords [natom, 3] in bohr, values [n1, n2, n3]."""
    with open(path) as f:
        text = f.read().split("\n")
    c1, c2 = text[0], text[1]
    head = text[2].split()
    natom, origin = int(head[0]), np.array([float(x) for x in head[1:4]])
    counts, axes = [], []
    for d in range(3):
        v = text[3 + d].split()
        counts.append(int(v[0]))
        axes.append([float(x) for x in v[1:4]])
    axes = np.array(axes)
    if any(n < 0 for n in counts):                              # negative count: Angstrom
        origin, axes = origin * molint.ANGSTROM, axes * molint.ANGSTROM
    counts = [abs(n) for n in counts]
    at = np.array([[float(x) for x in text[6 + a].split()[:5]] for a in range(natom)]).reshape(natom, 5)
    vals = np.array(" ".join(text[6 + natom:]).split(), dtype=np.float64)
    if vals.size != counts[0] * counts[1] * counts[2]:
        raise ValueError("cube file %s: %d values for a %d x %d x %d grid" % ((path, vals.size) + tuple(counts)))
    return {"comment": (c1, c2), "origin": origin, "axes": axes, "Z": at[:, 0].astype(int), "charge": at[:, 1],
            "coords": at[:, 2:5], "values": vals.reshape(counts)}
