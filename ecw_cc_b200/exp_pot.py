"""Host-side mirror of the reference `exp_pot.Exp` (exp_pot.py:11-490): the experimental potentials Vexp[n, m] that
dress the Fock matrix of the ECW fit, their relative deviations Delta, and the weight check.

Targets (exp_pot.py:131-345): 'mat' (ground or excited state rdm1), 'trmat' (left/right transition rdm1), 'Ek', 'v1e',
'dip' (state properties), 'DEk..' (kinetic-energy difference to the ground state, acts on Vexp[0, 0]) and 'trdip'
(squared transition dipole, acts on Vexp[0, n] / Vexp[n, 0]), 'F' (X-ray structure factors, any diagonal state) and
'Fobs' (measured X-ray amplitudes of a unit cell, any diagonal state).
Property targets take their AO integrals from `mol`, which may be a PySCF `Mole` or `ecw_cc_b200.molint.Molecule` (same
`intor_symmetric` / `with_common_orig` / `atom_charges` / `atom_coords`); 'F' and 'Fobs' need a `molint.Molecule`.

'F' = ['F', F_exp, hkl, cell]: N_h structure factors (complex, or real = phase 0), integer Miller indices [N_h, 3] and
orthorhombic cell lengths (a, b, c) in Angstrom; G_h = 2 pi (h/a, k/b, l/c).  The reference's own 'F' branch needs PySCF
and is not pinned; the target is defined by the penalty it minimises, P = (w/2) sum_h |F_exp(h) - F_calc(h)|^2 with
F_calc(h) = sum_mu,nu D_mu,nu A_mu,nu(G_h), A = `molint.ft_aopair` (exp(+i G.r)), D = C_g rdm1 C_g^T spin-summed.  The
potential is -dP/drdm1 = w sum_h Re[conj(dF_h) C_g^T blockdiag(A_h, A_h) C_g]: on purpose NOT the `convert_aoint`
convention (C^-1 A C^-T, |diff|) of the other property targets, since there is no reference behaviour to mirror and the
fit needs the true gradient.  Delta = sum_h |dF_h| / sum_h |F_exp(h)| (HF_prop: / sum_h |F_exp - F_HF|), vmax =
max |V_F|, and ['F', F_calc] goes to `prop_calc`.

'Fobs' = ['Fobs', F_obs, sigma, hkl, crystal] or [..., crystal, k]: measured amplitudes.  F_obs: N_h non-negative
|F_obs|; sigma: N_h positive standard uncertainties or None (unit weights), w_h = 1/sigma_h^2; hkl: integer [N_h, 3];
crystal: a `molint.Crystal` (general cell with G_h = 2 pi M^-T h, symmetry operations x' = R x + t in fractional
coordinates that generate the distinct copies of the molecule in the cell, centring included, and Cartesian ADPs per
atom, Angstrom^2; Z' = 1).  The planes are
    B_mu,nu(h) = sum_s exp(+2 pi i h.t_s) T_mu,nu(G_{h_s}) A_mu,nu(G_{h_s}),   h_s = R_s^T h,
T_mu,nu(G) = (T_A(G) + T_B(G)) / 2 for mu on atom A and nu on atom B, T_A(G) = exp(-G^T U_A G / 2): exact for one-centre
pairs (Debye-Waller factor of a rigidly displaced atom), a convention for two-centre pairs; the ADP of a symmetry copy
rotates with it because T is evaluated at G_{h_s}.  F_calc(h) = sum D_mu,nu B_mu,nu(h) (`molint.ft_aopair_cryst`).
Scale k: refined (default) k = argmin chi^2 = sum w |F_o| |F_c| / sum w |F_c|^2, N_p = 1, N_h >= 2; or fixed by the
optional sixth element (positive), N_p = 0.  P = L chi^2, chi^2 = sum_h w_h (k |F_c| - |F_o|)^2 / (N_h - N_p) (on
purpose not the (L/2) sum of 'F': L stays comparable across data sets and chi^2 ~ 1 is the usual stopping point).  The
potential is -dP/drdm1 at fixed k (dP/dk = 0 at the refined k): sum_h Re[conj(c_h) C_g^T blockdiag(B_h, B_h) C_g],
c_h = 2 L k / (N_h - N_p) w_h (|F_o| - k |F_c|) F_c / |F_c|, and c_h = 0 where |F_c| <= 1e-12 max_h |F_c|
(`molint.FOBS_ZERO`): |F| has a cusp at 0, and a reflection that a point symmetry of the density extinguishes has an
F_c of rounding noise whose direction must not steer the fit.  Delta = R1 = sum |k|F_c| - |F_o|| /
sum |F_o| (HF_prop: the target's entry holds F_HF, complex or amplitudes, and the denominator is
sum |k_HF |F_HF| - |F_o||, k_HF the HF amplitudes' own refined scale or the fixed k), vmax = max |V|, and
['Fobs', F_calc (complex, unscaled), k, chi^2] goes to `prop_calc`.

Scope: the 'mat' ground-state target is part of the product (SURVEY §8 f-2; `mat_update_device`, `ecw_vexp_mat`),
and so are the 'F' ground-state target (`sf_update_device`, `ecw_ft_aopair`, `ecw_vexp_sf`) and the 'Fobs' one
(`fobs_update_device`, `ecw_ft_aopair_cryst`, `ecw_vexp_sfobs`).
The other targets are n x n host code kept as test HARNESS (callers of the path, SURVEY §2 "out of scope"): they let the
excited-state configuration of BASELINE.json be driven on a box without PySCF, and are pinned to the reference class
in tests/test_exp_pot_cpu.py.

n x n work on the host, except for the case `Main.CCSD_GS` runs — one density-matrix target for the ground state —
which `mat_update_device` evaluates on the GPU (`ecw_vexp_mat`), and one structure-factor target for the ground state,
which `sf_update_device` evaluates there (`ecw_ft_aopair` builds the AO-pair planes once, `ecw_vexp_sf` forms the
potential per iteration): the device-resident solver (`ecw_cc_b200.Solver_CCSD`)
then moves only scalars per iteration; for every other target it sends the rdm1 (n x n) to the host once per iteration
and takes the dressed Fock back (3 MB of PCIe traffic per iteration at (40,400)).
"""
import numpy as np

from . import molint, utilities


class Exp(object):
    def __init__(self, L, exp_data, mol=None, mo_coeff=None, Ek_exp_GS=None, Ek_HF_GS=None, HF_prop=False):
        """Same signature as the reference (exp_pot.py:11).  exp_data = [[GS targets], [ES1 targets], ...], a target
        being ['mat', rdm1], ['trmat', (left, right)], ['Ek', x], ['v1e', x], ['dip', [x, y, z]], ['trdip', [x, y, z]],
        ['DEk..', x], ['F', F_exp, hkl, cell], ['Fobs', F_obs, sigma, hkl, crystal(, k)]; mo_coeff in spin-orbital (G)
        format; HF_prop in the layout of exp_data
        switches Delta to the deviation relative to |exp - HF|."""
        self.nbr_states = len(exp_data)
        self.exp_data = exp_data
        self.mol, self.mo_coeff = mol, mo_coeff
        self.prop_calc = []
        self.HF_prop = HF_prop if HF_prop else [[None for _ in st] for st in exp_data]
        self.Ek_HF_GS = Ek_HF_GS
        self.L = self.L_check(L)
        self.charge_center = None
        self.Ek_int = self.dip_int = self.v1e_int = self.F_int = None
        self.dic_int = {}
        self.prop_names = []
        self.sf = {}                                                # 'F' data per (state, target index)
        for k, st in enumerate(exp_data):
            for i, prop in enumerate(st):
                name = prop[0]
                if name == 'F':
                    self.sf[k, i] = self._sf_setup(prop, mol, mo_coeff, self.HF_prop[k][i])
                    continue
                if name == 'Fobs':
                    self.sf[k, i] = self._fobs_setup(prop, mol, mo_coeff, self.HF_prop[k][i])
                    continue
                if name not in ('mat', 'trmat') and mol is None:
                    raise ValueError("target %r needs AO integrals: pass mol (PySCF Mole or molint.Molecule)" % (name,))
                if 'dip' in name and self.dip_int is None:          # 'dip' and 'trdip' (exp_pot.py:90-98)
                    charges, coords = mol.atom_charges(), mol.atom_coords()
                    self.charge_center = np.einsum('z,zr->r', charges, coords) / charges.sum()
                    with mol.with_common_orig(self.charge_center):
                        self.dip_int = mol.intor_symmetric('int1e_r', comp=3)
                    self.dic_int['dip'] = utilities.convert_aoint(self.dip_int, mo_coeff)
                if 'v1e' in name and self.v1e_int is None:          # exp_pot.py:101-104
                    self.v1e_int = mol.intor_symmetric('int1e_nuc')
                    self.dic_int['v1e'] = utilities.convert_aoint(self.v1e_int, mo_coeff)
                if 'Ek' in name and self.Ek_int is None:            # 'Ek' and 'DEk..' (exp_pot.py:107-110)
                    self.Ek_int = mol.intor_symmetric('int1e_kin')
                    self.dic_int['Ek'] = utilities.convert_aoint(self.Ek_int, mo_coeff)
            self.prop_names.append([prop[0] for prop in st])
        self.DEk_GS_idx = None                                      # weight slot of the GS 'DEk' target, if any
        for i, name in enumerate(self.prop_names[0] if self.prop_names else []):
            if 'DEk' in name:
                self.DEk_GS_idx = i
        self.Ek_exp_GS = Ek_exp_GS
        self.Ek_calc_GS = None
        self.Delta_Ek_GS = None
        self.Vexp = np.full((self.nbr_states, self.nbr_states), None)

    # -- the structure-factor target --------------------------------------------------------------------------------
    def _sf_setup(self, prop, mol, mo_coeff, hf):
        """Validate ['F', F_exp, hkl, cell] and derive the scattering vectors G_h = 2 pi (h/a, k/b, l/c) in bohr^-1.
        The AO-pair transforms are built on first use: on the host by `Vexp_update`, on the device by
        `sf_update_device`."""
        if mol is None or not isinstance(mol, molint.Molecule):
            raise NotImplementedError("the structure-factor target 'F' needs the AO pairs of an ecw_cc_b200.molint."
                                      "Molecule" + ("" if mol is None else " (a PySCF Mole is not supported)"))
        if len(prop) != 4:
            raise ValueError("the structure-factor target is ['F', F_exp, hkl, cell]")
        F_exp = np.asarray(prop[1])
        if F_exp.ndim != 1 or F_exp.size == 0 or not np.issubdtype(F_exp.dtype, np.number) \
                or not np.all(np.isfinite(F_exp)):
            raise ValueError("'F' target: F_exp must be a non-empty 1-D array of finite (real or complex) values")
        hkl = np.asarray(prop[2])
        if hkl.shape != (F_exp.size, 3) or not np.issubdtype(hkl.dtype, np.number) or not np.all(np.isfinite(hkl)) \
                or np.any(hkl != np.round(hkl)):
            raise ValueError("'F' target: hkl must be an (N_h, 3) array of integer Miller indices, N_h = len(F_exp)")
        cell = np.asarray(prop[3], dtype=np.float64)
        if cell.shape != (3,) or not np.all(np.isfinite(cell)) or np.any(cell <= 0):
            raise ValueError("'F' target: cell must be three positive orthorhombic cell lengths (a, b, c), Angstrom")
        if mo_coeff is None or np.shape(mo_coeff)[0] != 2 * mol.nao:
            raise ValueError("'F' target: mo_coeff in spin-orbital (G) format, [2 nao, n], is required")
        F_exp = F_exp.astype(np.complex128)
        G = 2 * np.pi * hkl.astype(np.float64) / cell / molint.ANGSTROM
        ref = F_exp if hf is None else F_exp - np.asarray(hf, dtype=np.complex128)
        return {"F_exp": F_exp, "G": G, "norm": float(np.sum(np.abs(ref))), "A": None}

    # -- the amplitude target -----------------------------------------------------------------------------------------
    @staticmethod
    def _fobs_scale(a, F_obs, w, k_fixed):
        """The scale k of |F_calc| = a: k_fixed, or the closed-form argmin of chi^2, sum w F_obs a / sum w a^2."""
        return k_fixed if k_fixed is not None else float(np.sum(w * F_obs * a) / np.sum(w * a * a))

    def _fobs_setup(self, prop, mol, mo_coeff, hf):
        """Validate ['Fobs', F_obs, sigma, hkl, crystal(, k)].  The symmetrised planes are built on first use: on the
        host by `Vexp_update`, on the device by `fobs_update_device`."""
        if mol is None or not isinstance(mol, molint.Molecule):
            raise NotImplementedError("the amplitude target 'Fobs' needs the AO pairs of an ecw_cc_b200.molint."
                                      "Molecule" + ("" if mol is None else " (a PySCF Mole is not supported)"))
        if len(prop) not in (5, 6):
            raise ValueError("the amplitude target is ['Fobs', F_obs, sigma, hkl, crystal] or [..., crystal, k]")
        F_obs = np.asarray(prop[1])
        if F_obs.ndim != 1 or F_obs.size == 0 or not np.issubdtype(F_obs.dtype, np.number) \
                or np.iscomplexobj(F_obs) or not np.all(np.isfinite(F_obs)) or np.any(F_obs < 0):
            raise ValueError("'Fobs' target: F_obs must be a non-empty 1-D array of finite, non-negative amplitudes")
        nh = F_obs.size
        if prop[2] is None:
            sigma = np.ones(nh)
        else:
            sigma = np.asarray(prop[2])
            if sigma.shape != (nh,) or not np.issubdtype(sigma.dtype, np.number) or np.iscomplexobj(sigma) \
                    or not np.all(np.isfinite(sigma)) or np.any(sigma <= 0):
                raise ValueError("'Fobs' target: sigma must be None or N_h finite positive values, N_h = len(F_obs)")
        hkl = np.asarray(prop[3])
        if hkl.shape != (nh, 3) or not np.issubdtype(hkl.dtype, np.number) or not np.all(np.isfinite(hkl)) \
                or np.any(hkl != np.round(hkl)):
            raise ValueError("'Fobs' target: hkl must be an (N_h, 3) array of integer Miller indices")
        crystal = prop[4]
        if not isinstance(crystal, molint.Crystal):
            raise ValueError("'Fobs' target: the fifth element must be an ecw_cc_b200.molint.Crystal")
        crystal.adp_bohr(len(mol.Z))                                # one ADP entry per atom
        k_fixed = None
        if len(prop) == 6:
            k = prop[5]
            if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, float, np.integer, np.floating)) \
                    or not np.isfinite(k) or k <= 0:
                raise ValueError("'Fobs' target: a fixed scale k must be a positive number")
            k_fixed = float(k)
        n_p = 0 if k_fixed is not None else 1
        if nh - n_p < 1:
            raise ValueError("'Fobs' target: a refined scale needs at least two reflections")
        if mo_coeff is None or np.shape(mo_coeff)[0] != 2 * mol.nao:
            raise ValueError("'Fobs' target: mo_coeff in spin-orbital (G) format, [2 nao, n], is required")
        F_obs = F_obs.astype(np.float64)
        w = 1.0 / sigma.astype(np.float64) ** 2
        if hf is None:
            norm = float(np.sum(F_obs))
        else:
            a_hf = np.abs(np.asarray(hf))
            if a_hf.shape != (nh,):
                raise ValueError("'Fobs' target: HF_prop must hold N_h HF structure factors or amplitudes")
            norm = float(np.sum(np.abs(self._fobs_scale(a_hf, F_obs, w, k_fixed) * a_hf - F_obs)))
        return {"F_obs": F_obs, "w": w, "hkl": hkl.astype(np.int64), "crystal": crystal, "k": k_fixed, "n_p": n_p,
                "norm": norm, "B": None}

    # -- weights (exp_pot.py:459-490) -------------------------------------------------------------------------------
    def L_check(self, L):
        if isinstance(L, (float, int)):
            return [[float(L)] * len(st) for st in self.exp_data]
        if isinstance(L, (list, np.ndarray)):
            if len(L) != self.nbr_states:
                raise SyntaxError('Given constrain weight length does not equal the number of states. '
                                  'You might have forgotten to put L_loop = True.')
            out = []
            for k, (st, l) in enumerate(zip(self.exp_data, L)):
                l = list(np.atleast_1d(l))
                if len(st) != len(l) and len(l) == 1:               # one weight for all targets of the state
                    l = l * len(st)
                elif len(st) != len(l):
                    raise SyntaxError("Wrong syntax for L list")
                out.append(l)
            return out
        raise SyntaxError('L must be a number or a list with one entry per state')

    # -- <A> and <A>_nm <A>_mn (exp_pot.py:347-390) -----------------------------------------------------------------
    def calc_prop(self, prop, rdm1, g_format=True, rdm1_add=None):
        fn, ints = {'Ek': (utilities.Ekin, self.Ek_int), 'v1e': (utilities.v1e, self.v1e_int),
                    'dip': (utilities.dipole, self.dip_int)}.get(prop, (None, None))
        if fn is None:
            raise NotImplementedError('The possible properties are: Ek, v1e and dip')
        one = fn(self.mol, rdm1, g_format, False, self.mo_coeff, ints)
        if rdm1_add is None:
            return list(one) if prop == 'dip' else one
        two = fn(self.mol, rdm1_add.transpose(), g_format, False, self.mo_coeff, np.conj(ints))
        return (list(one * two), list(two)) if prop == 'dip' else (one * two, two)

    # -- relative deviation (exp_pot.py:392-446) --------------------------------------------------------------------
    def Delta(self, n_st, i_prop, prop_diff, comp_idx=1, threshold=10 ** -6):
        exp = self.exp_data[n_st][i_prop][1]
        hf = self.HF_prop[n_st][i_prop]
        if isinstance(prop_diff, np.ndarray) and n_st == 0:        # ground-state density matrix
            ref = exp if hf is None else exp - hf
            return np.sum(abs(prop_diff)) / np.sum(abs(ref))
        if isinstance(exp, list) and abs(exp[comp_idx]) > threshold:          # vector property, one component
            return prop_diff / np.abs(exp[comp_idx] if hf is None else exp[comp_idx] - hf[comp_idx])
        if isinstance(exp, float) and abs(exp) > threshold:                   # scalar property
            return prop_diff / np.abs(exp if hf is None else exp - hf)
        return 0.                                                   # incl. excited-state 'mat' (as in the reference)

    # -- Vexp[n, m] (exp_pot.py:131-345) ----------------------------------------------------------------------------
    def Vexp_update(self, rdm1, rdm1_add, index, L=None):
        n, m = index
        self.Vexp[n, m] = np.zeros_like(rdm1)
        Delta, vmax = 0., 0.
        self.prop_calc = []
        L = self.L if L is None else self.L_check(L)
        st = max(n, m)                                              # the state whose target list applies
        for i, name in enumerate(self.prop_names[st]):
            w = L[st][i]
            target = self.exp_data[st][i][1]
            if name == 'mat' and n == m:
                diff = np.subtract(target, rdm1)
                self.Vexp[n, n] += w * diff
                Delta += self.Delta(n, i, diff)
                vmax += np.max(abs(diff))
                if n == 0 and self.Ek_exp_GS is not None:           # kinetic energy of the fitted ground state
                    self.Ek_calc_GS = utilities.Ekin(self.mol, rdm1, aobasis=False, mo_coeff=self.mo_coeff,
                                                     ek_int=self.Ek_int, g=True)
                    ref = self.Ek_exp_GS if self.Ek_HF_GS is None else self.Ek_exp_GS - self.Ek_HF_GS
                    self.Delta_Ek_GS = np.abs(self.Ek_exp_GS - self.Ek_calc_GS) / np.abs(ref)
            if name == 'trmat' and n != m:
                print("WARNING: The use of experimental transition density matrix is not tested")
                if n != 0 and m != 0:
                    raise ValueError("Only transition properties between GS and ES are implemented: m or n must be = 0")
                diff = np.subtract(target[0] if n == 0 else target[1], rdm1)
                self.Vexp[n, m] += w * diff
                # the reference sums |target| over ROWS only (builtin sum), so Delta becomes a vector here
                avg = np.sum(abs(target[1]), axis=0) + np.sum(abs(target[0]), axis=0)
                Delta += np.sum(abs(diff)) / (avg / 2.)
                vmax += np.max(abs(diff))
            if name in ('Ek', 'v1e') and n == m:
                calc = self.calc_prop(name, rdm1)
                diff = np.abs(target - calc)
                Delta += self.Delta(n, i, diff)
                diff = diff * self.dic_int[name]
                self.Vexp[n, n] += w * diff
                vmax += np.max(abs(diff))
                self.prop_calc.append([name, calc])
            if 'DEk' in name and n == m and n != 0:                 # -ES rdm1 + GS rdm1; feeds the GS potential
                calc = self.calc_prop('Ek', np.subtract(rdm1_add, rdm1))
                diff = np.abs(target - calc)
                Delta += self.Delta(st, i, diff)
                diff = diff * self.dic_int['Ek']
                if self.Vexp[0, 0] is None:
                    self.Vexp[0, 0] = 0.
                self.Vexp[0, 0] += (L[0][self.DEk_GS_idx] if self.DEk_GS_idx is not None else w) * diff
                vmax += np.max(np.abs(diff))
                self.prop_calc.append([name, calc])
            if name == 'dip' and n == m:
                calc = self.calc_prop('dip', rdm1)
                for j in range(3):
                    diff = np.abs(target[j] - calc[j])
                    Delta += self.Delta(st, i, diff, comp_idx=j)
                    diff = diff * self.dic_int['dip'][j]
                    self.Vexp[n, m] += w * diff
                    vmax += np.max(np.abs(diff))
                self.prop_calc.append([name, calc])
            if name == 'trdip' and n != m:
                calc, scale = self.calc_prop('dip', rdm1, rdm1_add=rdm1_add)
                for j in range(3):
                    diff = np.abs(target[j] - calc[j])
                    Delta += self.Delta(st, i, diff, comp_idx=j)
                    diff = diff * (self.dic_int['dip'][j] * scale[j])
                    self.Vexp[n, m] += w * diff
                    vmax += np.max(np.abs(diff))
                self.prop_calc.append([name, calc])
            if name == 'F' and n == m:
                sf = self.sf[st, i]
                if sf["A"] is None:
                    sf["A"] = molint.ft_aopair(self.mol, sf["G"])
                A, C = sf["A"], self.mo_coeff
                nao = A.shape[1]
                D = utilities.convert_g_to_ru_rdm1(C @ rdm1 @ C.T)[0]
                calc = np.einsum('hij,ij->h', A, D)
                dF = sf["F_exp"] - calc
                v_ao = w * np.einsum('h,hij->ij', np.conj(dF), A).real
                diff = C[:nao].T @ v_ao @ C[:nao] + C[nao:].T @ v_ao @ C[nao:]
                self.Vexp[n, n] += diff
                Delta += np.sum(np.abs(dF)) / sf["norm"]
                vmax += np.max(np.abs(diff))
                self.prop_calc.append([name, calc])
            if name == 'Fobs' and n == m:
                sf = self.sf[st, i]
                if sf["B"] is None:
                    sf["B"] = molint.ft_aopair_cryst(self.mol, sf["crystal"], sf["hkl"])
                B, C = sf["B"], self.mo_coeff
                nao = B.shape[1]
                D = utilities.convert_g_to_ru_rdm1(C @ rdm1 @ C.T)[0]
                calc = np.einsum('hij,ij->h', B, D)
                a, F_obs, wt = np.abs(calc), sf["F_obs"], sf["w"]
                k = self._fobs_scale(a, F_obs, wt, sf["k"])
                dof = len(a) - sf["n_p"]
                r = F_obs - k * a
                chi2 = float(np.sum(wt * r * r) / dof)
                unit = np.divide(calc, a, out=np.zeros_like(calc), where=a > molint.FOBS_ZERO * a.max())
                c = (2 * w * k / dof) * wt * r * unit
                v_ao = np.einsum('h,hij->ij', np.conj(c), B).real
                diff = C[:nao].T @ v_ao @ C[:nao] + C[nao:].T @ v_ao @ C[nao:]
                self.Vexp[n, n] += diff
                Delta += np.sum(np.abs(k * a - F_obs)) / sf["norm"]
                vmax += np.max(np.abs(diff))
                self.prop_calc.append([name, calc, k, chi2])
        return Delta, vmax

    # -- the 'mat' ground-state target without leaving the GPU (SURVEY §8f-2) ------------------------------------------
    def device_mat_ready(self):
        """True when Vexp[0, 0] is exactly one density-matrix target (what `Main.CCSD_GS` fits): then the potential and
        the dressed Fock matrix can be formed on the device by `mat_update_device`."""
        return bool(self.prop_names) and self.prop_names[0] == ['mat'] and self.Ek_exp_GS is None

    def mat_update_device(self, rdm1_dev, fock_dev, L=None):
        """Device version of `Vexp_update(rdm1, rdm1, (0, 0), L)` + `fsp = fock - Vexp[0, 0]` (exp_pot.py:185-195,
        Solver_GS.py:690-692) through `ecw_vexp_mat`: returns (Delta, vmax, fsp) with fsp a device tensor; only the two
        reduction results (16 bytes) come to the host.  `self.Vexp[0, 0]` holds the DEVICE potential afterwards; call
        `sync_host()` to turn it into the numpy array the host path leaves there."""
        import torch
        from ._lib import lib, EcwError
        if not self.device_mat_ready():
            raise EcwError("mat_update_device needs a single 'mat' ground-state target")
        L = self.L if L is None else self.L_check(L)
        dev = rdm1_dev.device
        st = getattr(self, "_dev", None)
        if st is None or st["device"] != dev:
            target = np.ascontiguousarray(self.exp_data[0][0][1], dtype=np.float64)
            hf = self.HF_prop[0][0]
            st = {"device": dev, "target": torch.from_numpy(target).to(dev),
                  "norm": float(np.sum(abs(target if hf is None else target - hf))),
                  "vexp": torch.empty_like(rdm1_dev), "stats": torch.zeros(2, dtype=torch.float64, device=dev)}
            self._dev = st
        if tuple(rdm1_dev.shape) != tuple(st["target"].shape) or not rdm1_dev.is_contiguous():
            raise ValueError("rdm1 must be a contiguous device matrix of the target's shape")
        fsp = torch.empty_like(rdm1_dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.ecw_vexp_mat(rdm1_dev.data_ptr(), st["target"].data_ptr(), fock_dev.data_ptr(), float(L[0][0]),
                              st["vexp"].data_ptr(), fsp.data_ptr(), st["stats"].data_ptr(), rdm1_dev.numel(), stream)
        if rc != 0:
            raise EcwError("ecw_vexp_mat failed")
        self.Vexp[0, 0] = st["vexp"]
        self.prop_calc = []
        s = st["stats"].cpu()
        return float(s[0]) / st["norm"], float(s[1]), fsp

    # -- the structure-factor ground-state target without leaving the GPU ---------------------------------------------
    def device_sf_ready(self):
        """True when Vexp[0, 0] is exactly one structure-factor target: then `sf_update_device` forms the potential and
        the dressed Fock matrix on the device."""
        return bool(self.prop_names) and self.prop_names[0] == ['F'] and self.Ek_exp_GS is None

    def sf_update_device(self, rdm1_dev, fock_dev, L=None):
        """Device version of `Vexp_update(rdm1, rdm1, (0, 0), L)` + `fsp = fock - Vexp[0, 0]` for one 'F' target through
        `ecw_vexp_sf`: returns (Delta, vmax, fsp) with fsp a device tensor; only the two reduction results come to the
        host.  The first call builds the AO-pair planes on the device (`ecw_ft_aopair`, 2 N_h nao^2 doubles) and
        uploads mo_coeff; both stay there.  Afterwards `self.Vexp[0, 0]` holds the DEVICE potential and `prop_calc`
        the device F_calc ([2, N_h]: Re, Im); `sync_host()` turns both into what the host path leaves there."""
        import torch
        from ._lib import lib, EcwError
        if not self.device_sf_ready():
            raise EcwError("sf_update_device needs a single 'F' ground-state target")
        L = self.L if L is None else self.L_check(L)
        dev = rdm1_dev.device
        sf = self.sf[0, 0]
        C = np.ascontiguousarray(self.mo_coeff, dtype=np.float64)
        nao, n = C.shape[0] // 2, C.shape[1]
        nG = len(sf["G"])
        st = getattr(self, "_sf_dev", None)
        if st is None or st["device"] != dev:
            ws = lib.ecw_vexp_sf_workspace_bytes(n, nao, nG)
            if ws < 0:
                raise EcwError("ecw_vexp_sf_workspace_bytes failed")
            fe = np.stack([sf["F_exp"].real, sf["F_exp"].imag])
            st = {"device": dev, "ft": ft_aopair_device(self.mol, sf["G"], dev), "C": torch.from_numpy(C).to(dev),
                  "F_exp": torch.from_numpy(np.ascontiguousarray(fe)).to(dev),
                  "vexp": torch.empty((n, n), dtype=torch.float64, device=dev),
                  "F_calc": torch.empty((2, nG), dtype=torch.float64, device=dev),
                  "stats": torch.zeros(2, dtype=torch.float64, device=dev),
                  "ws": torch.empty((ws + 7) // 8, dtype=torch.float64, device=dev)}
            self._sf_dev = st
        for x in (rdm1_dev, fock_dev):
            if tuple(x.shape) != (n, n) or not x.is_contiguous() or x.dtype != torch.float64 or x.device != dev:
                raise ValueError("rdm1 and fock must be contiguous float64 (n, n) matrices on one device, n = mo_coeff "
                                 "columns")
        fsp = torch.empty_like(rdm1_dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.ecw_vexp_sf(rdm1_dev.data_ptr(), n, st["C"].data_ptr(), nao, st["ft"].data_ptr(), nG,
                             st["F_exp"].data_ptr(), float(L[0][0]), fock_dev.data_ptr(), st["vexp"].data_ptr(),
                             fsp.data_ptr(), st["F_calc"].data_ptr(), st["stats"].data_ptr(), st["ws"].data_ptr(),
                             stream)
        if rc != 0:
            raise EcwError("ecw_vexp_sf failed")
        self.Vexp[0, 0] = st["vexp"]
        self.prop_calc = [['F', st["F_calc"]]]
        s = st["stats"].cpu()
        return float(s[0]) / sf["norm"], float(s[1]), fsp

    # -- the amplitude ground-state target without leaving the GPU ----------------------------------------------------
    def device_fobs_ready(self):
        """True when Vexp[0, 0] is exactly one amplitude target: then `fobs_update_device` forms the potential and the
        dressed Fock matrix on the device."""
        return bool(self.prop_names) and self.prop_names[0] == ['Fobs'] and self.Ek_exp_GS is None

    def fobs_update_device(self, rdm1_dev, fock_dev, L=None):
        """Device version of `Vexp_update(rdm1, rdm1, (0, 0), L)` + `fsp = fock - Vexp[0, 0]` for one 'Fobs' target
        through `ecw_vexp_sfobs`: returns (Delta, vmax, fsp) with fsp a device tensor; only the four statistics come to
        the host.  The first call builds the symmetrised planes on the device (`ecw_ft_aopair_cryst`, 2 N_h nao^2
        doubles) and uploads mo_coeff, F_obs and the weights; all stay there.  Afterwards `self.Vexp[0, 0]` holds the
        DEVICE potential and `prop_calc` = [['Fobs', F_calc, k, chi^2]] device tensors (F_calc [2, N_h]: Re, Im);
        `sync_host()` turns them into what the host path leaves there."""
        import torch
        from ._lib import lib, EcwError
        if not self.device_fobs_ready():
            raise EcwError("fobs_update_device needs a single 'Fobs' ground-state target")
        L = self.L if L is None else self.L_check(L)
        dev = rdm1_dev.device
        sf = self.sf[0, 0]
        C = np.ascontiguousarray(self.mo_coeff, dtype=np.float64)
        nao, n = C.shape[0] // 2, C.shape[1]
        nG = len(sf["F_obs"])
        st = getattr(self, "_fobs_dev", None)
        if st is None or st["device"] != dev:
            ws = lib.ecw_vexp_sfobs_workspace_bytes(n, nao, nG)
            if ws < 0:
                raise EcwError("ecw_vexp_sfobs_workspace_bytes failed")
            st = {"device": dev, "ft": ft_aopair_cryst_device(self.mol, sf["crystal"], sf["hkl"], dev),
                  "C": torch.from_numpy(C).to(dev), "F_obs": torch.from_numpy(sf["F_obs"]).to(dev),
                  "w": torch.from_numpy(sf["w"]).to(dev),
                  "vexp": torch.empty((n, n), dtype=torch.float64, device=dev),
                  "F_calc": torch.empty((2, nG), dtype=torch.float64, device=dev),
                  "stats": torch.zeros(4, dtype=torch.float64, device=dev),
                  "ws": torch.empty((ws + 7) // 8, dtype=torch.float64, device=dev)}
            self._fobs_dev = st
        for x in (rdm1_dev, fock_dev):
            if tuple(x.shape) != (n, n) or not x.is_contiguous() or x.dtype != torch.float64 or x.device != dev:
                raise ValueError("rdm1 and fock must be contiguous float64 (n, n) matrices on one device, n = mo_coeff "
                                 "columns")
        fsp = torch.empty_like(rdm1_dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.ecw_vexp_sfobs(rdm1_dev.data_ptr(), n, st["C"].data_ptr(), nao, st["ft"].data_ptr(), nG,
                                st["F_obs"].data_ptr(), st["w"].data_ptr(), 0.0 if sf["k"] is None else sf["k"],
                                float(L[0][0]), fock_dev.data_ptr(), st["vexp"].data_ptr(), fsp.data_ptr(),
                                st["F_calc"].data_ptr(), st["stats"].data_ptr(), st["ws"].data_ptr(), stream)
        if rc != 0:
            raise EcwError("ecw_vexp_sfobs failed")
        self.Vexp[0, 0] = st["vexp"]
        self.prop_calc = [['Fobs', st["F_calc"], st["stats"][2], st["stats"][3]]]
        s = st["stats"].cpu()
        return float(s[0]) / sf["norm"], float(s[1]), fsp

    def sync_host(self):
        """Replace a device-resident Vexp[0, 0] (and a device F_calc, k or chi^2 in `prop_calc`) by numpy copies."""
        v = self.Vexp[0, 0]
        if v is not None and not isinstance(v, np.ndarray) and hasattr(v, "cpu"):
            self.Vexp[0, 0] = v.cpu().numpy()
        for pc in self.prop_calc:
            if pc[0] in ('F', 'Fobs') and not isinstance(pc[1], np.ndarray) and hasattr(pc[1], "cpu"):
                f = pc[1].cpu().numpy()
                pc[1] = f[0] + 1j * f[1]
            if pc[0] == 'Fobs':
                pc[2], pc[3] = (float(x.cpu()) if hasattr(x, "cpu") else x for x in pc[2:4])


def ft_aopair_device(mol, G, device):
    """`molint.ft_aopair(mol, G)` on the GPU (`ecw_ft_aopair`): a float64 tensor [2, nG, nao, nao] holding the real
    and imaginary planes.  G: [nG, 3] scattering vectors in bohr^-1."""
    import torch
    from ._lib import lib, EcwError
    G = np.ascontiguousarray(np.atleast_2d(np.asarray(G, dtype=np.float64)))
    if G.ndim != 2 or G.shape[1] != 3 or len(G) == 0:
        raise ValueError("G must be a non-empty [nG, 3] array of scattering vectors")
    ao = np.asarray(mol.ao)
    if np.any(np.diff(ao) < 0) or ao[0] != 0 or ao[-1] != mol.nao - 1:
        raise ValueError("the primitives of each AO must be contiguous (molint.Molecule.ao non-decreasing)")
    if np.any(mol.lmn > 2) or np.any(mol.lmn < 0):
        raise ValueError("ecw_ft_aopair takes Cartesian powers up to 2 per direction (s, p, d)")
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: ecw_ft_aopair has no CPU implementation (molint.ft_aopair is the host path)")
    prim = np.ascontiguousarray(np.concatenate([mol.cen, mol.ex[:, None], mol.coef[:, None], mol.lmn], axis=1),
                                dtype=np.float64)
    ao_first = np.searchsorted(ao, np.arange(mol.nao + 1)).astype(np.int64)
    t_prim, t_first, t_G = (torch.from_numpy(x).to(device) for x in (prim, ao_first, G))
    out = torch.empty((2, len(G), mol.nao, mol.nao), dtype=torch.float64, device=device)
    rc = lib.ecw_ft_aopair(t_prim.data_ptr(), len(prim), t_first.data_ptr(), mol.nao, t_G.data_ptr(), len(G),
                           out.data_ptr(), torch.cuda.current_stream(out.device).cuda_stream)
    if rc != 0:
        raise EcwError("ecw_ft_aopair failed")
    return out


def ft_aopair_cryst_device(mol, crystal, hkl, device):
    """`molint.ft_aopair_cryst(mol, crystal, hkl)` on the GPU (`ecw_ft_aopair_cryst`): a float64 tensor
    [2, N_h, nao, nao] holding the real and imaginary planes.  The rotated vectors and phases per (h, s) are tabulated
    here by `Crystal.tables`, the same numbers the host path uses."""
    import torch
    from ._lib import lib, EcwError
    hkl = np.asarray(hkl)
    if hkl.ndim != 2 or hkl.shape[1] != 3 or len(hkl) == 0 or np.any(hkl != np.round(hkl)):
        raise ValueError("hkl must be a non-empty (N_h, 3) array of integer Miller indices")
    if not 1 <= crystal.nsym <= 192:
        raise ValueError("ecw_ft_aopair_cryst takes 1 to 192 symmetry operations")
    ao = np.asarray(mol.ao)
    if np.any(np.diff(ao) < 0) or ao[0] != 0 or ao[-1] != mol.nao - 1:
        raise ValueError("the primitives of each AO must be contiguous (molint.Molecule.ao non-decreasing)")
    if np.any(mol.lmn > 2) or np.any(mol.lmn < 0):
        raise ValueError("ecw_ft_aopair_cryst takes Cartesian powers up to 2 per direction (s, p, d)")
    U = crystal.adp_bohr(len(mol.Z))
    if not torch.cuda.is_available():
        raise EcwError("no CUDA device: ecw_ft_aopair_cryst has no CPU implementation (molint.ft_aopair_cryst is the "
                       "host path)")
    Gs, phase = crystal.tables(hkl)
    U6 = np.ascontiguousarray(U[:, [0, 1, 2, 0, 0, 1], [0, 1, 2, 1, 2, 2]])       # xx, yy, zz, xy, xz, yz
    prim = np.ascontiguousarray(np.concatenate([mol.cen, mol.ex[:, None], mol.coef[:, None], mol.lmn], axis=1),
                                dtype=np.float64)
    ao_first = np.searchsorted(ao, np.arange(mol.nao + 1)).astype(np.int64)
    t_prim, t_first, t_atom, t_U, t_G, t_ph = (
        torch.from_numpy(np.ascontiguousarray(x)).to(device)
        for x in (prim, ao_first, mol.ao_atom.astype(np.int64), U6, Gs, phase))
    out = torch.empty((2, len(hkl), mol.nao, mol.nao), dtype=torch.float64, device=device)
    rc = lib.ecw_ft_aopair_cryst(t_prim.data_ptr(), len(prim), t_first.data_ptr(), t_atom.data_ptr(), mol.nao,
                                 t_U.data_ptr(), len(U6), t_G.data_ptr(), t_ph.data_ptr(), crystal.nsym, len(hkl),
                                 out.data_ptr(), torch.cuda.current_stream(out.device).cuda_stream)
    if rc != 0:
        raise EcwError("ecw_ft_aopair_cryst failed")
    return out
