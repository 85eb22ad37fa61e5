"""Device-resident mirror of the reference ground-state solver `Solver_GS.Solver_CCSD`
(Solver_GS.py:522-742): same constructor and `SCF` signatures, same iteration order, same convergence bookkeeping
(Q7: `Dconv` stays 1.0 on iteration 0; divergence threshold 1.0) and the same return tuple — but the o^2v^2 amplitudes
never leave the GPU.  With `ecw_cc_b200.exp_pot.Exp` and a single density-matrix target (what `Main.CCSD_GS` fits), or a
single structure-factor or amplitude target, the potential and the dressed Fock matrix are formed on the device too
(`ecw_vexp_mat`, `ecw_vexp_sf`, `ecw_vexp_sfobs`) and only scalars cross PCIe; with
any other `VX_exp` object (e.g. the unchanged reference `exp_pot.Exp`, exp_pot.py:131-345) the rdm1 (n x n) goes to the
host once per iteration and the dressed Fock comes back.  The convergence vector and its norm are formed on the device
(`ecw_conv_check`).

The reference loop driven through the numpy API of `GCC` moves 16 GB over PCIe per iteration at (40,400); this loop
moves 3 MB.  DIIS (Solver_GS.py:666-674, 683-686, 709-718) is provided by `ecw_cc_b200.diis.DIIS`: 'tl' extrapolates
the amplitude sets on the device (history in HBM, only the Gram row comes to the host), 'rdm1' the n x n rdm1 on the
host.  `pyscf.lib.diis` is not part of the reference tree, so DIIS-accelerated runs are pinned to the restatement of its
published algorithm (parity unpinned against PySCF itself, SURVEY §8c); the default is diis='' as in `Main.CCSD_GS` (Q5).
"""
import numpy as np

from ._lib import lib, EcwError
from .diis import DIIS


class Solver_CCSD(object):
    def __init__(self, mycc, VX_exp, conv='tl', conv_thres=10 ** -6, tsini=None, lsini=None, tdini=None, ldini=None,
                 diis='', maxiter=40, maxdiis=15):
        """mycc: `ecw_cc_b200.GCC`; VX_exp: object with `Vexp_update(rdm1, rdm1_add, index, L=)` and `Vexp[0, 0]`
        (the reference's `exp_pot.Exp`).  Other parameters as in the reference (Solver_GS.py:523-538)."""
        import torch
        self.torch = torch
        self.nocc = mycc.nocc
        self.nvir = mycc.nvir
        self.fock = mycc.fock
        self.mycc = mycc
        self.myVexp = VX_exp
        dev = mycc.eris.device
        o, v = self.nocc, self.nvir

        def up(x, shape):
            if x is None:
                return None
            if isinstance(x, torch.Tensor):
                return x.to(dev).reshape(shape).contiguous()
            return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64).reshape(shape)).to(dev)

        self.tsini = up(tsini, (o, v)) if tsini is not None else torch.zeros((o, v), dtype=torch.float64, device=dev)
        self.lsini = up(lsini, (o, v)) if lsini is not None else torch.zeros((o, v), dtype=torch.float64, device=dev)
        if tdini is None:                                  # MP2 start (Solver_GS.py:554-559), formed on the device
            ops = mycc._dev_ops()
            oovv = mycc._oovv
            tdini = ops.denom(oovv, oovv)                  # oovv / (e_i - e_a + e_j - e_b), bare Fock (amp unused)
            ldini = tdini.clone()
        self.tdini = up(tdini, (o, o, v, v))
        self.ldini = up(ldini, (o, o, v, v)) if ldini is not None else self.tdini.clone()
        self.diis = diis
        self.maxdiis = maxdiis
        self.maxiter = maxiter
        self.conv_thres = conv_thres
        if conv not in ('Ep', 'l', 'tl'):
            raise ValueError('Accepted convergence parameter is Ep, l or tl')
        self.conv = conv
        self._scratch = torch.zeros(1024 + 1, dtype=torch.float64, device=dev)

    # -- convergence (Solver_GS.py:591-612): the vector lives on the device, only its distance comes back ------------
    def _conv_distance(self, new, old, ts, ls, td, ld):
        """Fill `new` = [conv(singles) | conv(doubles)] and return ||new - old||_2 (None when old is None)."""
        torch = self.torch
        st = self.mycc.eris.stream()
        n1, n2 = ts.numel(), td.numel()
        sumsq = self._scratch[1024:]
        pairs = ((ls, ts, 0, n1), (ld, td, n1, n2))
        for k, (l, t, off, n) in enumerate(pairs):
            b = t.data_ptr() if self.conv == 'tl' else None
            prev = old.data_ptr() + 8 * off if old is not None else None
            rc = lib.ecw_conv_check(l.data_ptr(), b, prev, new.data_ptr() + 8 * off, n, self._scratch.data_ptr(),
                                    sumsq.data_ptr(), 1 if k else 0, st)
            if rc != 0:
                raise EcwError("ecw_conv_check failed")
        if old is None:
            return None
        return float(torch.sqrt(sumsq)[0].cpu())

    def SCF(self, L, ts=None, ls=None, td=None, ld=None, alpha=None, diis='', return_device=False):
        """Same loop as Solver_GS.py:621-742.  Returns (text, Ep(it), (Delta, vmax)(it), conv(it), last rdm1,
        [ts, ls, td, ld]) with numpy arrays (torch CUDA tensors for the amplitudes when return_device)."""
        torch = self.torch
        if diis is None:                                   # Q5 (Solver_GS.py:648-649): only None selects self.diis
            diis = self.diis
        mycc, VXexp = self.mycc, self.myVexp
        dev = mycc.eris.device
        o, v = self.nocc, self.nvir

        def up(x, shape):
            if isinstance(x, torch.Tensor):
                return x.to(dev).reshape(shape).contiguous()
            return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64).reshape(shape)).to(dev)

        if ts is None:
            ts, ls = self.tsini, self.lsini
        if td is None:
            td, ld = self.tdini, self.ldini
        ts, ls, td, ld = up(ts, (o, v)), up(ls, (o, v)), up(td, (o, o, v, v)), up(ld, (o, o, v, v))

        nconv = ts.numel() + td.numel()
        conv_new = torch.empty(nconv, dtype=torch.float64, device=dev)
        conv_old = torch.empty(nconv, dtype=torch.float64, device=dev)
        have_old = False
        ep_old = 0.
        Dconv = 1.0
        ite = 0
        conv_ite, Delta_ite, Ep_ite = [], [], []
        rdm1 = []
        Conv_text = ''
        adiis = tl_diis = None
        if 'rdm1' in diis:                                 # Solver_GS.py:666-674
            adiis = DIIS()
            adiis.space, adiis.min_space = self.maxdiis, 2
        if 'tl' in diis:
            tl_diis = DIIS(mycc._dev_ops())
            tl_diis.space, tl_diis.min_space = self.maxdiis, 2
        # a single density-matrix target (ecw_vexp_mat), structure-factor target (ecw_vexp_sf) or amplitude target
        # (ecw_vexp_sfobs) of our own Exp class is evaluated on the device: then nothing but scalars crosses PCIe inside
        # the loop.  Any other potential object, and DIIS on the rdm1, take the host route.
        dev_update = None
        if adiis is None:
            if getattr(VXexp, "device_mat_ready", lambda: False)():
                dev_update = VXexp.mat_update_device
            elif getattr(VXexp, "device_sf_ready", lambda: False)():
                dev_update = VXexp.sf_update_device
            elif getattr(VXexp, "device_fobs_ready", lambda: False)():
                dev_update = VXexp.fobs_update_device
        on_device = dev_update is not None
        fock_dev = mycc.eris.fock_dev if on_device else None
        rdm1_dev = None
        while Dconv > self.conv_thres:
            if on_device:
                rdm1_dev = mycc.gamma(ts, td, ls, ld)
                Delta, vmax, fsp = dev_update(rdm1_dev, fock_dev, L=L)
            else:
                rdm1 = mycc.gamma(ts, td, ls, ld).cpu().numpy()                   # n x n to the host
                if adiis is not None:
                    rdm1 = adiis.update(rdm1)
                Delta, vmax = VXexp.Vexp_update(rdm1, rdm1, (0, 0), L=L)
                fsp_h = np.subtract(self.fock, VXexp.Vexp[0, 0])
                fsp = torch.from_numpy(np.ascontiguousarray(fsp_h, dtype=np.float64)).to(dev)
            Delta_ite.append((Delta, vmax))
            Ep_ite.append(float(mycc.energy(ts, td, fsp)))
            ts, td = mycc.tupdate(ts, td, fsp=fsp, alpha=alpha)
            ls, ld = mycc.lupdate(ts, td, ls, ld, fsp=fsp, alpha=alpha)
            if tl_diis is not None:
                ls, ts, ld, td = tl_diis.update([ls, ts, ld, td])
            if self.conv == 'Ep':
                ep = float(mycc.energy(ts, td, fsp))
                if ite > 0:
                    Dconv = abs(ep - ep_old)
                ep_old = ep
            else:
                d = self._conv_distance(conv_new, conv_old if have_old else None, ts, ls, td, ld)
                if ite > 0:
                    Dconv = d
                conv_new, conv_old = conv_old, conv_new
                have_old = True
            conv_ite.append(Dconv)
            if ite >= self.maxiter:
                Conv_text = 'Max iteration reached'
                break
            if Dconv > 1.0:
                Conv_text = 'Diverges for lambda = {} after {} iterations'.format(L, ite)
                break
            ite += 1
        else:
            Conv_text = 'Convergence reached for lambda= {} and alpha={}, after {} iteration'.format(L, alpha, ite)
        if on_device:
            rdm1 = rdm1_dev.cpu().numpy() if rdm1_dev is not None else []
            VXexp.sync_host()
        amps = [ts, ls, td, ld]
        if not return_device:
            amps = [a.cpu().numpy() for a in amps]
        return Conv_text, np.asarray(Ep_ite), np.asarray(Delta_ite), np.asarray(conv_ite), rdm1, amps
