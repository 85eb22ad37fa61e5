"""numpy restatement of the ground-state ECW-CCSD iteration — TEST INFRASTRUCTURE ONLY.

`ExpMat`  : the 'mat' branch of the reference's exp_pot.Exp (exp_pot.py:131-214, Delta :392-430, L_check :459-472):
            Vexp[0,0] = L (rdm1_exp - rdm1), Delta = sum|diff| / sum|rdm1_exp|, vmax = max|diff|.
`scf_loop`: Solver_GS.Solver_CCSD.SCF (Solver_GS.py:621-742), DIIS through oracle/pyscf_stub's restatement of
            pyscf.lib.diis, for any object with the GCC method surface.
Pinned against the unmodified reference's runs stored in tests/golden/solver_ccsd_*.npz by
tests/test_oracle_pins_solver.py.
"""
import numpy as np


class ExpMat(object):
    def __init__(self, L, rdm1_exp):
        self.exp = np.asarray(rdm1_exp, dtype=np.float64)
        self.L = float(L)
        self.Vexp = np.full((1, 1), None)

    def Vexp_update(self, rdm1, rdm1_add, index, L=None):
        if tuple(index) != (0, 0):
            raise NotImplementedError("only the ground-state 'mat' target")
        L = self.L if L is None else float(L)
        diff = np.subtract(self.exp, rdm1)
        self.Vexp[0, 0] = np.zeros_like(rdm1) + L * diff                    # exp_pot.py:165, 191-192
        return np.sum(abs(diff)) / np.sum(abs(self.exp)), np.max(abs(diff))  # exp_pot.py:193-195, 416-419


def mp2_start(fock, oovv, nocc):
    e = np.diagonal(fock)
    fia = e[:nocc, None] - e[None, nocc:]
    eijab = fia[:, None, :, None] + fia[None, :, None, :]                   # lib.direct_sum('ia,jb->ijab')
    td = oovv / eijab
    return td, td.copy()


def scf_loop(mycc, vx, L, alpha=None, conv_thres=1e-6, maxiter=40, conv='tl', diis='', maxdiis=15):
    from .pyscf_stub.pyscf.lib.diis import DIIS
    o, v = mycc.nocc, mycc.nvir
    adiis = tl_diis = None
    if 'rdm1' in diis:                                                      # Solver_GS.py:666-674
        adiis = DIIS()
        adiis.space, adiis.min_space = maxdiis, 2
    if 'tl' in diis:
        tl_diis = DIIS()
        tl_diis.space, tl_diis.min_space = maxdiis, 2
    ts, ls = np.zeros((o, v)), np.zeros((o, v))
    td, ld = mp2_start(mycc.fock, mycc.eris.oovv, o)
    cv = 0.
    Dconv, ite = 1.0, 0
    conv_ite, Delta_ite, Ep_ite = [], [], []
    while Dconv > conv_thres:
        cv_old = cv
        rdm1 = mycc.gamma(ts, td, ls, ld)
        if adiis is not None:
            rdm1 = adiis.update(np.ravel(rdm1)).reshape(rdm1.shape)
        Delta, vmax = vx.Vexp_update(rdm1, rdm1, (0, 0), L=L)
        fsp = np.subtract(mycc.fock, vx.Vexp[0, 0])
        Delta_ite.append((Delta, vmax))
        Ep_ite.append(mycc.energy(ts, td, fsp))
        ts, td = mycc.tupdate(ts, td, fsp=fsp, alpha=alpha)
        ls, ld = mycc.lupdate(ts, td, ls, ld, fsp=fsp, alpha=alpha)
        if tl_diis is not None:                                             # Solver_GS.py:709-718
            vec = tl_diis.update(np.concatenate((np.ravel(ls), np.ravel(ts), np.ravel(ld), np.ravel(td))))
            ls, ts = vec[:o * v].reshape(o, v), vec[o * v:2 * o * v].reshape(o, v)
            ld, td = (x.reshape(o, o, v, v) for x in np.split(vec[2 * o * v:], 2))
        if conv == 'tl':
            cv = np.concatenate((abs(ls.flatten()) + abs(ts.flatten()), abs(ld.flatten()) + abs(td.flatten())))
        elif conv == 'l':
            cv = np.concatenate((ls.flatten(), ld.flatten()))
        else:
            cv = mycc.energy(ts, td, fsp)
        if ite > 0:
            Dconv = np.linalg.norm(cv - cv_old)
        conv_ite.append(Dconv)
        if ite >= maxiter:
            text = 'Max iteration reached'
            break
        if Dconv > 1.0:
            text = 'Diverges for lambda = {} after {} iterations'.format(L, ite)
            break
        ite += 1
    else:
        text = 'Convergence reached for lambda= {} and alpha={}, after {} iteration'.format(L, alpha, ite)
    return text, np.asarray(Ep_ite), np.asarray(Delta_ite), np.asarray(conv_ite), rdm1, [ts, ls, td, ld]
