"""TEST INFRASTRUCTURE — CPU oracle of the adjoint of mode 2 with respect to per-problem constants when the box bounds are functions
of them (cpdp_aux_adjoint_pd's pdata_bar, DESIGN.md §3.12).  Not part of the product path.

Extends ``tests.bounded_oracle.BoundedOracle`` (unchanged) with bounds bnd(pd) -> (xlb, xub, ulb, uub) and d(X, U)/dpdata by dense
implicit differentiation of the barrier-perturbed KKT system with the bound multipliers as unknowns -- the matrix of
``aux_discrete_bounded``.  Its right-hand side, d(residual)/dpdata at fixed (w, lam, z_L, z_U), is the fourth-order central stencil of
``discrete_oracle._fd`` over the FULL residual: the rows of ``pdata_oracle._resid_pd`` and the complementarity rows
(w - lb(pd)) z_L - mu and (ub(pd) - w) z_U - mu with the bounds re-evaluated at the perturbed pd.  It does not share the kernels'
elimination of z into Sigma, nor their Sigma dbound/dpd term."""
import numpy as np

from tests.adjoint_oracle import _split
from tests.bounded_oracle import BoundedOracle
from tests.discrete_oracle import _fd
from tests.pdata_oracle import _resid_pd


class PdBoundedOracle(BoundedOracle):
    def __init__(self, model, bnd, pd, n_grid=10, steps_per_grid=4):
        """bnd(pd) -> (xlb, xub, ulb, uub) numeric arrays; the oracle solves at the bounds of `pd` (self.pd = pd)."""
        super().__init__(model, *bnd(pd), n_grid=n_grid, steps_per_grid=steps_per_grid)
        self.bnd = bnd
        self.pd = np.asarray(pd, dtype=float)

    def _tiled(self, pd):
        xlb, xub, ulb, uub = (np.asarray(v, dtype=float) for v in self.bnd(pd))
        lb = np.tile(np.concatenate([xlb, ulb]), self.N + 1)[:self.nw]
        ub = np.tile(np.concatenate([xub, uub]), self.N + 1)[:self.nw]
        return lb, ub

    def dpd_discrete_pdbounded(self, time_grid, X, U, Lam, Zl, Zu, theta):
        """(DX [N+1, n, q], DU [N+1, m, q]) = d(X, U)/dpdata of the barrier-perturbed KKT system, bounds depending on pdata."""
        n, m, N = self.n, self.m, self.N
        nz, nw, ng = n + m, self.nw, (N + 1) * n
        th = np.asarray(theta, dtype=float)
        tg = np.asarray(time_grid, dtype=float)
        DT = tg[-1] / N / self.S
        w = np.concatenate([np.hstack([X[:N], U[:N]]).ravel(), X[N]])
        zl = np.asarray(Zl, dtype=float).ravel()[:nw]
        zu = np.asarray(Zu, dtype=float).ravel()[:nw]
        _, _, _, W, Ag = self._assemble(w, np.asarray(Lam, dtype=float).ravel(), th, np.zeros(n), tg, DT)
        sl, su = self._slacks(w)
        il, iu = np.flatnonzero(self.fl), np.flatnonzero(self.fu)
        tot = nw + ng + len(il) + len(iu)
        K = np.zeros((tot, tot))
        K[:nw, :nw] = W
        K[:nw, nw:nw + ng] = Ag.T
        K[nw:nw + ng, :nw] = Ag
        o = nw + ng
        for a, i in enumerate(il):
            K[i, o + a], K[o + a, i], K[o + a, o + a] = -1.0, zl[i], sl[i]
        o += len(il)
        for a, i in enumerate(iu):
            K[i, o + a], K[o + a, i], K[o + a, o + a] = 1.0, -zu[i], su[i]
        kkt = _resid_pd(self, X, U, Lam, th, tg, DT, nw, ng)

        def resid(pd):
            lb, ub = self._tiled(pd)
            return np.concatenate([kkt(pd), (w[il] - lb[il]) * zl[il], (ub[iu] - w[iu]) * zu[iu]])
        dR = np.stack([_fd(resid, self.pd, i) for i in range(len(self.pd))], axis=1)
        return _split(np.linalg.solve(K, -dR)[:nw], n, m, N)
