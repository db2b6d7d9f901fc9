"""TEST INFRASTRUCTURE — CPU oracle of the adjoint of mode 2 with respect to the per-problem constants pdata (cpdp_aux_adjoint_pd's
pdata_bar).  Not part of the product path.

Extends ``tests.discrete_oracle.DiscreteOracle`` and ``tests.bounded_oracle.BoundedOracle`` (both unchanged) with d(X, U)/dpdata by
dense implicit differentiation of the same KKT matrices their ``aux_discrete`` / ``aux_discrete_bounded`` assemble.  The right-hand
side, d(KKT residual)/dpdata at fixed (w, lam), is taken by the fourth-order central stencil of ``discrete_oracle._fd`` over
``interval_derivs`` / ``term`` with ``self.pd`` perturbed, as those oracles do for theta; it does not share the kernels' analytic
mixed Hessians (ModelPd::dir_pd, term2_pd).  Only the q user constants are differentiated: the time of a time-varying model,
which ``_pd`` appends, is not a column."""
import numpy as np

from tests.adjoint_oracle import _split
from tests.bounded_oracle import BoundedOracle
from tests.discrete_oracle import DiscreteOracle, _fd


def _resid_pd(orc, X, U, Lam, th, tg, DT, nw, ng):
    """pd -> pdata-dependent part of [grad_w L; g] at fixed (w, lam) (the rows of ``aux_discrete``'s resid)."""
    n, m, N = orc.n, orc.m, orc.N
    nz = n + m

    def resid(pd):
        keep = orc.pd
        orc.pd = np.asarray(pd, dtype=float)
        try:
            gl = np.zeros(nw)
            g = np.zeros(ng)
            for k in range(N):
                xe, _, _, _, _, gL, _ = orc.interval_derivs(X[k], U[k], th, Lam[k + 1], DT, tg[k])
                gl[k * nz:(k + 1) * nz] += gL
                g[(k + 1) * n:(k + 2) * n] = xe
            gl[N * nz:N * nz + n] += np.ravel(orc.fn.term(X[N], th, orc._pd(tg[-1]))[1])
        finally:
            orc.pd = keep
        return np.concatenate([gl, g])
    return resid


class PdataOracle(DiscreteOracle):
    def dpd_discrete(self, time_grid, X, U, Lam, theta):
        """(DX [N+1, n, q], DU [N+1, m, q]) = d(X, U)/dpdata of the unbounded NLP at the converged point, DU[N] = DU[N-1]."""
        n, m, N = self.n, self.m, self.N
        nz = n + m
        th = np.asarray(theta, dtype=float)
        tg = np.asarray(time_grid, dtype=float)
        DT = tg[-1] / N / self.S
        nw, ng = (N + 1) * n + N * m, (N + 1) * n
        K = np.zeros((nw + ng, nw + ng))
        Ag = np.zeros((ng, nw))
        Ag[:n, :n] = -np.eye(n)
        for k in range(N):
            _, _, A, B, _, _, H = self.interval_derivs(X[k], U[k], th, Lam[k + 1], DT, tg[k])
            K[k * nz:(k + 1) * nz, k * nz:(k + 1) * nz] += H
            Ag[(k + 1) * n:(k + 2) * n, k * nz:k * nz + n] = A
            Ag[(k + 1) * n:(k + 2) * n, k * nz + n:(k + 1) * nz] = B
            Ag[(k + 1) * n:(k + 2) * n, (k + 1) * nz:(k + 1) * nz + n] = -np.eye(n)
        K[N * nz:nw, N * nz:nw] += self.fn.term(X[N], th, self._pd(tg[-1]))[2]
        K[:nw, nw:] = Ag.T
        K[nw:, :nw] = Ag
        resid = _resid_pd(self, X, U, Lam, th, tg, DT, nw, ng)
        dR = np.stack([_fd(resid, self.pd, i) for i in range(len(self.pd))], axis=1)
        return _split(np.linalg.solve(K, -dR)[:nw], n, m, N)


class BoundedPdataOracle(BoundedOracle):
    def dpd_discrete_bounded(self, time_grid, X, U, Lam, Zl, Zu, theta):
        """(DX, DU) = d(X, U)/dpdata of the barrier-perturbed KKT system with the bound multipliers as unknowns (the matrix of
        ``aux_discrete_bounded``; the bounds do not depend on pdata)."""
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
        resid = _resid_pd(self, X, U, Lam, th, tg, DT, nw, ng)
        dR = np.zeros((tot, len(self.pd)))
        dR[:nw + ng] = np.stack([_fd(resid, self.pd, i) for i in range(len(self.pd))], axis=1)
        return _split(np.linalg.solve(K, -dR)[:nw], n, m, N)
