"""TEST INFRASTRUCTURE — CPU oracle of the adjoint of mode 2 with respect to x0 (cpdp_aux_adjoint's x0_bar).  Not part of the
product path.

Extends ``tests.discrete_oracle.DiscreteOracle`` and ``tests.bounded_oracle.BoundedOracle`` (both unchanged) with dX/dx0 and dU/dx0
by dense implicit differentiation of the same KKT matrices their ``aux_discrete`` / ``aux_discrete_bounded`` assemble: x0 enters
the KKT residual only through the initial-value rows g_0 = x0 - X_0, so the right-hand side is minus the identity in those rows.
The kernels instead transpose the Riccati rollout; the two share nothing but the stage derivatives."""
import numpy as np

from tests.bounded_oracle import BoundedOracle
from tests.discrete_oracle import DiscreteOracle


def _split(dw, n, m, N):
    """d(w)/dx0 [nw, n] -> (DX [N+1, n, n], DU [N+1, m, n]) with DU[N] = DU[N-1] (CPDP.py:191)."""
    nz = n + m
    DX = np.stack([dw[k * nz:k * nz + n] for k in range(N + 1)])
    DU = np.stack([dw[k * nz + n:(k + 1) * nz] for k in range(N)] + [dw[(N - 1) * nz + n:N * nz]])
    return DX, DU


def _solve_g0(K, nw, n):
    rhs = np.zeros((K.shape[0], n))
    rhs[nw:nw + n] = -np.eye(n)                    # d(g_0)/dx0 = I
    return np.linalg.solve(K, rhs)[:nw]


def contract(DX, DU, Xbar, Ubar):
    """sum_k DX_k' Xbar_k + DU_k' Ubar_k (the adjoint a kernel returns for cotangents Xbar [N+1, n], Ubar [N+1, m])."""
    return np.einsum("kin,ki->n", DX, Xbar) + np.einsum("kjn,kj->n", DU, Ubar)


class AdjointOracle(DiscreteOracle):
    def dx0_discrete(self, time_grid, X, U, Lam, theta):
        """(DX [N+1, n, n], DU [N+1, m, n]) = d(X, U)/dx0 of the unbounded NLP at the converged point (X, U, Lam)."""
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
        return _split(_solve_g0(K, nw, n), n, m, N)


class BoundedAdjointOracle(BoundedOracle):
    def dx0_discrete_bounded(self, time_grid, X, U, Lam, Zl, Zu, theta):
        """(DX, DU) = d(X, U)/dx0 of the barrier-perturbed KKT system with the bound multipliers as unknowns (the matrix of
        ``aux_discrete_bounded``)."""
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
        return _split(_solve_g0(K, nw, n), n, m, N)
