"""TEST INFRASTRUCTURE — CPU oracle of the warm-started solve (cpdp_solve_warm).  Not part of the product path.

  * ``warm_point``: the starting point the kernels build from a guess (X, U, Lam), with or without the one-interval shift, as
    the flat w = (X_0, U_0, ..., X_N) and lam;
  * ``WarmOracle``: the Newton-KKT iteration of ``oracle.cpdp_oracle.Oracle.solve`` (dense linear solver: inertia-corrected
    Newton step on the assembled KKT matrix, IPOPT's filter line search on phi = J, theta = |g|_1) started from (w0, lam0)
    instead of the zero seed.  ``Oracle.solve`` fixes its seed, so ``solve_warm`` restates that iteration, statement for
    statement, on the assembled NLP pieces of ``tests.bounded_oracle.BoundedOracle`` (with no finite bound);
  * ``WarmBoundedOracle``: ``tests.bounded_oracle.BoundedOracle`` started as IPOPT's ``warm_start_init_point`` does: the guess
    pushed into the interior by warm_start_bound_push = warm_start_bound_frac = 1e-3 (``start``), z = max(z guess, 1e-3) or
    mu_init / slack, mu = mu_init.  ``BoundedOracle.solve_bounded`` fixes its z and mu start, so ``solve_warm`` restates its
    iteration with the start as an argument; the iteration is the same, statement for statement.
"""
import numpy as np

from oracle.cpdp_oracle import _inertia_ok
from tests.bounded_oracle import BoundedOracle, BIG

WARM_PUSH = 1e-3
WARM_MULT_PUSH = 1e-3


def shifted(A, shift, last):
    """Rows min(k + shift, last) of A for k = 0 .. len(A) - 1."""
    return A[np.minimum(np.arange(len(A)) + shift, last)]


def warm_point(x0, X, U, Lam, shift=0):
    """(w0, lam0) of the kernels' warm start from the guess (X [N+1,n], U [N+1,m], Lam [N+1,n]): X_0 = x0, U_N unused."""
    N = X.shape[0] - 1
    Xs, Us, Ls = shifted(X, shift, N), shifted(U, shift, N - 1), shifted(Lam, shift, N)
    Xs[0] = x0
    w = np.concatenate([np.hstack([Xs[:N], Us[:N]]).ravel(), Xs[N]])
    return w, Ls.ravel()


class WarmOracle(BoundedOracle):
    def __init__(self, model, n_grid=10, steps_per_grid=4):
        n, m = model.n, model.m
        super().__init__(model, [-1e20] * n, [1e20] * n, [-1e20] * m, [1e20] * m, n_grid, steps_per_grid)

    def solve_warm(self, x0, horizon, theta, w0, lam0, tol=1e-10, max_iter=200):
        """Oracle.solve(linear_solver='dense') from (w0, lam0).  Returns (time_grid, X, U, Lam, info) as Oracle.solve does."""
        n, m, N = self.n, self.m, self.N
        nz, nw, ng = n + m, self.nw, (N + 1) * n
        th = np.asarray(theta, dtype=float)
        x0 = np.asarray(x0, dtype=float).ravel()
        DT = horizon / N / self.S
        tg = np.linspace(0, horizon, N + 1) if self.tv else np.array([horizon / N * k for k in range(N + 1)])
        w = np.array(w0, dtype=float)
        lam = np.array(lam0, dtype=float)
        filt = []
        theta_min = theta_max = None
        delta_last = 0.0
        info = dict(iters=0, status='max_iter', reg=[], alphas=[])
        for it in range(max_iter + 1):
            J, g, gradJ, W, Ag = self._assemble(w, lam, th, x0, tg, DT)
            kkt_err = max(np.abs(gradJ + Ag.T @ lam).max(), np.abs(g).max())
            if kkt_err < tol:
                info['status'] = 'converged'
                break
            if it == max_iter:
                break
            delta, first = 0.0, True
            while True:
                K = np.zeros((nw + ng, nw + ng))
                K[:nw, :nw] = W + delta * np.eye(nw)
                K[:nw, nw:] = Ag.T
                K[nw:, :nw] = Ag
                if _inertia_ok(K, nw, ng):
                    break
                if first:
                    delta = 1e-4 if delta_last == 0.0 else max(1e-20, delta_last / 3.0)
                    first = False
                else:
                    delta = delta * (100.0 if delta_last == 0.0 else 8.0)
                if delta > 1e40:
                    raise FloatingPointError('inertia correction failed')
            if delta > 0:
                delta_last = delta
            info['reg'].append(delta)
            sol = np.linalg.solve(K, -np.concatenate([gradJ, g]))
            d, lam_new = sol[:nw], sol[nw:]
            th0 = np.abs(g).sum()
            if theta_min is None:
                theta_min, theta_max = 1e-4 * max(1.0, th0), 1e4 * max(1.0, th0)
            gd = gradJ @ d
            alpha = 1.0
            accepted = ftype = False
            for _ls in range(31):
                try:
                    with np.errstate(all='ignore'):
                        Jt, gt = self._evaluate(w + alpha * d, th, x0, tg, DT)
                    tht = np.abs(gt).sum()
                except (ValueError, OverflowError, FloatingPointError):
                    Jt = tht = np.inf
                ok = np.isfinite(Jt) and np.isfinite(tht) and tht <= theta_max
                if ok and any(tht >= tf and Jt >= pf for tf, pf in filt):
                    ok = False
                if ok:
                    switching = gd < 0 and alpha * (-gd) ** 2.3 > th0 ** 1.1
                    if switching and th0 <= theta_min:
                        accepted = ftype = Jt <= J + 1e-8 * alpha * gd
                    else:
                        accepted = tht <= (1 - 1e-5) * th0 or Jt <= J - 1e-8 * th0
                if accepted:
                    break
                alpha *= 0.5
            if not accepted:
                info['status'] = 'linesearch_fail'
                break
            if not ftype:
                filt.append(((1 - 1e-5) * th0, J - 1e-8 * th0))
            info['alphas'].append(alpha)
            w = w + alpha * d
            lam = lam + alpha * (lam_new - lam)
            info['iters'] = it + 1
        info['J'] = J
        info['kkt'] = kkt_err
        sc = np.concatenate([w, np.zeros(m)]).reshape(-1, nz)
        X = sc[:, :n].copy()
        U = sc[:, n:].copy()
        U[-1, :] = U[-2, :]
        return tg, X, U, lam.reshape(-1, n).copy(), info


class WarmBoundedOracle(BoundedOracle):
    def start(self, w=None):
        """IPOPT's warm-start push of w (the cold start's zero seed with bound_push 1e-2 when w is None)."""
        if w is None:
            return super().start()
        lb, ub, fl, fu = self.lb, self.ub, self.fl, self.fu
        k = WARM_PUSH
        pl = np.where(fu, np.minimum(k * np.maximum(1.0, np.abs(lb)), k * (ub - lb)), k * np.maximum(1.0, np.abs(lb)))
        pu = np.where(fl, np.minimum(k * np.maximum(1.0, np.abs(ub)), k * (ub - lb)), k * np.maximum(1.0, np.abs(ub)))
        w = np.array(w, dtype=float)
        lo = fl & (w < lb + pl)
        w[lo] = (lb + pl)[lo]
        hi = ~lo & fu & (w > ub - pu)
        w[hi] = (ub - pu)[hi]
        return w

    def warm_z(self, w, Zl, Zu, mu_init):
        """Starting z_L, z_U [nw]: max(guess, 1e-3) where a bound is finite, or mu_init / slack without a guess."""
        sl, su = self._slacks(w)
        if Zl is None:
            return np.where(self.fl, mu_init / sl, 0.0), np.where(self.fu, mu_init / su, 0.0)
        zl = np.asarray(Zl, dtype=float).ravel()[:self.nw]
        zu = np.asarray(Zu, dtype=float).ravel()[:self.nw]
        return np.where(self.fl, np.maximum(zl, WARM_MULT_PUSH), 0.0), np.where(self.fu, np.maximum(zu, WARM_MULT_PUSH), 0.0)

    def solve_warm(self, x0, horizon, theta, X, U, Lam, Zl=None, Zu=None, mu_init=1e-8, tol=1e-10, max_iter=200):
        """solve_bounded started from the guess (X, U, Lam, Zl, Zu [N+1, n+m]) at mu = mu_init.  Returns solve_bounded's dict."""
        n, m, N = self.n, self.m, self.N
        nz, nw, ng = n + m, self.nw, (N + 1) * n
        th = np.asarray(theta, dtype=float)
        x0 = np.asarray(x0, dtype=float).ravel()
        DT = horizon / N / self.S
        tg = np.array([horizon / N * k for k in range(N + 1)])
        fl, fu = self.fl, self.fu
        xl, xu = self.lb[:n], self.ub[:n]
        if np.any((np.abs(xl) < BIG) & ~(x0 > xl)) or np.any((np.abs(xu) < BIG) & ~(x0 < xu)):
            return dict(status='infeasible', iters=0)
        w0, lam = warm_point(x0, np.asarray(X, dtype=float), np.asarray(U, dtype=float), np.asarray(Lam, dtype=float))
        w = self.start(w0)
        zl, zu = self.warm_z(w, Zl, Zu, mu_init)
        mu = mu_init
        filt = []
        theta_min = theta_max = None
        delta_last = 0.0
        info = dict(status='max_iter', iters=0, alphas=[], mus=[], iterates=[w.copy()])
        for it in range(max_iter + 1):
            J, g, gradJ, W, Ag = self._assemble(w, lam, th, x0, tg, DT)
            sl, su = self._slacks(w)
            e = max(np.abs(gradJ + Ag.T @ lam - zl + zu).max(), np.abs(g).max())
            sz = np.concatenate([(sl * zl)[fl], (su * zu)[fu]])
            kkt = max(e, sz.max())
            if kkt >= tol:
                while max(e, np.abs(sz - mu).max()) <= 10.0 * mu:
                    mn = max(tol / 10.0, min(0.2 * mu, mu ** 1.5))
                    if not mn < mu:
                        break
                    mu = mn
                    filt = []
            info['mus'].append(mu)
            if kkt < tol:
                info['status'] = 'converged'
                break
            if it == max_iter:
                break
            phi0 = J - mu * self._logsum(w)
            sig = np.where(fl, zl / sl, 0.0) + np.where(fu, zu / su, 0.0)
            bg = np.where(fl, -mu / sl, 0.0) + np.where(fu, mu / su, 0.0)
            delta, first = 0.0, True
            while True:
                K = np.zeros((nw + ng, nw + ng))
                K[:nw, :nw] = W + np.diag(sig) + delta * np.eye(nw)
                K[:nw, nw:] = Ag.T
                K[nw:, :nw] = Ag
                if _inertia_ok(K, nw, ng):
                    break
                if first:
                    delta = 1e-4 if delta_last == 0.0 else max(1e-20, delta_last / 3.0)
                    first = False
                else:
                    delta = delta * (100.0 if delta_last == 0.0 else 8.0)
                if delta > 1e40:
                    raise FloatingPointError('inertia correction failed')
            if delta > 0:
                delta_last = delta
            sol = np.linalg.solve(K, -np.concatenate([gradJ + bg, g]))
            d, lam_new = sol[:nw], sol[nw:]
            gd = (gradJ + bg) @ d
            tau = max(0.99, 1.0 - mu)
            dzl = np.where(fl, mu / sl - zl - (zl / sl) * d, 0.0)
            dzu = np.where(fu, mu / su - zu - (zu / su) * (-d), 0.0)
            with np.errstate(divide='ignore', invalid='ignore'):
                amax = min([1.0] + list((-tau * sl / d)[fl & (d < 0)]) + list((tau * su / d)[fu & (d > 0)]))
                az = min([1.0] + list((-tau * zl / dzl)[fl & (dzl < 0)]) + list((-tau * zu / dzu)[fu & (dzu < 0)]))
            th0 = np.abs(g).sum()
            if theta_min is None:
                theta_min, theta_max = 1e-4 * max(1.0, th0), 1e4 * max(1.0, th0)
            alpha = amax
            accepted = ftype = False
            for _ls in range(31):
                wt = w + alpha * d
                try:
                    with np.errstate(all='ignore'):
                        Jt, gt = self._evaluate(wt, th, x0, tg, DT)
                        Pt = Jt - mu * self._logsum(wt)
                    tht = np.abs(gt).sum()
                except (ValueError, OverflowError, FloatingPointError):
                    Pt = tht = np.inf
                ok = np.isfinite(Pt) and np.isfinite(tht) and tht <= theta_max
                if ok and any(tht >= tf and Pt >= pf for tf, pf in filt):
                    ok = False
                if ok:
                    switching = gd < 0 and alpha * (-gd) ** 2.3 > th0 ** 1.1
                    if switching and th0 <= theta_min:
                        accepted = ftype = Pt <= phi0 + 1e-8 * alpha * gd
                    else:
                        accepted = tht <= (1 - 1e-5) * th0 or Pt <= phi0 - 1e-8 * th0
                if accepted:
                    break
                alpha *= 0.5
            if not accepted:
                info['status'] = 'linesearch_fail'
                break
            if not ftype:
                filt.append(((1 - 1e-5) * th0, phi0 - 1e-8 * th0))
            info['alphas'].append(alpha)
            wn = w + alpha * d
            sln, sun = self._slacks(wn)
            zl = np.where(fl, np.maximum(np.minimum(zl + az * dzl, 1e10 * mu / sln), mu / (1e10 * sln)), 0.0)
            zu = np.where(fu, np.maximum(np.minimum(zu + az * dzu, 1e10 * mu / sun), mu / (1e10 * sun)), 0.0)
            w = wn
            lam = lam + alpha * (lam_new - lam)
            info['iters'] = it + 1
            info['iterates'].append(w.copy())
        pad = lambda v: np.concatenate([v, np.zeros(m)]).reshape(N + 1, nz)
        sc = pad(w)
        Uo = sc[:, n:].copy()
        Uo[N] = Uo[N - 1]
        info.update(X=sc[:, :n].copy(), U=Uo, Lam=lam.reshape(N + 1, n).copy(), Zl=pad(zl), Zu=pad(zu), mu=mu, J=J, kkt=kkt,
                    time_grid=tg)
        return info
