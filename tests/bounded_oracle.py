"""TEST INFRASTRUCTURE — CPU oracle of the box-bounded solve and of mode 2 through active bounds.  Not part of the product path.

Extends ``tests.discrete_oracle.DiscreteOracle`` (and through it the unchanged ``oracle.cpdp_oracle.Oracle``) with
  * ``solve_bounded``: IPOPT's primal-dual barrier method (Waechter & Biegler 2006, §2-3) for box bounds on
    w = (X_0, U_0, ..., X_N), restated on the assembled dense KKT matrix with the inertia test of ``_inertia_ok``:
    the zero seed pushed into the interior (bound_push = bound_frac = 1e-2), z = 1, mu = 0.1; Newton steps on
    [W + Sigma + delta I, Ag'; Ag, 0] with the barrier gradient; fraction to the boundary tau = max(0.99, 1 - mu) for the
    primal and the dual step; the filter line search on phi_mu = J - mu sum ln s; z += alpha_z dz and the kappa_Sigma = 1e10
    safeguard; mu <- max(tol/10, min(0.2 mu, mu^1.5)) while E_mu <= 10 mu (filter emptied); stop at E_0 < tol (unscaled);
  * ``aux_discrete_bounded``: d(X, U)/dtheta by dense implicit differentiation of the barrier-perturbed KKT system with the
    bound multipliers as unknowns (the rows S_L z_L = mu, S_U z_U = mu included), so that it does not share the kernels'
    elimination of z into Sigma.
"""
import numpy as np

from oracle.cpdp_oracle import _inertia_ok
from tests.discrete_oracle import DiscreteOracle, _fd

BIG = 1e19


class BoundedOracle(DiscreteOracle):
    def __init__(self, model, xlb, xub, ulb, uub, n_grid=10, steps_per_grid=4):
        super().__init__(model, n_grid, steps_per_grid)
        n, m, N = self.n, self.m, self.N
        nz = n + m
        self.nw = (N + 1) * nz - m
        self.lb = np.tile(np.concatenate([xlb, ulb]).astype(float), N + 1)[:self.nw]
        self.ub = np.tile(np.concatenate([xub, uub]).astype(float), N + 1)[:self.nw]
        self.fl = np.abs(self.lb) < BIG
        self.fu = np.abs(self.ub) < BIG

    # ------------------------------------------------------------------------------------------------ NLP pieces
    def _assemble(self, w, lam, th, x0, tg, DT):
        """J, g, gradJ, W (Hessian of the Lagrangian at lam), Ag."""
        n, m, N = self.n, self.m, self.N
        nz, nw, ng = n + m, self.nw, (N + 1) * n
        J = 0.0
        g = np.zeros(ng)
        gradJ = np.zeros(nw)
        W = np.zeros((nw, nw))
        Ag = np.zeros((ng, nw))
        g[:n] = x0 - w[:n]
        Ag[:n, :n] = -np.eye(n)
        for k in range(N):
            o = k * nz
            xe, q, A, B, dQ, _, H = self.interval_derivs(w[o:o + n], w[o + n:o + nz], th, lam[(k + 1) * n:(k + 2) * n], DT, tg[k])
            J += q
            g[(k + 1) * n:(k + 2) * n] = xe - w[o + nz:o + nz + n]
            gradJ[o:o + nz] += dQ
            W[o:o + nz, o:o + nz] += H
            Ag[(k + 1) * n:(k + 2) * n, o:o + n] = A
            Ag[(k + 1) * n:(k + 2) * n, o + n:o + nz] = B
            Ag[(k + 1) * n:(k + 2) * n, o + nz:o + nz + n] = -np.eye(n)
        hv, hx, hxx, _ = self.fn.term(w[N * nz:], th, self._pd(tg[-1]))
        J += hv
        gradJ[N * nz:] += np.ravel(hx)
        W[N * nz:, N * nz:] += hxx
        return J, g, gradJ, W, Ag

    def _evaluate(self, w, th, x0, tg, DT):
        n, N, nz = self.n, self.N, self.n + self.m
        J = 0.0
        g = np.zeros((N + 1) * n)
        g[:n] = x0 - w[:n]
        for k in range(N):
            o = k * nz
            xe, q = self.interval(w[o:o + n], w[o + n:o + nz], th, DT, tg[k])
            J += q
            g[(k + 1) * n:(k + 2) * n] = xe - w[o + nz:o + nz + n]
        J += self.fn.term(w[N * nz:], th, self._pd(tg[-1]))[0]
        return J, g

    def _slacks(self, w):
        sl = np.where(self.fl, w - self.lb, 1.0)
        su = np.where(self.fu, self.ub - w, 1.0)
        return sl, su

    def _logsum(self, w):
        sl, su = self._slacks(w)
        with np.errstate(all='ignore'):
            return np.sum(np.log(sl[self.fl])) + np.sum(np.log(su[self.fu]))

    def start(self):
        """IPOPT's projection of the zero seed into the interior (bound_push = bound_frac = 1e-2)."""
        lb, ub, fl, fu = self.lb, self.ub, self.fl, self.fu
        pl = np.where(fu, np.minimum(1e-2 * np.maximum(1.0, np.abs(lb)), 1e-2 * (ub - lb)), 1e-2 * np.maximum(1.0, np.abs(lb)))
        pu = np.where(fl, np.minimum(1e-2 * np.maximum(1.0, np.abs(ub)), 1e-2 * (ub - lb)), 1e-2 * np.maximum(1.0, np.abs(ub)))
        w = np.zeros(self.nw)
        lo = fl & (w < lb + pl)
        w[lo] = (lb + pl)[lo]
        hi = ~lo & fu & (w > ub - pu)
        w[hi] = (ub - pu)[hi]
        return w

    # ------------------------------------------------------------------------------------------------ barrier solve
    def solve_bounded(self, x0, horizon, theta, tol=1e-10, max_iter=200):
        """Returns dict(X, U, Lam, Zl, Zu [N+1, n+m], mu, status, iters, J, kkt, alphas)."""
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
        w = self.start()
        lam = np.zeros(ng)
        zl = fl.astype(float)
        zu = fu.astype(float)
        mu = 0.1
        filt = []
        theta_min = theta_max = None
        delta_last = 0.0
        info = dict(status='max_iter', iters=0, alphas=[], mus=[])
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
            with np.errstate(divide='ignore', invalid='ignore'):          # (quotients are taken only where the step shrinks)
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
        pad = lambda v: np.concatenate([v, np.zeros(m)]).reshape(N + 1, nz)
        sc = pad(w)
        U = sc[:, n:].copy()
        U[N] = U[N - 1]
        info.update(X=sc[:, :n].copy(), U=U, Lam=lam.reshape(N + 1, n).copy(), Zl=pad(zl), Zu=pad(zu), mu=mu, J=J, kkt=kkt,
                    time_grid=tg)
        return info

    # ------------------------------------------------------------------------------------------------ mode 2, bounded
    def aux_discrete_bounded(self, time_grid, X, U, Lam, Zl, Zu, theta):
        """(Xa [N+1, n*r], Ua [N+1, m*r]) = d(X, U)/dtheta of the barrier-perturbed KKT system at (w, lam, z):
        [W Ag' -I_L I_U; Ag 0 0 0; Z_L 0 S_L 0; -Z_U 0 0 S_U] d(w, lam, z_L, z_U)/dtheta = -[d(grad L)/dtheta; dg/dtheta; 0; 0]."""
        n, m, r, N = self.n, self.m, self.r, self.N
        nz, nw, ng = n + m, self.nw, (N + 1) * n
        th = np.asarray(theta, dtype=float)
        tg = np.asarray(time_grid, dtype=float)
        DT = tg[-1] / N / self.S
        w = np.concatenate([np.hstack([X[:N], U[:N]]).ravel(), X[N]])
        lam = np.asarray(Lam, dtype=float).ravel()
        zl = np.asarray(Zl, dtype=float).ravel()[:nw]
        zu = np.asarray(Zu, dtype=float).ravel()[:nw]
        _, _, _, W, Ag = self._assemble(w, lam, th, np.zeros(n), tg, DT)
        sl, su = self._slacks(w)
        il, iu = np.flatnonzero(self.fl), np.flatnonzero(self.fu)
        nl, nu = len(il), len(iu)
        tot = nw + ng + nl + nu
        K = np.zeros((tot, tot))
        K[:nw, :nw] = W
        K[:nw, nw:nw + ng] = Ag.T
        K[nw:nw + ng, :nw] = Ag
        o = nw + ng
        for a, i in enumerate(il):
            K[i, o + a] = -1.0
            K[o + a, i] = zl[i]
            K[o + a, o + a] = sl[i]
        o += nl
        for a, i in enumerate(iu):
            K[i, o + a] = 1.0
            K[o + a, i] = -zu[i]
            K[o + a, o + a] = su[i]

        def resid(t):
            """theta-dependent part of [grad_w L; g] at fixed (w, lam)"""
            gl = np.zeros(nw)
            g = np.zeros(ng)
            for k in range(N):
                xe, _, _, _, _, gL, _ = self.interval_derivs(X[k], U[k], t, Lam[k + 1], DT, tg[k])
                gl[k * nz:(k + 1) * nz] += gL
                g[(k + 1) * n:(k + 2) * n] = xe
            gl[N * nz:] += np.ravel(self.fn.term(X[N], t, self._pd(tg[-1]))[1])
            return np.concatenate([gl, g])

        dR = np.zeros((tot, r))
        dR[:nw + ng] = np.stack([_fd(resid, th, i) for i in range(r)], axis=1)
        dw = np.linalg.solve(K, -dR)[:nw]
        Xa = np.zeros((N + 1, n * r))
        Ua = np.zeros((N + 1, m * r))
        for k in range(N + 1):
            Xa[k] = dw[k * nz:k * nz + n].ravel()
            if k < N:
                Ua[k] = dw[k * nz + n:(k + 1) * nz].ravel()
        Ua[N] = Ua[N - 1]
        return Xa, Ua
