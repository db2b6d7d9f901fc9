"""TEST INFRASTRUCTURE — CPU oracle of the discrete auxiliary mode (cpdp_aux mode 2).  Not part of the product path.

Extends ``oracle.cpdp_oracle.Oracle`` (unchanged) with
  * ``interval_theta_derivs``: E_k = dF_k/dtheta and Hth_k = d(grad_z (q_k + lam_{k+1}'F_k))/dtheta of one RK4 interval,
    analytically through the same stage recursion as ``Oracle.interval_derivs`` (forward theta-sensitivities of the stages,
    stage adjoints of the discrete adjoint sweep, mixed second derivatives of the stage Hamiltonians);
  * ``aux_discrete``: dX/dtheta and dU/dtheta of the converged NLP by implicit differentiation of its KKT system, assembled
    densely; d(KKT residual)/dtheta is taken by finite differences of ``interval_derivs`` / ``term`` so that it does not share
    the kernels' analytic mixed-Hessian formula.
"""
import numpy as np
import sympy as sp

from oracle.cpdp_oracle import Oracle


def _fd(fun, th, i, rel=1e-3):
    """d fun / d theta_i by the fourth-order central stencil (truncation O(h^4))."""
    h = rel * max(1.0, abs(th[i]))
    def at(s):
        t = np.array(th, dtype=float)
        t[i] += s * h
        return fun(t)
    return (8.0 * (at(1) - at(-1)) - (at(2) - at(-2))) / (12.0 * h)


class DiscreteOracle(Oracle):
    def __init__(self, model, n_grid=10, steps_per_grid=4):
        super().__init__(model, n_grid, steps_per_grid)
        n, m = self.n, self.m
        x, u, th = model.x, model.u, model.theta
        pd = list(getattr(model, 'pdata', [])) + ([model.time] if getattr(model, 'time', None) is not None else [])
        z = x + u
        mu = [sp.Symbol('mu%d' % i, real=True) for i in range(n)]
        wc = sp.Symbol('wc', real=True)
        f, c = model.dyn, model.path
        ham = wc * c + (sp.Matrix(mu).T * f)[0, 0]
        hz = sp.Matrix([ham]).jacobian(z).T
        fth, hzz, hzth = f.jacobian(th), hz.jacobian(z), hz.jacobian(th)
        shapes = [fth.shape, hzz.shape, hzth.shape]
        fn = sp.lambdify([x, u, th, pd, mu, wc], list(fth) + list(hzz) + list(hzth), modules='math', cse=True)

        def mixed(*a):
            v = np.array(fn(*a), dtype=float)
            out, k = [], 0
            for s in shapes:
                out.append(v[k:k + s[0] * s[1]].reshape(s))
                k += s[0] * s[1]
            return out
        self._mixed = mixed
        self._nz = n + m

    def interval_theta_derivs(self, x, u, th, lam_next, DT, tk=0.0):
        """(E [n, r], Hth [n+m, r]) of one interval: Sth_s propagated with zero start, and
        Hth = sum_s Sz_s' (Hess_zz(Ham_s) [Sth_s; 0] + Hess_ztheta(Ham_s)), Ham_s = w_s c + mu_s'f."""
        n, m, r = self.n, self.m, self.r
        nz = n + m
        pd = self._pd(tk)
        Eu = np.zeros((m, nz)); Eu[:, n:] = np.eye(m)
        X = np.array(x, dtype=float)
        Sx = np.zeros((n, nz)); Sx[:, :n] = np.eye(n)
        St = np.zeros((n, r))
        bco = [1.0 / 6, 2.0 / 6, 2.0 / 6, 1.0 / 6]
        aco = [0.0, 0.5, 0.5, 1.0]
        rec = []
        for _ in range(self.S):
            stages = []
            Xn, Sn, Stn = X.copy(), Sx.copy(), St.copy()
            kp = dkp = dtp = None
            for s in range(4):
                xs = X if s == 0 else X + aco[s] * DT * kp
                Ss = Sx if s == 0 else Sx + aco[s] * DT * dkp
                Sts = St if s == 0 else St + aco[s] * DT * dtp
                f, c, fz, cz = self.fn.stage1(xs, u, th, pd)
                fth = self._mixed(xs, u, th, pd, np.zeros(n), 0.0)[0]
                Sz = np.vstack([Ss, Eu])
                dk = fz @ Sz
                dt = fz[:, :n] @ Sts + fth
                stages.append((xs, fz, cz.ravel(), Sz, Sts))
                Xn = Xn + bco[s] * DT * f
                Sn = Sn + bco[s] * DT * dk
                Stn = Stn + bco[s] * DT * dt
                kp, dkp, dtp = f, dk, dt
            rec.append(stages)
            X, Sx, St = Xn, Sn, Stn
        Ht = np.zeros((nz, r))
        a = np.array(lam_next, dtype=float)
        for stages in reversed(rec):
            ax = np.zeros(n)
            xi_next = None
            for s in (3, 2, 1, 0):
                kap = bco[s] * DT * a
                if s < 3:
                    kap = kap + aco[s + 1] * DT * xi_next
                w = bco[s] * DT
                xs, fz, cz, Sz, Sts = stages[s]
                _, hzz, hzth = self._mixed(xs, u, th, pd, kap, w)
                Ht += Sz.T @ (hzz[:, :n] @ Sts + hzth)
                xi = fz[:, :n].T @ kap + w * cz[:n]
                ax += xi
                xi_next = xi
            a = a + ax
        return St, Ht

    def aux_discrete(self, time_grid, X, U, Lam, theta):
        """(Xa [N+1, n*r], Ua [N+1, m*r]) = d(X, U)/dtheta of the NLP at the converged point (X, U, Lam), rows n x r / m x r
        row-major, Ua[N] = Ua[N-1] (CPDP.py:191).  Dense solve of  [W Ag'; Ag 0] d(w, lam)/dtheta = -d(KKT residual)/dtheta."""
        n, m, r, N = self.n, self.m, self.r, self.N
        nz = n + m
        th = np.asarray(theta, dtype=float)
        tg = np.asarray(time_grid, dtype=float)
        DT = tg[-1] / N / self.S
        nw, ng = (N + 1) * n + N * m, (N + 1) * n
        Wm = np.zeros((nw, nw))
        Ag = np.zeros((ng, nw))
        Ag[:n, :n] = -np.eye(n)
        for k in range(N):
            _, _, A, B, _, _, H = self.interval_derivs(X[k], U[k], th, Lam[k + 1], DT, tg[k])
            Wm[k * nz:(k + 1) * nz, k * nz:(k + 1) * nz] += H
            Ag[(k + 1) * n:(k + 2) * n, k * nz:k * nz + n] = A
            Ag[(k + 1) * n:(k + 2) * n, k * nz + n:(k + 1) * nz] = B
            Ag[(k + 1) * n:(k + 2) * n, (k + 1) * nz:(k + 1) * nz + n] = -np.eye(n)
        Wm[N * nz:, N * nz:] += self.fn.term(X[N], th, self._pd(tg[-1]))[2]

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

        dR = np.stack([_fd(resid, th, i) for i in range(r)], axis=1)
        K = np.zeros((nw + ng, nw + ng))
        K[:nw, :nw] = Wm
        K[:nw, nw:] = Ag.T
        K[nw:, :nw] = Ag
        dw = np.linalg.solve(K, -dR)[:nw]
        Xa = np.zeros((N + 1, n * r))
        Ua = np.zeros((N + 1, m * r))
        for k in range(N + 1):
            Xa[k] = dw[k * nz:k * nz + n].ravel()
            if k < N:
                Ua[k] = dw[k * nz + n:(k + 1) * nz].ravel()
        Ua[N] = Ua[N - 1]
        return Xa, Ua
