#!/usr/bin/env python3
"""Developer tool (CPU, numpy; not part of the product path): how far the eigenbasis of L = A' - P R drifts from one
interval-start Jacobian of the backward BDF sweep to the next, and whether Newton refinement of the previous basis recovers
the new one -- the experiment behind bdf_eig_refine (csrc/cpdp_bdf.cuh, DESIGN.md section 3.2).

On the six cases of tests/golden/oracle_quad50.npz (quadrotor, N = 50) the oracle's backward BDF sweep gives P at every
node.  Going backwards, each node starts from the exact eigenbasis of the previous node's L (when that basis passes the
kernel's conditioning test) and iterates  M = H L G,  F_ij = M_ij / (d_j - d_i),  G <- G (I + F),  H = G^{-1}, abandoning
as soon as max |F| > 0.5.  Output: one line per case (per node: steps to convergence, F = rejected, - = no warm basis) and
a summary line, also written to profiles/r08_eig_refine_drift.txt.

  python tools/eig_refine_drift.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import models  # noqa: E402
from oracle.cpdp_oracle import Oracle  # noqa: E402

KAPPA = 1e4            # CPDP_BDF_EIG_KAPPA
FMAX = 0.5             # BDF_REFINE_FMAX
TOL = 1e-11            # converged: ||offdiag M||_F <= TOL ||L||_F (complex arithmetic here; the kernel works in the real basis)
MAXIT = 8


def main():
    z = np.load(os.path.join(ROOT, "tests", "golden", "oracle_quad50.npz"))
    N, T = int(z["n_grid"]), float(z["T"])
    orc = Oracle(models.quadrotor(), n_grid=N)
    lines, nodes, ok_n, its = [], 0, 0, []
    for case in range(z["X"].shape[0]):
        orc.pd = z["pdata"][case]
        X, U, Lam, th = z["X"][case], z["U"][case], z["Lam"][case], z["theta"][case]
        tg = np.linspace(0, T, N + 1)
        _, _, PW = orc.aux(tg, X, U, Lam, th, back={"method": "BDF"}, fwd={})
        n = X.shape[1]
        Ls = []
        for k in range(N + 1):
            fx, fu, fe, Hxx, Hxu, Hxe, Huu, Hue, iH = orc._coeffs(X[k], U[k], Lam[k], th, tg[k])
            G = fu @ iH
            Ls.append((fx - G @ Hxu.T).T - PW[k, :n * n].reshape(n, n) @ (G @ fu.T))
        row = []
        for k in range(N - 1, -1, -1):
            _, Vp = np.linalg.eig(Ls[k + 1])
            if np.linalg.norm(Vp) * np.linalg.norm(np.linalg.inv(Vp)) > KAPPA:
                row.append("-")
                continue
            Gm, Hm = Vp, np.linalg.inv(Vp)
            ok, it = False, 0
            for it in range(MAXIT + 1):
                M = Hm @ Ls[k] @ Gm
                d = np.diag(M).copy()
                if np.linalg.norm(M - np.diag(d)) <= TOL * np.linalg.norm(Ls[k]):
                    ok = True
                    break
                gap = d[None, :] - d[:, None]
                np.fill_diagonal(gap, 1.0)
                F = (M - np.diag(d)) / gap
                if not np.all(np.isfinite(F)) or np.abs(F).max() > FMAX:
                    break
                Gm = Gm @ (np.eye(n) + F)
                Hm = np.linalg.inv(Gm)
            ok = ok and np.linalg.norm(Gm) * np.linalg.norm(Hm) <= KAPPA
            nodes += 1
            ok_n += ok
            if ok:
                its.append(it)
            row.append(str(it) if ok else "F")
        lines.append("case %d  %s" % (case, "".join(row)))
    hist = np.bincount(np.array(its, dtype=int)) if its else []
    lines.append("refinement accepted at %d of %d interval-start Jacobians with a warm basis (%.0f %%); steps to convergence "
                 "0, 1, 2, ...: %s" % (ok_n, nodes, 100.0 * ok_n / max(nodes, 1), list(map(int, hist))))
    text = "\n".join(lines) + "\n"
    print(text, end="")
    with open(os.path.join(ROOT, "profiles", "r08_eig_refine_drift.txt"), "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
