"""Extended-precision references of the Newton-solve linear algebra of the backward BDF sweep (csrc/cpdp_bdf.cuh):
the Lyapunov system X + c (L X + X L') = B_P, the W block dW = (I + c L)^{-1} (B_W + c X C), the condition of the
Lyapunov operator, the eigenvalues of L and the conditioning of its real eigenvector basis, and residuals of what the
kernel returns -- all in mpmath at 40 significant digits (numpy / scipy only for starting points and condition numbers).
Also the seeded matrix families the tests run.  TEST INFRASTRUCTURE."""
import mpmath
import numpy as np
import scipy.linalg

DPS = 40
U = 2.220446049250313e-16


def _mp(A):
    return mpmath.matrix(np.asarray(A, dtype=np.float64).tolist())


def _np(M):
    return np.array([[float(M[i, j]) for j in range(M.cols)] for i in range(M.rows)])


def kron_operator(L, c):
    """I + c (I (x) L + L (x) I): vec(X + c (L X + X L')) with vec stacking columns."""
    n = L.shape[0]
    I = np.eye(n)
    return np.eye(n * n) + c * (np.kron(I, L) + np.kron(L, I))


def kappa_op(L, c):
    """2-norm condition of the Lyapunov operator (singular values of its Kronecker matrix); inf when singular."""
    s = np.linalg.svd(kron_operator(L, c), compute_uv=False)
    return float(s[0] / s[-1]) if s[-1] > 0 else np.inf


def _lyap_residual_mp(Lm, c, Bm, Xm):
    return Bm - (Xm + c * (Lm * Xm + Xm * Lm.T))


def lyap_ref(L, c, BP):
    """Reference X of X + c (L X + X L') = B_P (float64 rounding of a 40-digit solution).  n <= 8: the Kronecker system solved
    in mpmath; larger n: the float64 solution refined with mpmath residuals until the correction is below 1e-30 relative."""
    n = L.shape[0]
    with mpmath.workdps(DPS):
        cm = mpmath.mpf(float(c))
        Lm, Bm = _mp(L), _mp(BP)
        if n <= 8:
            Lk = np.kron(np.eye(n), L) + np.kron(L, np.eye(n))        # exact in float64: entries of L or sums of two
            K = mpmath.eye(n * n) + cm * mpmath.matrix(Lk.tolist())
            b = mpmath.matrix([Bm[i, j] for j in range(n) for i in range(n)])
            x = mpmath.lu_solve(K, b)
            Xm = mpmath.matrix(n, n)
            for j in range(n):
                for i in range(n):
                    Xm[i, j] = x[j * n + i]
        else:
            lu = scipy.linalg.lu_factor(kron_operator(L, float(c)))
            Xm = mpmath.matrix(n, n)
            for _ in range(12):
                R = _lyap_residual_mp(Lm, cm, Bm, Xm)
                d = scipy.linalg.lu_solve(lu, _np(R).reshape(-1, order="F")).reshape(n, n, order="F")
                Xm = Xm + _mp(d)
                if np.linalg.norm(d) <= 1e-30 * max(np.linalg.norm(_np(Xm)), 1e-300):
                    break
        return _np(Xm)


def dw_ref(L, c, X, C, BW):
    """Reference dW = (I + c L)^{-1} (B_W + c X C) in mpmath (X: the reference solution)."""
    n = L.shape[0]
    with mpmath.workdps(DPS):
        cm = mpmath.mpf(float(c))
        A = mpmath.eye(n) + cm * _mp(L)
        rhs = _mp(BW) + cm * (_mp(X) * _mp(C))
        out = np.empty(np.shape(BW))
        for k in range(out.shape[1]):
            x = mpmath.lu_solve(A, rhs.column(k))
            out[:, k] = [float(x[i]) for i in range(n)]
        return out


def inv_residual(A, Ainv):
    """||A Ainv - I||_F in mpmath."""
    with mpmath.workdps(DPS):
        R = _mp(A) * _mp(Ainv) - mpmath.eye(A.shape[0])
        return float(mpmath.mnorm(R, "F"))


def orth_residual(Q):
    """||Q'Q - I||_F in mpmath."""
    with mpmath.workdps(DPS):
        Qm = _mp(Q)
        return float(mpmath.mnorm(Qm.T * Qm - mpmath.eye(Q.shape[0]), "F"))


def _mpc(A):
    return _mp(np.real(A)) + mpmath.mpc(0, 1) * _mp(np.imag(A))


def similarity_residual(A, Q, T, rel=True):
    """||A - Q T Q^H||_F (/ ||A||_F) in mpmath; Q and T may be complex."""
    with mpmath.workdps(DPS):
        Qm = _mpc(Q)
        R = _mp(A) - Qm * _mpc(T) * Qm.H
        r = float(mpmath.mnorm(R, "F"))
        return r / float(np.linalg.norm(A)) if rel else r


def product_residual(H, L, G, D):
    """||H L G - D||_F in mpmath."""
    with mpmath.workdps(DPS):
        return float(mpmath.mnorm(_mp(H) * _mp(L) * _mp(G) - _mp(D), "F"))


def eigvals_ref(L):
    """Eigenvalues of L at 40 digits (complex128) and their condition numbers 1 / |y^H x| (unit x, y)."""
    with mpmath.workdps(DPS):
        ev, _ = mpmath.eig(_mp(L))
    lam = np.array([complex(e) for e in ev])
    w, vl, vr = scipy.linalg.eig(L, left=True, right=True)
    cond = np.empty(len(lam))
    for k, e in enumerate(lam):
        m = int(np.argmin(np.abs(w - e)))
        cond[k] = 1.0 / max(abs(np.vdot(vl[:, m], vr[:, m])) / (np.linalg.norm(vl[:, m]) * np.linalg.norm(vr[:, m])), 1e-300)
    return lam, cond


def kappa_v(L):
    """||V||_F ||V^{-1}||_F of the real eigenvector basis normalised as bdf_eig_basis does (columns Re x, Im x of a unit
    complex eigenvector x per pair, unit real eigenvectors).  Invariant under the phase of x and under the orthogonal Schur
    vectors, so computed from L's own eigenvectors.  inf when V is singular (defective L)."""
    with mpmath.workdps(DPS):
        E, ER = mpmath.eig(_mp(L))
    n = L.shape[0]
    lam = [complex(e) for e in E]
    tol = 1e-25 * max(float(np.linalg.norm(L)), 1e-300)      # (40-digit eigenvalues: imaginary parts of real ones ~1e-40)
    V = np.zeros((n, n))
    done = set()
    k = 0
    for a in range(n):
        if a in done:
            continue
        done.add(a)
        x = np.array([complex(ER[i, a]) for i in range(n)])
        x = x / np.linalg.norm(x)
        if abs(lam[a].imag) > tol:
            b = min((q for q in range(n) if q not in done), key=lambda q: abs(lam[q] - np.conj(lam[a])))
            done.add(b)
            V[:, k], V[:, k + 1] = x.real, x.imag
            k += 2
        else:
            V[:, k] = x.real / np.linalg.norm(x.real)
            k += 1
    with mpmath.workdps(DPS):
        Vm = _mp(V)
        try:
            Vi = mpmath.inverse(Vm)
        except ZeroDivisionError:
            return np.inf
        return float(mpmath.mnorm(Vm, "F") * mpmath.mnorm(Vi, "F"))


# ---------------------------------------------------------------------------------------------------------------------
# Matrix families (seeded)
# ---------------------------------------------------------------------------------------------------------------------
def mixed_spectrum(n, rng, scale=1.0):
    """Random dense nonsymmetric L = S D S^{-1} with about half of the spectrum in complex pairs, ||L||_2 = scale."""
    D = np.zeros((n, n))
    k = 0
    while k < n:
        if k + 1 < n and rng.random() < 0.5:
            a, b = rng.normal(), 0.3 + abs(rng.normal())
            D[k:k + 2, k:k + 2] = [[a, b], [-b, a]]
            k += 2
        else:
            D[k, k] = rng.normal()
            k += 1
    S = np.eye(n) + 0.3 * rng.normal(size=(n, n))
    L = S @ D @ np.linalg.inv(S)
    return L * (scale / np.linalg.norm(L, 2))


def jordan(n, lam=0.0, blocks=None):
    """Jordan matrix with eigenvalue lam: one block of size n (blocks=None) or the given block sizes."""
    blocks = blocks or [n]
    J = lam * np.eye(n)
    k = 0
    for s in blocks:
        for i in range(s - 1):
            J[k + i, k + i + 1] = 1.0
        k += s
    return J


def random_orthogonal(n, rng):
    q, r = np.linalg.qr(rng.normal(size=(n, n)))
    return q * np.sign(np.diag(r))


def real_block_schur(n, rng):
    """Q T Q' with T quasi-triangular whose leading 2 x 2 block [[1, 4], [0.5, 1]] has real eigenvalues 1 +- sqrt(2) and is
    left un-split: the kernel's QR iteration deflates it as a block (the exact zeros below make it a standing 2 x 2)."""
    T = np.triu(rng.normal(size=(n, n)) * 0.3)
    for i in range(n):
        T[i, i] = 3.0 + i
    T[0:2, 0:2] = [[1.0, 4.0], [0.5, 1.0]]
    return T


def repeated_pairs(n, eps, rng):
    """Two complex pairs -0.3 +- 2i and -0.3 +- (2 + eps) i (x/y-symmetric dynamics), the rest real and spread, in a random
    orthogonal basis."""
    D = np.zeros((n, n))
    D[0:2, 0:2] = [[-0.3, 2.0], [-2.0, -0.3]]
    D[2:4, 2:4] = [[-0.3, 2.0 + eps], [-2.0 - eps, -0.3]]
    for k in range(4, n):
        D[k, k] = -1.0 - 0.5 * k
    Q = random_orthogonal(n, rng)
    return Q @ D @ Q.T


def sym_rhs(n, rng):
    B = rng.normal(size=(n, n))
    return 0.5 * (B + B.T)
