"""The Newton solve of the backward BDF sweep (csrc/cpdp_bdf.cuh) against extended-precision references, at every state
dimension the kernel admits a representative of (NX = 1 .. 15, NC up to 31), on the thread emulation.

The probe kernel (tests/bdf_probe/bdf_probe.cuh) calls the kernel's own device functions in bdf_interval's order --
bdf_decompose (Schur form, eigenbasis and its kappa gate, warm refinement), bdf_factor, bdf_solve_cols -- on given
(L, C, c, [B_P | B_W]) and returns everything they leave behind.  tests/bdf_linalg_reference.py solves the same systems in
mpmath at 40 digits.  Every bound is  C * n * u * (condition)  with one constant C per property, fixed below; each run
prints the largest observed ratio of error to bound per property, path and dimension.

Two builds per dimension: the shipped configuration, and -DCPDP_BDF_EIG_KAPPA=0 (every solve on the Bartels-Stewart sweep,
so that the Schur vectors are returned and the sweep is checked on well-conditioned matrices too).

The accuracy contract of the eigen path: the solve is a two-sided similarity with G = Q V and H = V^{-1} Q', so its error
may grow with kappa_V^2 = (||G||_F ||H||_F)^2, up to 1e8 at the gate.  The largest eigen-path error reached on the
near-defective family is printed as 'solve X eig max rel err' and asserted below EIG_MAX_REL_ERR, far below the BDF Newton
iteration's own tolerance (its corrections are accepted at ~1e-3 relative)."""
import collections
import concurrent.futures as cf
import os

import numpy as np
import pytest

from tests import bdf_linalg_reference as ref
from tests.emu.bdf_probe_support import Probe, build_probe, schur_T

HERE = os.path.dirname(os.path.abspath(__file__))
U = ref.U
KAPPA = 1e4                    # CPDP_BDF_EIG_KAPPA
REFINE_TOL = 1e-13             # CPDP_BDF_REFINE_TOL
# (NX, NP): every NX in {1, 2, 3, 4, 5, 7, 8, 12, 13, 15}; NC = 31 (the largest the kernel admits) and NP = 1 at NX = 15
DIMS = [(1, 1), (2, 1), (3, 2), (4, 3), (5, 2), (7, 4), (8, 8), (12, 5), (13, 12), (15, 16), (15, 1)]
DIM_IDS = ["nx%d_np%d" % d for d in DIMS]
# the one constant of each bound
C_ORTH = 8.0                   # ||Q'Q - I||_F <= C n u
C_BACK = 8.0                   # ||L - Z T Z^H||_F / ||L||_F <= C n u
C_EIGVAL = 8.0                 # |lambda - lambda_ref| <= C n u ||L||_F cond(lambda)
C_SOLVE = 4.0                  # X, dW: rel err <= C n u kappa_op (sweep), C n u kappa_op kappa_V^2 (eigen path)
C_GJ = 4.0                     # ||A A^{-1} - I||_F <= C n u kappa_F(A)
C_WARM = 2.0                   # accepted refinement: ||G H - I||_F <= C n u ||G||_F ||H||_F
EIG_MAX_REL_ERR = 1e-9         # largest eigen-path solve error allowed anywhere in the suite

RATIOS = collections.defaultdict(float)


def record(what, path, n, ratio):
    key = (what, path, n)
    RATIOS[key] = max(RATIOS[key], float(ratio))


def report(config, title):
    tr = config.pluginmanager.get_plugin("terminalreporter")
    lines = ["%s: largest error / bound (constant) per property, path, NX" % title]
    for (what, path, n), r in sorted(RATIOS.items()):
        lines.append("  %-28s %-6s NX=%-3d %.3g" % (what, path, n, r))
    for ln in lines:
        (tr.write_line(ln) if tr is not None else print(ln))


@pytest.fixture(scope="module", autouse=True)
def _print_ratios(request):
    RATIOS.clear()
    yield
    report(request.config, "test_bdf_linalg (emulation)")


def build_all(device=False):
    """{(n, r): (shipped probe, sweep-only probe)}, built in parallel."""
    jobs = [(d, f) for d in DIMS for f in ((), ("-DCPDP_BDF_EIG_KAPPA=0",))]
    with cf.ThreadPoolExecutor(min(8, os.cpu_count() or 1)) as ex:
        sos = list(ex.map(lambda j: build_probe(j[0][0], j[0][1], device=device, flags=j[1]), jobs))
    out = {}
    for (d, f), so in zip(jobs, sos):
        out.setdefault(d, [None, None])[1 if f else 0] = Probe(so, device=device)
    return out


@pytest.fixture(scope="module")
def probes():
    return build_all()


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def families(n, seed=0):
    """[(name, L, kind)] for one dimension; kind: 'defective' (must take the sweep) or 'any'."""
    rng = np.random.default_rng(1000 * n + seed)
    out = []
    for s in (1e-3, 1.0, 1e3):
        for k in range(2):
            out.append(("mixed_%g_%d" % (s, k), ref.mixed_spectrum(n, rng, s), "any"))
    A = rng.normal(size=(n, n))
    out += [("symmetric", A + A.T, "any"), ("skew", A - A.T, "any"), ("triangular", np.triu(A), "any"),
            ("diagonal", np.diag(rng.normal(size=n)), "any"), ("zero", np.zeros((n, n)), "any")]
    if n >= 3:
        B = np.zeros((n, n))
        h = n // 2
        B[:h, :h], B[h:, h:] = rng.normal(size=(h, h)), rng.normal(size=(n - h, n - h))
        out.append(("block_diagonal", B, "any"))
        P = np.roll(np.eye(n), 1, axis=0)                      # cyclic shift: the standard shifts stall on it
        out.append(("cyclic", P, "any"))
    if n >= 2:
        out.append(("jordan0", ref.jordan(n, 0.0), "defective"))
        out.append(("jordan_m05", ref.jordan(n, -0.5), "defective"))
        out.append(("chains", ref.jordan(n, 0.0, [2] * (n // 2) + [1] * (n % 2)), "defective"))
        E = rng.normal(size=(n, n))
        for e in (1e-2, 1e-4, 1e-6, 1e-8, 1e-10):
            out.append(("near_defective_%g" % e, ref.jordan(n, -0.5, [2] * (n // 2) + [1] * (n % 2)) + e * E, "any"))
        out.append(("real_block", ref.real_block_schur(n, rng), "any"))
    if n >= 4:
        for e in (0.0, 1e-9, 1e-3):
            out.append(("pairs_%g" % e, ref.repeated_pairs(n, e, rng), "any"))
    return out


def rhs(n, nc, rng):
    B = rng.normal(size=(n, nc))
    B[:, :n] = ref.sym_rhs(n, rng)
    return B


def c_for(L, s=0.4):
    nl = np.linalg.norm(L, 2)
    return s / nl if nl > 0 else 0.1


def run_cases(pr, Ls, cs, seed=0):
    """Run single-step cases (or multi-step sequences, Ls of shape (cases, S, n, n)); returns (record, inputs)."""
    rng = np.random.default_rng(seed)
    Ls = np.asarray(Ls, dtype=np.float64)
    if Ls.ndim == 3:
        Ls = Ls[:, None]
    cases, S, n = Ls.shape[0], Ls.shape[1], pr.n
    C = rng.normal(size=(cases, S, n, pr.np_))
    B = np.stack([np.stack([rhs(n, pr.nc, rng) for _ in range(S)]) for _ in range(cases)])
    c = np.broadcast_to(np.asarray(cs, dtype=np.float64).reshape(cases, -1), (cases, S)).copy()
    return pr.run(Ls, C, c, B), dict(L=Ls, C=C, c=c, B=B)


def G_H(rec, idx):
    """G and H of an eigen-path record: QT holds G' (k-major G), Q holds H'."""
    return rec["QT"][idx].T, rec["Q"][idx].T


def D_of(rec, idx):
    """Real block-diagonal D from TD (a, b) and ROT's partner row."""
    TD, part = rec["TD"][idx], rec["ROT"][idx][3].astype(int)
    n = TD.shape[0]
    D = np.zeros((n, n))
    for j in range(n):
        D[j, j] = TD[j, 0]
        if part[j] != j:
            D[part[j], j] = -TD[j, 1] if part[j] > j else TD[j, 1]
    return D


# ---------------------------------------------------------------------------------------------------------------------
# checks (shared with tests/test_bdf_linalg_gpu.py)
# ---------------------------------------------------------------------------------------------------------------------
def check_solve(rec, inp, idx, path_tag=""):
    """X bitwise symmetric; X and dW against the references within C n u kappa (kappa_V^2 on the eigen path).
    Returns the relative error of X."""
    L, C, c, B = inp["L"][idx], inp["C"][idx], float(inp["c"][idx]), inp["B"][idx]
    n = L.shape[0]
    assert rec["fok"][idx] == 1, idx
    R = rec["R"][idx]
    X, dW = R[:, :n], R[:, n:]
    assert np.all(np.isfinite(R))
    assert np.array_equal(X, X.T), "X not bitwise symmetric"
    eig = rec["flag3"][idx] == 1
    path = "eig" if eig else "sweep"
    kv2 = 1.0
    if eig:
        G, H = G_H(rec, idx)
        kv2 = (np.linalg.norm(G) * np.linalg.norm(H)) ** 2
    kop = ref.kappa_op(L, c)
    Xr = ref.lyap_ref(L, c, B[:, :n])
    err = np.linalg.norm(X - Xr) / max(np.linalg.norm(Xr), 1e-300)
    r = err / (n * U * kop * kv2)
    record("solve X" + path_tag, path, n, r)
    if eig:
        record("solve X eig max rel err", path, n, err)
        assert err <= EIG_MAX_REL_ERR, err
    assert r <= C_SOLVE, (path, err, kop, kv2)
    if dW.size:
        Wr = ref.dw_ref(L, c, Xr, C, B[:, n:])
        kw = np.linalg.cond(np.eye(n) + c * L)
        errw = np.linalg.norm(dW - Wr) / max(np.linalg.norm(Wr), 1e-300)
        rw = errw / (n * U * max(kop, kw) * kv2)
        record("solve dW" + path_tag, path, n, rw)
        assert rw <= C_SOLVE, (path, errw, kop, kw, kv2)
    return err


def check_schur_sweep(rec, L, idx):
    """Sweep-path decomposition (the sweep-only build): Q orthogonal, L = Z T Z^H with Z = Q G^H, T triangular with exact
    zeros below the diagonal, eigenvalues against the reference."""
    n = L.shape[0]
    assert rec["dk"][idx] == 1 and rec["flag1"][idx] == 1
    Q = rec["Q"][idx]                                       # Q slot holds the Schur vectors Z[r][c]
    ro = ref.orth_residual(Q) / (n * U)
    record("schur Q'Q - I", "sweep", n, ro)
    assert ro <= C_ORTH, ro
    Tc = schur_T(rec, idx)
    Tr, Ti = rec["PV"][idx]
    assert np.all(np.tril(Tr, -1) == 0.0) and np.all(np.tril(Ti, -1) == 0.0), "complex T not triangular"
    rot = rec["ROT"][idx]
    Gr = np.zeros((n, n), dtype=complex)
    for i in range(n):
        Gr[i, i] = rot[0, i]
        p = int(rot[3, i])
        if p != i:
            Gr[i, p] = rot[1, i] + 1j * rot[2, i]
    assert np.linalg.norm(Gr.conj().T @ Gr - np.eye(n)) <= 8 * U * n
    Z = Q @ Gr.conj().T
    if np.linalg.norm(L) > 0:
        rb = ref.similarity_residual(L, Z, Tc) / (n * U)
        record("schur L - ZTZ^H", "sweep", n, rb)
        assert rb <= C_BACK, rb
    else:
        assert np.all(Tc == 0)
    return Tc


def check_eigvals(L, lam, tag="sweep"):
    n = L.shape[0]
    lr, cond = ref.eigvals_ref(L)
    nl = max(np.linalg.norm(L), 1e-300)
    for k, e in enumerate(lr):
        d = np.abs(lr - e)
        d[k] = np.inf
        if d.min() <= 1e-3 * nl or cond[k] > 1e6:
            continue                                        # (not well separated / ill-conditioned: no per-eigenvalue claim)
        err = np.abs(lam - e).min()
        r = err / (n * U * nl * cond[k])
        record("eigenvalues", tag, n, r)
        assert r <= C_EIGVAL, (e, err, cond[k])


def check_quasi_triangular(Tr):
    assert np.all(np.tril(Tr, -2) == 0.0), "nonzero below the subdiagonal"
    sub = np.diag(Tr, -1)
    assert not np.any((sub[:-1] != 0.0) & (sub[1:] != 0.0)), "two consecutive nonzero subdiagonal entries"


def check_eig_record(rec, L, idx):
    """Eigen-path decomposition: kappa of the returned G, H within the gate; H L G = D; real T quasi-triangular."""
    n = L.shape[0]
    G, H = G_H(rec, idx)
    kv = np.linalg.norm(G) * np.linalg.norm(H)
    assert kv <= KAPPA, kv
    D = D_of(rec, idx)
    part = rec["ROT"][idx][3].astype(int)
    assert np.all(rec["TD"][idx][part != np.arange(n), 1] > 0.0), "complex pair with b <= 0"
    if rec["dk"][idx] == 1 or rec["dk"][idx] == 3:
        check_quasi_triangular(rec["PV"][idx][0])
    res = ref.product_residual(H, L, G, D)
    r = res / (n * U * max(np.linalg.norm(L), 1e-300) * kv * kv)
    record("eig H L G - D", "eig", n, r)
    assert r <= C_BACK, (res, kv)
    return kv


# ---------------------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------------------
def eig_gap(L):
    """Smallest distance between two eigenvalues.  The eigen path is promised to well-conditioned bases of DISTINCT
    eigenvalues: bdf_eig_basis perturbs nothing, so an exactly repeated eigenvalue of a diagonalisable L (the zero matrix,
    exactly repeated pairs) divides by lambda_i - lambda_j = 0 and goes to the sweep like a defective one."""
    lam = np.linalg.eigvals(L)
    d = np.abs(lam[:, None] - lam[None, :]) + np.diag(np.full(len(lam), np.inf))
    return float(d.min()) if len(lam) > 1 else np.inf


def schur_and_solve(pr_ship, pr_sweep, n):
    fam = families(n)
    Ls = [f[1] for f in fam]
    cs = [c_for(L) for L in Ls]
    recs, inp = run_cases(pr_sweep, Ls, cs, seed=n)
    rece, inpe = run_cases(pr_ship, Ls, cs, seed=n)
    for k, (name, L, kind) in enumerate(fam):
        idx = (k, 0)
        Tc = check_schur_sweep(recs, L, idx)
        if name.startswith("mixed") or name in ("symmetric", "skew", "real_block", "cyclic"):
            check_eigvals(L, np.diag(Tc))
        check_solve(recs, inp, idx)
        # shipped build
        assert rece["dk"][idx] == 1, name
        if rece["flag3"][idx]:
            check_eig_record(rece, L, idx)
        else:
            assert np.array_equal(rece["R"][idx], recs["R"][idx]), "sweep path differs from the sweep-only build"
        check_solve(rece, inpe, idx)
        kv = ref.kappa_v(L) if kind != "defective" else np.inf
        if kv <= 1e2 and eig_gap(L) > 1e-6 * np.linalg.norm(L):
            assert rece["flag3"][idx] == 1, (name, kv)
        if kind == "defective":
            assert rece["flag3"][idx] == 0, name
    return fam, recs, rece


@pytest.mark.parametrize("dim", DIMS, ids=DIM_IDS)
def test_schur_eigen_gate_and_newton_solve(probes, dim):
    """Every family at every dimension on both builds: Schur form, eigen gate, Newton solve (X and dW)."""
    pr_ship, pr_sweep = probes[dim]
    n = dim[0]
    fam, recs, rece = schur_and_solve(pr_ship, pr_sweep, n)
    names = [f[0] for f in fam]
    if n >= 2:      # the 2 x 2 block with real eigenvalues stays a standing block and reaches bdf_eig_basis's disc >= 0 branch
        k = names.index("real_block")
        assert rece["flag3"][k, 0] == 1
        Tr = rece["PV"][k, 0][0]
        assert Tr[1, 0] != 0.0 and np.all(rece["TD"][k, 0][:2, 1] == 0.0)
        assert list(rece["ROT"][k, 0][3][:2].astype(int)) == [0, 1]
    if n >= 2:      # the near-defective family crosses the gate from both sides
        fl = [rece["flag3"][names.index("near_defective_%g" % e), 0] for e in (1e-2, 1e-10)]
        assert fl[0] == 1 and fl[1] == 0, fl


@pytest.mark.parametrize("dim", [d for d in DIMS if d[0] >= 2], ids=[i for d, i in zip(DIMS, DIM_IDS) if d[0] >= 2])
def test_scale_equivariance(probes, dim):
    """L scaled by 2^k, k = -40, -20, ..., 40: every operation of the Schur iteration commutes with a power-of-two scaling,
    so T scales exactly and the Schur vectors do not change (bitwise on the emulation)."""
    pr = probes[dim][1]
    n = dim[0]
    L = ref.mixed_spectrum(n, np.random.default_rng(7 + n), 1.0)
    ks = list(range(-40, 41, 20))
    rec, _ = run_cases(pr, [L * 2.0 ** k for k in ks], [0.1 * 2.0 ** -k for k in ks])
    base = ks.index(0)
    for i, k in enumerate(ks):
        assert np.array_equal(rec["Q"][i, 0], rec["Q"][base, 0]), k
        assert np.array_equal(rec["TD"][i, 0], rec["TD"][base, 0] * 2.0 ** k), k
        assert np.array_equal(rec["T2S"][i, 0], rec["T2S"][base, 0] * 2.0 ** k), k


def singular_cases(n):
    """(L, c, singular) with L upper triangular with diagonal 1, 2, ..., n (the Schur form keeps its diagonal exactly).
    singular = True: 1 + c (l_i + l_j) = 0 exactly, for c = -1/2 (i = j = 0) and c = -1/4 (i = j = 1);  False: c within
    (1 +- delta) of -1/2;  None: c = fl(-1/3), where 1 + 3c = 5.6e-17 is zero only after rounding the product -- an
    FMA-contracted pivot (the device build) sees a nonsingular operator with kappa ~ 1e16, the separately rounded one (the
    emulation) a singular one; either answer is right, provided a reported success carries finite output."""
    rng = np.random.default_rng(50 + n)
    L = np.triu(rng.normal(size=(n, n)) * 0.3, 1) + np.diag(np.arange(1.0, n + 1))
    out = [(L, -0.5, True)]
    if n >= 2:
        out += [(L, -0.25, True), (L, -1.0 / 3.0, None)]
    for d in (1e-3, 1e-6, 1e-10):
        out += [(L, -0.5 * (1 + d), False), (L, -0.5 * (1 - d), False)]
    return out


def check_singular(rec, inp, cases, tag=" near-singular c"):
    for k, (L, c, sing) in enumerate(cases):
        idx = (k, 0)
        assert rec["dk"][idx] == 1
        if sing:
            assert rec["fok"][idx] == 0, (c, rec["flag3"][idx])
        elif sing is None:
            assert rec["fok"][idx] == 0 or np.all(np.isfinite(rec["R"][idx])), c
        else:
            assert rec["fok"][idx] == 1
            check_solve(rec, inp, idx, tag)


@pytest.mark.parametrize("dim", DIMS, ids=DIM_IDS)
def test_singular_operator(probes, dim):
    """An exactly singular operator makes bdf_factor return false on both paths (never non-finite output reported as
    true); close to singular it solves within the kappa_op bound."""
    n = dim[0]
    cases = singular_cases(n)
    for pr in probes[dim]:
        rec, inp = run_cases(pr, [c[0] for c in cases], [c[1] for c in cases], seed=3)
        check_singular(rec, inp, cases)
    assert rec["flag3"][0, 0] == 0        # (the sweep-only build)


def gj_matrices(n, rng):
    out = [rng.normal(size=(n, n)), np.eye(n) + 0.1 * rng.normal(size=(n, n)), rng.normal(size=(n, n)) * 1e150,
           rng.normal(size=(n, n)) * 1e-150]
    P = np.eye(n)[rng.permutation(n)]
    out.append(P @ np.diag(rng.uniform(1, 2, size=n)))                     # needs the row exchanges
    if n >= 2:
        A = rng.normal(size=(n, n))
        A[np.arange(n), np.arange(n)] = 0.0                                  # zero diagonal
        out.append(A)
    return out


@pytest.mark.parametrize("dim", DIMS, ids=DIM_IDS)
def test_gauss_jordan(probes, dim):
    """bdf_gauss_jordan: residual within C n u kappa; a zero pivot column returns false and leaves no output."""
    pr = probes[dim][0]
    n = dim[0]
    rng = np.random.default_rng(90 + n)
    mats = gj_matrices(n, rng)
    sing = []
    z = rng.normal(size=(n, n))
    z[:, n // 2] = 0.0
    sing.append(z)
    sing.append(np.zeros((n, n)))
    ok, inv = pr.gj(np.stack(mats + sing))
    for k, A in enumerate(mats):
        assert ok[k] == 1 and np.all(np.isfinite(inv[k])), k
        kap = np.linalg.cond(A, "fro")
        r = ref.inv_residual(A, inv[k]) / (n * U * kap)
        record("gauss-jordan A A^-1 - I", "-", n, r)
        assert r <= C_GJ, (k, r)
    for k in range(len(mats), len(mats) + len(sing)):
        assert ok[k] == 0 and np.all(inv[k] == 0.0), k


# ---- warm refinement ------------------------------------------------------------------------------------------------
def warm_sequences(n, rng):
    """[(name, L0, L1, expect)] with expect in {'accept', 'reject', 'any'}."""
    out = []
    L0 = ref.mixed_spectrum(n, rng, 1.0)
    E = rng.normal(size=(n, n))
    E /= np.linalg.norm(E)
    for d in (1e-8, 1e-6, 1e-4, 1e-3, 1e-2, 1e-1):
        out.append(("delta_%g" % d, L0, L0 + d * E, "accept" if d <= 1e-6 else "any"))
    if n >= 2:
        Q = ref.random_orthogonal(n, rng)
        D = np.diag(-1.0 - np.arange(n, dtype=float))

        def blk(a, s):                                         # 2 x 2 leading block: a pair (s > 0) or two reals (s < 0)
            M = D.copy()
            M[0:2, 0:2] = [[a, 1.0], [-s, a]]
            return Q @ M @ Q.T
        out.append(("pair_to_reals", blk(0.3, 0.04), blk(0.3, -0.04), "reject"))
        out.append(("reals_to_pair", blk(0.3, -0.04), blk(0.3, 0.04), "reject"))
        M0 = D.copy()
        M0[0:2, 0:2] = [[0.3, 0.5], [-0.5, 0.3]]
        M1 = D.copy()
        M1[0:2, 0:2] = [[0.3, -0.5], [0.5, 0.3]]
        out.append(("pair_conjugated", Q @ M0 @ Q.T, Q @ M1 @ Q.T, "reject"))
        M0 = D.copy()
        M0[0, 0], M0[1, 1] = -1.0, -1.2
        M1 = D.copy()
        M1[0, 0], M1[1, 1] = -1.2, -1.0
        M0[0, 1] = M1[0, 1] = 0.3
        out.append(("reals_cross", Q @ M0 @ Q.T, Q @ M1 @ Q.T, "any"))
    return out


def check_warm(rec2, inp2, rec1, n, expect, name):
    """rec2: (L0, L1) sequences; rec1: L1 cold, each as its own single-step case (same inputs as step 1 of rec2)."""
    for k in range(len(expect)):
        i2, i1 = (k, 1), (k, 0)
        if rec2["flag3"][k, 0] != 1:
            assert rec2["dk"][i2] == 1
            continue
        dk = rec2["dk"][i2]
        assert dk in (2, 3), (name[k], dk)
        if expect[k] == "accept":
            assert dk == 2, name[k]
        if expect[k] == "reject":
            assert dk == 3, name[k]
        if dk == 2:
            L1 = inp2["L"][i2]
            G, H = G_H(rec2, i2)
            kv = np.linalg.norm(G) * np.linalg.norm(H)
            assert kv <= KAPPA
            part = rec2["ROT"][i2][3].astype(int)
            assert np.all(rec2["TD"][i2][part != np.arange(n), 1] > 0.0), "accepted with a pair b <= 0"
            res = ref.product_residual(H, L1, G, D_of(rec2, i2))
            record("warm H L1 G - D / ||L1||", "eig", n, res / (REFINE_TOL * np.linalg.norm(L1)))
            assert res <= REFINE_TOL * np.linalg.norm(L1), (name[k], res)
            rg = np.linalg.norm(G @ H - np.eye(n)) / (n * U * kv)
            record("warm G H - I", "eig", n, rg)
            assert rg <= C_WARM * 1e3 or np.linalg.norm(G @ H - np.eye(n)) <= 1e-12, rg
            check_solve(rec2, inp2, i2, " warm")
            e1 = rec1["R"][i1][:, :n]
            e2 = rec2["R"][i2][:, :n]
            assert np.linalg.norm(e2 - e1) <= 2 * C_SOLVE * n * U * ref.kappa_op(L1, inp2["c"][i2]) * kv ** 2 * np.linalg.norm(e1)
        else:
            # a rejected refinement leaves exactly what a cold decomposition of L1 leaves
            assert rec1["dk"][i1] == 1 and rec2["flag3"][i2] == rec1["flag3"][i1], name[k]
            eig = rec1["flag3"][i1] == 1
            for key in ("Q", "QT", "TD", "PV", "WT", "R"):
                assert np.array_equal(rec2[key][i2], rec1[key][i1]), (name[k], key)
            assert np.array_equal(rec2["ROT"][i2][3], rec1["ROT"][i1][3]), name[k]
            if not eig:
                assert np.array_equal(rec2["ROT"][i2], rec1["ROT"][i1]) and np.array_equal(rec2["T2S"][i2], rec1["T2S"][i1])
            else:
                assert np.array_equal(rec2["T2S"][i2].reshape(-1)[:n * n], rec1["T2S"][i1].reshape(-1)[:n * n])


def run_warm(pr, seqs, seed=11):
    """Each (L0, L1) as a two-step case, and L1 alone as a one-step case with the same C, c, B."""
    n = pr.n
    L2 = np.stack([np.stack([s[1], s[2]]) for s in seqs])
    cs = np.array([[c_for(s[1]), c_for(s[2])] for s in seqs])
    rec2, inp2 = run_cases(pr, L2, cs, seed=seed)
    rec1 = pr.run(inp2["L"][:, 1:], inp2["C"][:, 1:], inp2["c"][:, 1:], inp2["B"][:, 1:])
    return rec2, inp2, rec1


@pytest.mark.parametrize("dim", [d for d in DIMS if d[0] >= 2], ids=[i for d, i in zip(DIMS, DIM_IDS) if d[0] >= 2])
def test_warm_refinement(probes, dim):
    """Accepted refinements meet the r8 conditions in mpmath and solve like a cold decomposition; rejected ones leave,
    bit for bit, a cold decomposition of the new L; pair-structure changes are rejected; small steps are accepted."""
    pr = probes[dim][0]
    n = dim[0]
    seqs = warm_sequences(n, np.random.default_rng(300 + n))
    rec2, inp2, rec1 = run_warm(pr, seqs)
    check_warm(rec2, inp2, rec1, n, [s[3] for s in seqs], [s[0] for s in seqs])
    assert rec2["flag3"][0, 0] == 1 and rec2["dk"][0, 1] == 2, "small step on a well-conditioned L not accepted"


# ---- the quadrotor's Jacobians --------------------------------------------------------------------------------------
def quad_jacobians():
    """L = A' - P R at the 51 nodes of the six oracle_quad50 cases, P from the oracle's backward BDF sweep, as in
    tools/eig_refine_drift.py; also C = R W - r_.  Node order backwards (the sweep's order)."""
    from oracle import models
    from oracle.cpdp_oracle import Oracle
    z = np.load(os.path.join(HERE, "golden", "oracle_quad50.npz"))
    N, T = int(z["n_grid"]), float(z["T"])
    orc = Oracle(models.quadrotor(), n_grid=N)
    Ls, Cs = [], []
    for case in range(z["X"].shape[0]):
        orc.pd = z["pdata"][case]
        X, Uc, Lam, th = z["X"][case], z["U"][case], z["Lam"][case], z["theta"][case]
        tg = np.linspace(0, T, N + 1)
        _, _, PW = orc.aux(tg, X, Uc, Lam, th, back={"method": "BDF"}, fwd={})
        n = X.shape[1]
        rowL, rowC = [], []
        for k in range(N, -1, -1):
            fx, fu, fe, Hxx, Hxu, Hxe, Huu, Hue, iH = orc._coeffs(X[k], Uc[k], Lam[k], th, tg[k])
            G = fu @ iH
            P = PW[k, :n * n].reshape(n, n)
            W = PW[k, n * n:].reshape(n, -1)
            R = G @ fu.T
            rowL.append((fx - G @ Hxu.T).T - P @ R)
            rowC.append(R @ W - (fe - G @ Hue))
        Ls.append(rowL)
        Cs.append(rowC)
    return np.array(Ls), np.array(Cs)


@pytest.fixture(scope="module")
def quad_L():
    return quad_jacobians()


def quad_run(pr, quad_L, step_fraction=0.05):
    Ls, Cs = quad_L
    cases, S, n = Ls.shape[0], Ls.shape[1], Ls.shape[2]
    rng = np.random.default_rng(5)
    B = np.stack([np.stack([rhs(n, pr.nc, rng) for _ in range(S)]) for _ in range(cases)])
    c = np.array([[-step_fraction / max(np.linalg.norm(L, 2), 1e-300) for L in row] for row in Ls])
    seq = pr.run(Ls, Cs, c, B)
    cold = pr.run(Ls.reshape(cases * S, 1, n, n), Cs.reshape(cases * S, 1, n, -1), c.reshape(-1, 1),
                  B.reshape(cases * S, 1, n, -1))
    return seq, cold, dict(L=Ls, C=Cs, c=c, B=B)


def test_quadrotor_jacobians(probes, quad_L):
    """The quadrotor's 6 x 51 Jacobians (NX = 13, NP = 7 in the model; the probe's NP = 12 carries C in its first 7
    columns), in the sweep's order as one sequence per case (warm refinements) and each on its own (cold): every solve
    within its bound, the terminal node (integrator chains, defective) on the sweep."""
    pr = probes[(13, 12)][0]
    Ls, Cs = quad_L
    Cp = np.zeros(Ls.shape[:2] + (13, 12))
    Cp[..., :Cs.shape[-1]] = Cs
    seq, cold, inp = quad_run(pr, (Ls, Cp))
    cases, S = Ls.shape[:2]
    cold = {k: (v.reshape((cases, S) + v.shape[2:]) if isinstance(v, np.ndarray) else v) for k, v in cold.items()}
    dks = collections.Counter(seq["dk"].reshape(-1).tolist())
    for a in range(cases):
        assert seq["flag3"][a, 0] == 0 and cold["flag3"][a, 0] == 0, "terminal node must fall back to the sweep"
        for s in range(S):
            check_solve(seq, inp, (a, s), " quadrotor")
            check_solve(cold, inp, (a, s), " quadrotor")
            if seq["flag3"][a, s] and seq["dk"][a, s] != 2:
                check_eig_record(seq, Ls[a, s], (a, s))
            if seq["dk"][a, s] == 3:
                for key in ("Q", "QT", "TD", "PV", "WT", "R"):
                    assert np.array_equal(seq[key][a, s], cold[key][a, s]), (a, s, key)
    assert dks[2] > 0.5 * cases * S, dks


# ---- a one-state model end to end -------------------------------------------------------------------------------------
GRAD_RTOL = 1e-5               # tests/test_gpu_parity.py's parity tolerance of dL/dtheta


def one_state_models():
    """The same one-state problem as an OracleModel and a COCSys: x' = a x + u, path th0 x^2 + 0.1 u^2, final th1 x^2."""
    import sympy as sp
    from lfsd_b200.CPDP import COCSys
    from lfsd_b200.sx import SX
    from oracle.models import OracleModel
    xs, us, t0, t1 = (sp.Symbol(s, real=True) for s in ("x", "u", "th0", "th1"))
    om = OracleModel("onestate", [xs], [us], [t0, t1], [0.3 * xs + us], t0 * xs ** 2 + 0.1 * us ** 2, t1 * xs ** 2, sel=[0])
    x, u, th = SX.sym('x', 1), SX.sym('u', 1), SX.sym('th', 2)
    oc = COCSys("onestate")
    oc.setAuxvarVariable(th)
    oc.setStateVariable(x)
    oc.setControlVariable(u)
    oc.setDyn(0.3 * x[0] + u[0])
    oc.setPathCost(th[0] * x[0] * x[0] + 0.1 * u[0] * u[0])
    oc.setFinalCost(th[1] * x[0] * x[0])
    return om, oc


def _host(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def one_state_check(oc):
    """Mode 1 (BDF) of the one-state model against the oracle running scipy's BDF with the closed-form Jacobian: same
    backward right-hand-side count, dL/dtheta within GRAD_RTOL."""
    from oracle.cpdp_oracle import Oracle
    om, _ = one_state_models()
    N, th, x0 = 10, np.array([1.0, 2.0]), np.array([1.0])
    oc.setIntegrator(n_grid=N)
    oc.aux_mode = oc.MODE_BDF
    oc.rtol_back, oc.atol_back, oc.rtol_fwd, oc.atol_fwd = 1e-3, 1e-6, 1e-3, 1e-6
    sol = oc.cocSolverBatch(x0.reshape(1, 1), 1.0, th)
    taus, wp = np.array([0.3, 0.8]), np.array([[[0.5], [0.2]]])
    aux = oc.auxSysSolverBatch(sol, taus, wp, [0])
    orc = Oracle(om, n_grid=N)
    tg, X, Uo, Lam = orc.solve(x0, 1.0, th)
    assert np.abs(_host(sol["X"])[0] - X).max() < 1e-8
    Xa, Ua, PW, cnt = orc.aux(tg, X, Uo, Lam, th, back={"method": "BDF", "jac": "closed"}, fwd={}, return_counts=True)
    loss, dl = orc.loss_grad(taus, wp[0], tg, X, Xa, sel=[0])
    assert int(_host(aux["aux_status"])[0]) == 0
    cn = _host(aux["counters"])[0]
    assert int(cn[0]) == cnt["back_rhs"], (cn, cnt)
    dth = _host(aux["dtheta"])[0]
    assert abs(float(_host(aux["loss"])[0]) - loss) <= 1e-9 * max(1.0, loss)
    assert np.linalg.norm(dth - dl) <= GRAD_RTOL * np.linalg.norm(dl), (dth, dl)
    return dth, dl


def test_one_state_model_bdf_matches_oracle():
    """NX = 1: the full kernel library builds (the sweep's terms per lane were 0 there) and its BDF sweep matches the
    oracle, on the eigen path and on the sweep-only build."""
    import hashlib
    from lfsd_b200 import _capi, codegen
    from tests.emu.build_emu import build
    from tests.emu.support import NumpyMem, _BUILD
    for flags in ([], ["-DCPDP_BDF_EIG_KAPPA=0"]):
        _, oc = one_state_models()
        text, _ = codegen.generate_model_header("onestate", oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost,
                                                oc.final_cost, oc.pvar)
        src = "".join(open(os.path.join(_capi.CSRC, fn)).read() for fn in sorted(os.listdir(_capi.CSRC))
                      if os.path.isfile(os.path.join(_capi.CSRC, fn)))
        src += open(os.path.join(HERE, "emu", "emu_lib.cpp")).read()
        tag = hashlib.sha1((text + src + " ".join(flags)).encode()).hexdigest()[:12]
        os.makedirs(_BUILD, exist_ok=True)
        hdr = os.path.join(_BUILD, "model_onestate_%s.cuh" % tag)
        so = os.path.join(_BUILD, "libemu_onestate_%s.so" % tag)
        if not os.path.exists(so):
            with open(hdr, "w") as f:
                f.write(text)
            build(hdr, so, ns="cpdp_emu_onestate", extra=["-DCPDP_WITH_BDF"] + flags)
        oc._lib = _capi.CpdpLib(so)
        oc._mem = NumpyMem()
        one_state_check(oc)
