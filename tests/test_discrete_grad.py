"""Discrete auxiliary mode (cpdp_aux mode 2, COCSys.MODE_DISCRETE): dx/dtheta, du/dtheta and dL/dtheta as the exact derivative
of the solver's own output.  CPU tests: the kernels of csrc/cpdp_disc.cuh run in the thread emulation of tests/emu/ through the
same C ABI and COCSys host class as on the GPU, against the dense implicit-differentiation oracle of tests/discrete_oracle.py."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import sympy as sp

from tests.emu.support import emu_oc, _BUILD
from tests.emu.disc_support import emu_disc_oc
from tests.emu.build_emu import CSRC
from tests.discrete_oracle import DiscreteOracle, _fd
from oracle import models

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DISC = 2


def _rel(a, b, floor=1e-300):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), floor)


def _fx(name):
    return np.load(os.path.join(HERE, "golden", "oracle_%s.npz" % name))


def host_sol(oc, T, th, X, U, Lam, pd=None, status=None):
    """cocSolverBatch-shaped dict around a trajectory given on the host (B = X.shape[0])."""
    mem = oc._device()
    B = X.shape[0]
    thd, ths = oc._theta_arg(np.asarray(th, dtype=float), B)
    return dict(B=B, horizon=float(T), theta=thd, theta_stride=ths,
                pdata=None if pd is None else mem.from_host(np.asarray(pd, dtype=float).reshape(B, -1)),
                X=mem.from_host(X), U=mem.from_host(U), Lam=mem.from_host(Lam),
                status=None if status is None else mem.from_host(np.asarray(status), "i4"))


# fixture, standard model, oracle model, observed states
CASES = {
    "pendulum": ("pendulum", lambda: models.pendulum(), [0]),
    "robotarm": ("robotarm", lambda: models.robotarm(), [0, 1]),
    "rocket": ("rocket", lambda: models.rocket(), [0, 1, 2, 6, 7, 8, 9]),
    "quadkat": ("quadrotor", lambda: models.quadrotor(), [0, 1, 2]),
    "quad50": ("quadrotor", lambda: models.quadrotor(), [0, 1, 2]),
    "pendulum_tw2": ("pendulum_tw2", lambda: models.pendulum_timewarp(2), [0]),
}


def _case(fix, layout_probe=False):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = (emu_disc_oc if layout_probe else emu_oc)(name, n_grid=N)
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    orc = DiscreteOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    return oc, orc, fx, pd, sel


# ------------------------------------------------------------------------------------------------ code generation
_PROBE = r"""
#include "cpdp_port.h"
#include MODEL
extern "C" __attribute__((visibility("default"))) void probe(const double* x, const double* u, const double* th, const double* pd,
        const double* mu, double w, const double* dx, const double* du, const double* dth, double* df, double* hz) {
    Model::dir_th(x, u, th, pd, mu, w, dx, du, dth, df, hz);
}
"""


@pytest.mark.parametrize("name", ["pendulum", "pendulum_tw2", "robotarm", "rocket", "quadrotor", "cartpole", "robotarm_wd",
                                  "quadrotor_cost1", "quadrotor_cost2", "rocket_cost1"])
def test_dir_th_matches_sympy(name):
    """Model::dir_th of the generated C (compiled with g++) = fx dx + fu du + fth dth and Hzz dz + Hztheta dth from sympy."""
    from lfsd_b200 import standard, codegen
    oc = (standard.STANDARD.get(name) or standard.VARIANTS[name])()
    text, info = codegen.generate_model_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost,
                                               oc.pvar, time=getattr(oc, "time", None))
    assert info["ops_dir_th"] > 0
    os.makedirs(_BUILD, exist_ok=True)
    hdr = os.path.join(_BUILD, "dirth_%s_%s.cuh" % (name, info["hash"]))
    so = hdr[:-4] + ".so"
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        src = hdr[:-4] + ".cpp"
        with open(src, "w") as f:
            f.write(_PROBE)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", CSRC, '-DMODEL="%s"' % hdr, src, "-o", so])
    L = ctypes.CDLL(so)
    x, u, th = codegen._vec(oc.state), codegen._vec(oc.control), codegen._vec(oc.auxvar)
    pdv = (codegen._vec(oc.pvar) if oc.n_pvar else []) + (codegen._vec(oc.time) if getattr(oc, "time", None) is not None else [])
    n, m, r, q = len(x), len(u), len(th), len(pdv)
    f = sp.Matrix(codegen._vec(oc.dyn))
    c = codegen._to_matrix(oc.path_cost)[0, 0]
    mu = [sp.Symbol("mu_%d" % i, real=True) for i in range(n)]
    w = sp.Symbol("w_", real=True)
    ham = w * c + sum(mu[i] * f[i] for i in range(n))
    hz = sp.Matrix([ham]).jacobian(x + u).T
    fn = sp.lambdify([x, u, th, pdv, mu, w], [f.jacobian(x + u), f.jacobian(th), hz.jacobian(x + u), hz.jacobian(th)], modules="numpy")
    rng = np.random.default_rng(7)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    worst = 0.0
    for _ in range(5):
        xv, uv, tv, pv = rng.normal(size=n), rng.normal(size=m), rng.uniform(0.5, 1.5, size=r), rng.normal(size=max(q, 1))
        if n == 13:
            xv[6:10] /= np.linalg.norm(xv[6:10])
        muv, wv = rng.normal(size=n), float(rng.uniform(0.01, 0.1))
        dx, du, dth = rng.normal(size=n), rng.normal(size=m), rng.normal(size=r)
        df, hzo = np.zeros(n), np.zeros(n + m)
        L.probe(P(xv), P(uv), P(tv), P(pv), P(muv), ctypes.c_double(wv), P(dx), P(du), P(dth), P(df), P(hzo))
        fz, fth, hzz, hzth = (np.array(a, dtype=float) for a in fn(xv, uv, tv, pv[:q], muv, wv))
        dz = np.concatenate([dx, du])
        df_ref, hz_ref = fz @ dz + fth @ dth, hzz @ dz + hzth @ dth
        e = max(_rel(df, df_ref, 1e-12), _rel(hzo, hz_ref, 1e-12))
        worst = max(worst, e)
    print("%s: dir_th vs sympy, worst relative error %.2e" % (name, worst))
    assert worst < 1e-12


# ------------------------------------------------------------------------------------------------ stage level
@pytest.mark.parametrize("fix", ["pendulum", "quadkat", "pendulum_tw2"])
def test_stage_theta_vs_oracle(fix):
    """E_k, Hth_k written by k_stage_theta = the oracle's analytic stage recursion (1e-10) = finite differences of
    interval_derivs (1e-6)."""
    oc, orc, fx, pd, sel = _case(fix, layout_probe=True)
    N, S, n, m, r = oc.n_grid, oc.steps_per_grid, oc.n_state, oc.n_control, oc.n_auxvar
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    oc.auxSysSolverBatch(sol, fx["taus"][:1], fx["wp"][:1], sel, mode=DISC, phases=1)
    ws = oc._workspace(1)
    L = oc._lib.L
    L.cpdp_emu_disc_offset.restype = ctypes.c_size_t
    L.cpdp_emu_disc_offset.argtypes = [ctypes.c_int] * 4
    oH, oE = L.cpdp_emu_disc_offset(1, N, S, 0), L.cpdp_emu_disc_offset(1, N, S, 1)
    Hth = ws[oH:oH + N * (n + m) * r * 8].view(np.float64).reshape(N, n + m, r)
    E = ws[oE:oE + N * n * r * 8].view(np.float64).reshape(N, n, r)
    tg = oc._time_grid(T, N)
    DT = T / N / S
    e_or = e_fd = 0.0
    for k in range(N):
        Eo, Ho = orc.interval_theta_derivs(X[k], U[k], th, Lam[k + 1], DT, tg[k])
        e_or = max(e_or, _rel(E[k], Eo, 1e-300), _rel(Hth[k], Ho, 1e-300))
        if k % max(1, N // 4) == 0:
            Ef = np.stack([_fd(lambda t: orc.interval_derivs(X[k], U[k], t, Lam[k + 1], DT, tg[k])[0], th, i) for i in range(r)], 1)
            Hf = np.stack([_fd(lambda t: orc.interval_derivs(X[k], U[k], t, Lam[k + 1], DT, tg[k])[5], th, i) for i in range(r)], 1)
            e_fd = max(e_fd, _rel(Eo, Ef), _rel(Ho, Hf))
    print("%s: stage arrays vs oracle %.2e, oracle vs finite differences %.2e" % (fix, e_or, e_fd))
    assert e_or < 1e-10
    assert e_fd < 1e-6


# ------------------------------------------------------------------------------------------------ end to end against the oracle
@pytest.mark.parametrize("fix", list(CASES))
def test_mode2_vs_dense_oracle(fix):
    oc, orc, fx, pd, sel = _case(fix)
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:1], fx["wp"][:1], sel, mode=DISC)
    assert int(aux["aux_status"][0]) == 0 and not aux["counters"].any()
    tg = oc._time_grid(T, oc.n_grid)
    Xa, Ua = orc.aux_discrete(tg, X, U, Lam, th)
    loss, dl = orc.loss_grad(fx["taus"][0], fx["wp"][0], tg, X, Xa, sel=sel)
    errs = (_rel(aux["Xa"][0], Xa), _rel(aux["Ua"][0], Ua), abs(aux["loss"][0] - loss) / max(abs(loss), 1e-300),
            _rel(aux["dtheta"][0], dl))
    print("%s: Xa %.2e Ua %.2e loss %.2e dL/dtheta %.2e" % ((fix,) + errs))
    assert max(errs) < 1e-8, errs


def test_gradient_matches_finite_differences_of_the_solve():
    """dL/dtheta (mode 2) = central differences of the end-to-end loss, re-solved at tol 1e-12."""
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    oc.tol = 1e-12
    x0, th, taus, wp = fx["x0"][:1], fx["theta"][0], fx["taus"][:1], fx["wp"][:1]

    def run(t, mode=DISC):
        sol = oc.cocSolverBatch(x0, 1.0, t)
        assert int(sol["status"][0]) == 1
        return oc.auxSysSolverBatch(sol, taus, wp, [0], mode=mode)

    aux = run(th)
    g = aux["dtheta"][0].copy()
    fd = np.zeros_like(g)
    for i in range(len(th)):
        h = 1e-5 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += h
        tm[i] -= h
        fd[i] = (run(tp)["loss"][0] - run(tm)["loss"][0]) / (2 * h)
    fd *= 0.5                                   # reference convention: dl_dy = y - wp, half the derivative of the loss
    err = np.abs(g - fd).max() / np.abs(g).max()
    gap = np.abs(run(th, mode=oc.MODE_BDF)["dtheta"][0] - g).max() / np.abs(g).max()
    print("finite differences vs mode 2: %.2e (max-norm relative); mode 1 vs mode 2 (information only): %.2e" % (err, gap))
    assert err < 1e-6


def test_loss_bitwise_equal_to_mode0_and_rows_independent_of_batching():
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    sol = oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"])
    st = np.asarray(sol["status"])
    assert (st == 1).all()
    a2 = oc.auxSysSolverBatch(sol, fx["taus"], fx["wp"], [0], mode=DISC)
    a0 = oc.auxSysSolverBatch(sol, fx["taus"], fx["wp"], [0], mode=oc.MODE_RK45)
    assert np.array_equal(a2["loss"], a0["loss"])
    for b in range(3):
        one = host_sol(oc, 1.0, fx["theta"][b], sol["X"][b:b + 1], sol["U"][b:b + 1], sol["Lam"][b:b + 1], status=st[b:b + 1])
        a1 = oc.auxSysSolverBatch(one, fx["taus"][b:b + 1], fx["wp"][b:b + 1], [0], mode=DISC)
        for k in ("Xa", "Ua", "loss", "dtheta", "aux_status"):
            assert np.array_equal(a1[k][0], a2[k][b]), (k, b)


def test_status_cases():
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    X, U, Lam, th = fx["X"][:1], fx["U"][:1], fx["Lam"][:1], fx["theta"][0]
    # solve NUMERIC / RUNNING: skipped, zero row
    for s in (4, 0):
        aux = oc.auxSysSolverBatch(host_sol(oc, 1.0, th, X, U, Lam, status=[s]), fx["taus"][:1], fx["wp"][:1], [0], mode=DISC)
        assert int(aux["aux_status"][0]) == 3 and aux["loss"][0] == 0.0 and not aux["dtheta"][0].any()
    # MAXITER / LINESEARCH exits are processed
    for s in (2, 3):
        aux = oc.auxSysSolverBatch(host_sol(oc, 1.0, th, X, U, Lam, status=[s]), fx["taus"][:1], fx["wp"][:1], [0], mode=DISC)
        assert int(aux["aux_status"][0]) == 0
    # a waypoint time outside [0, T]
    aux = oc.auxSysSolverBatch(host_sol(oc, 1.0, th, X, U, Lam), np.array([[0.5, 1.5]]), np.zeros((1, 2, 1)), [0], mode=DISC)
    assert int(aux["aux_status"][0]) == 5 and aux["loss"][0] == 0.0 and not aux["dtheta"][0].any()
    # negative state weights make the final cost concave: Quu = Huu + B' hxx B is not positive definite on the last interval
    bad = np.array([1.0, -50.0, -50.0])
    aux = oc.auxSysSolverBatch(host_sol(oc, 1.0, bad, X, U, Lam), fx["taus"][:1], fx["wp"][:1], [0], mode=DISC)
    assert int(aux["aux_status"][0]) == 4 and aux["loss"][0] == 0.0 and not aux["dtheta"][0].any()
    # other mode values stay an argument error
    from lfsd_b200 import _capi
    with pytest.raises(_capi.CpdpError):
        oc.auxSysSolverBatch(host_sol(oc, 1.0, th, X, U, Lam), fx["taus"][:1], fx["wp"][:1], [0], mode=3)


def test_reference_shaped_aux_sys_solver():
    """auxSysSolver (X, U, Lam from the host) with aux_mode = MODE_DISCRETE: the node table of dx/dtheta | du/dtheta."""
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    th = fx["theta"][0]
    tg, opt_sol = oc.cocSolver(list(fx["x0"][0]), 1.0, th)
    oc.aux_mode = oc.MODE_DISCRETE
    got = oc.auxSysSolver(tg, opt_sol, th)(tg)
    assert oc.last_aux_status == 0
    nodes = opt_sol(tg)
    Xa, Ua = DiscreteOracle(models.pendulum(), n_grid=10).aux_discrete(tg, nodes[:, :2], nodes[:, 2:3], nodes[:, 3:], th)
    assert _rel(got[:, :6], Xa) < 1e-8 and _rel(got[:, 6:], Ua) < 1e-8


@pytest.mark.parametrize("model", ["pendulum", "quadrotor"])
def test_discrete_kernels_are_race_free(model):
    """ThreadSanitizer over the emulated kernels of mode 2 (the stage kernels, k_stage_theta, both phases of k_aux_discrete)."""
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "tsan_discrete_run.py"), model], capture_output=True,
                       text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("%s discrete" % model) == 1, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
