"""Adjoint of mode 2 with respect to the per-problem constants (cpdp_aux_adjoint_pd, COCSys.auxSysAdjointBatch(pdata_bar=True),
cpdp_layer(pdata_grad=True)).  CPU tests: the kernels run in the thread emulation of tests/emu/, built with the pdata companion header
(tests/emu/pd_support.py), through the same C ABI and host classes as on the GPU.  pdata_bar is checked against the dense implicit
differentiation of tests/pdata_oracle.py and against finite differences of the re-solved trajectory."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from lfsd_b200 import codegen, standard
from lfsd_b200.autograd import cpdp_layer
from tests.adjoint_oracle import contract
from tests.emu.build_emu import CSRC
from tests.emu.pd_support import emu_pd_from, pendulum_goal_model, pendulum_goal_oc
from tests.emu.support import emu_oc, _BUILD
from tests.pdata_oracle import BoundedPdataOracle, PdataOracle
from tests.test_adjoint import TorchCpuMem
from tests.test_bounds import CASES as BCASES
from tests.test_discrete_grad import _fx, _rel, host_sol
from oracle import models

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOALS = np.array([[2.6], [3.3], [2.9]])
X0 = np.array([[0.0, 0.0], [0.3, -0.2], [-0.1, 0.4]])
TH = {False: np.array([1.0, 1.0, 0.1]), True: np.array([1.0, 0.3, 1.0, 0.1])}


def _cot(rng, B, N, n, m):
    return rng.normal(size=(B, N + 1, n)), rng.normal(size=(B, N + 1, m))


def _goal_oc(tv=False, through=False, **kw):
    oc = pendulum_goal_oc(time_varying=tv, through_theta=through, **kw)
    return emu_pd_from(oc, "pgoal%s%s" % ("_tv" if tv else "", "_th" if through else ""))


# ------------------------------------------------------------------------------------------------ code generation
_PROBE = r"""
#include "cpdp_port.h"
#include MODEL
extern "C" __attribute__((visibility("default"))) void probe(const double* x, const double* u, const double* th, const double* pd,
        const double* mu, double w, const double* dx, const double* du, const double* dpd, double* df, double* hz, double* hxp) {
    ModelPd::dir_pd(x, u, th, pd, mu, w, dx, du, dpd, df, hz);
    ModelPd::term2_pd(x, th, pd, hxp);
}
"""


def _model(name):
    if name == "pendulum_goal_tv":
        return pendulum_goal_oc(time_varying=True)
    return (standard.VARIANTS.get(name) or standard.BOUNDED.get(name) or standard.STANDARD[name])()


@pytest.mark.parametrize("name", ["quadrotor", "quadrotor_cost1", "quadrotor_cost2", "quadrotor_bounded", "pendulum_goal_tv"])
def test_dir_pd_and_term2_pd_match_sympy(name):
    """ModelPd::dir_pd and term2_pd of the generated C (g++) = fz dz + f_pd dpd, Hzz dz + Hz,pd dpd and d(grad_x h)/dpd from sympy,
    with the time of a time-varying model held fixed (not a pdata column)."""
    import sympy as sp
    oc = _model(name)
    tv = getattr(oc, "time", None)
    text, info = codegen.generate_pdata_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost,
                                               oc.pvar, time=tv)
    assert info["nq"] == oc.n_pvar and info["ops_dir_pd"] > 0
    os.makedirs(_BUILD, exist_ok=True)
    hdr = os.path.join(_BUILD, "dirpd_%s_%s.cuh" % (name, info["hash"]))
    so = hdr[:-4] + ".so"
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        with open(hdr[:-4] + ".cpp", "w") as f:
            f.write(_PROBE)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", CSRC, '-DMODEL="%s"' % hdr, hdr[:-4] + ".cpp",
                               "-o", so])
    L = ctypes.CDLL(so)
    x, u, th = codegen._vec(oc.state), codegen._vec(oc.control), codegen._vec(oc.auxvar)
    pq = codegen._vec(oc.pvar)
    pdv = pq + (codegen._vec(tv) if tv is not None else [])
    n, m, r, q = len(x), len(u), len(th), len(pq)
    f, c, h = sp.Matrix(codegen._vec(oc.dyn)), codegen._to_matrix(oc.path_cost)[0, 0], codegen._to_matrix(oc.final_cost)[0, 0]
    z = x + u
    rng = np.random.default_rng(7)
    P = lambda k: rng.uniform(0.3, 1.2, size=k)
    xv, uv, tv_, pv, mu, dx, du, dpd = P(n), P(m), P(r), P(len(pdv)), rng.normal(size=n), rng.normal(size=n), rng.normal(size=m), \
        rng.normal(size=q)
    w = 0.37
    sub = dict(zip(x + u + th + pdv, list(xv) + list(uv) + list(tv_) + list(pv)))
    Ham = w * c + sum(mu[i] * f[i] for i in range(n))
    Hz = sp.Matrix([Ham]).jacobian(z)
    num = lambda M: np.array(M.subs(sub).evalf(), dtype=float)
    dz = np.concatenate([dx, du])
    df_ref = num(f.jacobian(z)) @ dz + num(f.jacobian(pq)) @ dpd
    hz_ref = num(Hz.jacobian(z)) @ dz + num(Hz.T.jacobian(pq)) @ dpd
    hxp_ref = num(sp.Matrix([h]).jacobian(x).jacobian(pq)).ravel()
    D = ctypes.POINTER(ctypes.c_double)
    a = lambda v: np.ascontiguousarray(v, dtype=float)
    args = [a(xv), a(uv), a(tv_), a(pv), a(mu)]
    df, hz, hxp = np.zeros(n), np.zeros(n + m), np.zeros(n * q)
    L.probe(*[v.ctypes.data_as(D) for v in args], ctypes.c_double(w), a(dx).ctypes.data_as(D), a(du).ctypes.data_as(D),
            a(dpd).ctypes.data_as(D), df.ctypes.data_as(D), hz.ctypes.data_as(D), hxp.ctypes.data_as(D))
    e = max(_rel(df, df_ref), _rel(hz, hz_ref), _rel(hxp, hxp_ref, floor=1.0))
    print("%s: dir_pd / term2_pd vs sympy %.2e" % (name, e))
    assert e <= 1e-12


def test_companion_header_of_a_model_without_constants_is_trivial():
    oc = standard.pendulum_oc()
    text, info = codegen.generate_pdata_header("pendulum", oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost,
                                               oc.pvar)
    assert info["nq"] == 0 and "static constexpr int NQ = 0;" in text and "dir_pd" not in text


# ------------------------------------------------------------------------------------------------ against the oracle
def test_quadrotor_pdata_bar_vs_oracle_and_unchanged_theta_bar():
    """quadrotor at the N = 25 fixture: pdata_bar against the dense oracle; theta_bar and x0_bar bit-identical to
    cpdp_aux_adjoint's."""
    fx = _fx("quadkat")
    N = int(fx["n_grid"])
    oc = emu_pd_from(standard.quadrotor_oc(n_grid=N), "quadrotor")
    pd = fx["pdata"][:1]
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    Xbar, Ubar = _cot(np.random.default_rng(3), 1, N, 13, 4)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    ref = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    assert int(adj["aux_status"][0]) == 0
    assert np.array_equal(adj["theta_bar"], ref["theta_bar"]) and np.array_equal(adj["x0_bar"], ref["x0_bar"])
    orc = PdataOracle(models.quadrotor(), n_grid=N)
    orc.pd = pd[0]
    DX, DU = orc.dpd_discrete(oc._time_grid(T, N), X, U, Lam, th)
    e = _rel(adj["pdata_bar"][0], contract(DX, DU, Xbar[0], Ubar[0]))
    print("quadrotor: pdata_bar vs dense oracle %.2e" % e)
    assert e <= 1e-9


def test_bounded_quadrotor_pdata_bar_vs_oracle():
    """Thrust-bounded quadrotor (1 <= f_i <= 4, active at the fixture's start): pdata_bar against the barrier-perturbed KKT oracle at
    the kernels' own solution (X, U, Lam, Zl, Zu)."""
    _, fix, mk, sel, bnd, _ = BCASES["quadrotor"]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = emu_pd_from(standard.quadrotor_bounded_oc(n_grid=N), "quadrotor_bounded")
    pd = fx["pdata"][:1]
    T = float(fx["T"])
    sol = oc.cocSolverBatch(fx["x0"][:1], T, fx["theta"][:1], pdata=pd)
    assert int(sol["status"][0]) == 1
    U = sol["U"][0]
    assert np.isclose(U[:N], 1.0, atol=1e-3).any() or np.isclose(U[:N], 4.0, atol=1e-3).any(), "no thrust bound active"
    Xbar, Ubar = _cot(np.random.default_rng(4), 1, N, 13, 4)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    assert int(adj["aux_status"][0]) == 0
    orc = BoundedPdataOracle(mk(), *bnd, n_grid=N)
    orc.pd = pd[0]
    DX, DU = orc.dpd_discrete_bounded(oc._time_grid(T, N), sol["X"][0], U, sol["Lam"][0], sol["Zl"][0], sol["Zu"][0],
                                      fx["theta"][0])
    e = _rel(adj["pdata_bar"][0], contract(DX, DU, Xbar[0], Ubar[0]))
    print("bounded quadrotor: pdata_bar vs dense oracle %.2e" % e)
    assert e <= 1e-8


@pytest.mark.parametrize("tv", [False, True])
def test_pendulum_goal_pdata_bar_vs_oracle(tv):
    """A pendulum whose goal angle is the constant, plain and time-varying (the time rides behind pdata and is no column)."""
    oc = _goal_oc(tv)
    sol = oc.cocSolverBatch(X0, 1.0, TH[tv], pdata=GOALS)
    assert (sol["status"] == 1).all()
    Xbar, Ubar = _cot(np.random.default_rng(5), 3, oc.n_grid, 2, 1)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    assert adj["pdata_bar"].shape == (3, 1) and (adj["aux_status"] == 0).all()
    orc = PdataOracle(pendulum_goal_model(tv), n_grid=oc.n_grid)
    e = 0.0
    for b in range(3):
        orc.pd = GOALS[b]
        DX, DU = orc.dpd_discrete(oc._time_grid(1.0, oc.n_grid), sol["X"][b], sol["U"][b], sol["Lam"][b], TH[tv])
        e = max(e, _rel(adj["pdata_bar"][b], contract(DX, DU, Xbar[b], Ubar[b])))
    print("pendulum goal (time-varying %s): pdata_bar vs dense oracle %.2e" % (tv, e))
    assert e <= 1e-9


def test_pdata_bar_matches_finite_differences_of_the_solve():
    """pdata_bar = central differences of l(pd) = sum Xbar.X + Ubar.U over the trajectory re-solved at tol 1e-12."""
    oc = _goal_oc()
    oc.tol = 1e-12
    Xbar, Ubar = _cot(np.random.default_rng(6), 1, oc.n_grid, 2, 1)

    def ell(g):
        s = oc.cocSolverBatch(X0[:1], 1.0, TH[False], pdata=g)
        assert int(s["status"][0]) == 1
        return float((s["X"] * Xbar).sum() + (s["U"] * Ubar).sum())
    sol = oc.cocSolverBatch(X0[:1], 1.0, TH[False], pdata=GOALS[:1])
    g = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)["pdata_bar"][0, 0]
    h = 1e-5
    fd = (ell(GOALS[:1] + h) - ell(GOALS[:1] - h)) / (2 * h)
    err = abs(g - fd) / abs(g)
    print("pdata_bar vs finite differences: %.2e" % err)
    assert err <= 1e-6


def test_pdata_entering_through_theta_plus_pdata_has_theta_bar():
    """A model whose constant g enters only through theta_4 + g: pdata_bar = theta_bar_4 to rounding."""
    oc = _goal_oc(through=True)
    th = np.array([1.0, 1.0, 0.1, 2.0])
    sol = oc.cocSolverBatch(X0, 1.0, th, pdata=GOALS - 2.0)
    assert (sol["status"] == 1).all()
    Xbar, Ubar = _cot(np.random.default_rng(8), 3, oc.n_grid, 2, 1)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    e = _rel(adj["pdata_bar"][:, 0], adj["theta_bar"][:, 3])
    print("pdata_bar vs theta_bar of theta + pdata: %.2e" % e)
    assert e <= 1e-13


# ------------------------------------------------------------------------------------------------ rows, errors
def test_status_rows_rebatching_and_errors():
    oc = _goal_oc()
    N = oc.n_grid
    sol = oc.cocSolverBatch(X0, 1.0, TH[False], pdata=GOALS)
    Xbar, Ubar = _cot(np.random.default_rng(1), 3, N, 2, 1)
    full = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    for b in range(3):
        one = host_sol(oc, 1.0, TH[False], sol["X"][b:b + 1], sol["U"][b:b + 1], sol["Lam"][b:b + 1], GOALS[b:b + 1], status=[1])
        a1 = oc.auxSysAdjointBatch(one, Xbar[b:b + 1], Ubar[b:b + 1], pdata_bar=True)
        for k in ("pdata_bar", "theta_bar", "x0_bar", "aux_status"):
            assert np.array_equal(a1[k][0], full[k][b]), (k, b)
    # converged / solve NUMERIC (aux 3) / MAXITER (aux 0, not converged) / Quu not positive definite (aux 4)
    th = np.vstack([TH[False]] * 3 + [[1.0, -50.0, -50.0]])
    idx = [0, 0, 0, 0]
    bad = host_sol(oc, 1.0, th, sol["X"][idx], sol["U"][idx], sol["Lam"][idx], GOALS[idx], status=[1, 4, 2, 1])
    Xb, Ub = _cot(np.random.default_rng(2), 4, N, 2, 1)
    adj = oc.auxSysAdjointBatch(bad, Xb, Ub, pdata_bar=True)
    assert list(adj["aux_status"]) == [0, 3, 0, 4]
    assert np.abs(adj["pdata_bar"][0]).max() > 0 and not adj["pdata_bar"][1:].any() and not adj["theta_bar"][1:].any()
    # argument errors
    with pytest.raises(ValueError):
        emu_oc("pendulum").auxSysAdjointBatch(host_sol(emu_oc("pendulum"), 1.0, [1, 1, .1], sol["X"], sol["U"], sol["Lam"]),
                                              Xbar, Ubar, pdata_bar=True)
    mem, p = oc._device(), oc._device().ptr
    ws, pws = oc._workspace(3), oc._pdata_workspace(3)
    out, o0, opd = np.zeros((3, 3)), np.zeros((3, 2)), np.zeros((3, 1))
    st = np.zeros(3, dtype=np.int32)

    def call(lib, pws_bytes, pdp=p(sol["pdata"])):
        return lib.L.cpdp_aux_adjoint_pd(p(ws), int(ws.shape[0]), p(pws), pws_bytes, 3, N, 4, 1.0, p(sol["theta"]), 0, pdp,
                                         p(sol["X"]), p(sol["U"]), p(sol["Lam"]), p(sol["status"]), p(Xbar), p(Ubar), p(out),
                                         p(o0), p(opd), p(st), None)
    assert oc._lib.pdata_workspace_bytes(3, N) == int(pws.shape[0]) > 0
    assert call(oc._lib, int(pws.shape[0])) == 0
    assert call(oc._lib, int(pws.shape[0]) - 1) == -3
    assert call(oc._lib, int(pws.shape[0]), pdp=None) == -8
    assert call(emu_oc("pendulum")._lib, int(pws.shape[0])) == -14
    assert emu_oc("pendulum")._lib.pdata_workspace_bytes(3, N) == 0
    plain = emu_oc("quadrotor", n_grid=4)                          # the emulation built without the companion header
    assert call(plain._lib, int(pws.shape[0])) == -15


# ------------------------------------------------------------------------------------------------ the autograd layer
def test_layer_gradcheck_with_pdata():
    """gradcheck of cpdp_layer(pdata_grad=True) with respect to pdata, x0 and theta together (pendulum goal, float64)."""
    oc = _goal_oc()
    oc._mem = TorchCpuMem()
    oc.tol = 1e-12
    g = torch.Generator().manual_seed(0)
    P = torch.randn(3, 2, 11, 2, generator=g, dtype=torch.float64)
    Q = torch.randn(3, 2, 11, 1, generator=g, dtype=torch.float64)

    def f(x0, th, pd):
        X, U, info = cpdp_layer(oc, x0, th, 1.0, pdata=pd, pdata_grad=True)
        assert (info["status"] == 1).all()
        return torch.einsum("pbki,bki->p", P, X) + torch.einsum("pbkj,bkj->p", Q, U)
    x0 = torch.tensor(X0[:2], dtype=torch.float64, requires_grad=True)
    th = torch.tensor(TH[False], dtype=torch.float64, requires_grad=True)
    pd = torch.tensor(GOALS[:2], dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(f, (x0, th, pd), eps=1e-6, atol=1e-6, rtol=1e-4)
    with pytest.raises(NotImplementedError):
        cpdp_layer(oc, x0, th, 1.0, pdata=pd)
    with pytest.raises(ValueError):
        cpdp_layer(oc, x0, th, 1.0, pdata=None, pdata_grad=True)


# ------------------------------------------------------------------------------------------------ races
def test_pdata_kernels_are_race_free():
    """ThreadSanitizer over the emulated k_stage_theta_pd, k_aux_discrete_pd and k_aux_adjoint_pd (quadrotor, N = 4)."""
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from tests.emu.pd_support import emu_pd_from\n"
            "from lfsd_b200 import standard, synthetic\n"
            "oc = emu_pd_from(standard.quadrotor_oc(n_grid=4), 'quadrotor', tsan=True)\n"
            "qb = synthetic.quad_batch(1)\n"
            "sol = oc.cocSolverBatch(qb['x0'], 1.0, qb['theta'], pdata=qb['goal'])\n"
            "rng = np.random.default_rng(0)\n"
            "adj = oc.auxSysAdjointBatch(sol, rng.normal(size=sol['X'].shape), rng.normal(size=sol['U'].shape), pdata_bar=True)\n"
            "print('pdata adjoint run', adj['aux_status'], adj['pdata_bar'][0])\n") % ROOT
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("pdata adjoint run [0]") == 1, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
