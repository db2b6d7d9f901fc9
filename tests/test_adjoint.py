"""Adjoint of mode 2 (cpdp_aux_adjoint, COCSys.auxSysAdjointBatch) and the torch.autograd layer over the batched solve
(lfsd_b200.autograd.cpdp_layer).  CPU tests: the kernels run in the thread emulation of tests/emu/ through the same C ABI and host
classes as on the GPU.  theta_bar is checked against mode 2's forward-mode columns of the same library, x0_bar against the dense
implicit differentiation of tests/adjoint_oracle.py and against finite differences of the re-solved trajectory."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from lfsd_b200.autograd import cpdp_layer
from tests.adjoint_oracle import AdjointOracle, BoundedAdjointOracle, contract
from tests.emu.support import emu_oc
from tests.test_bounds import CASES as BCASES, _solved
from tests.test_discrete_grad import CASES, host_sol, _fx, _rel

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DISC = 2


def forward_mode(aux, Xbar, Ubar, n, m, r):
    """theta_bar from mode 2's columns: sum_k Xa_k' Xbar_k + Ua_k' Ubar_k, rows [B, r]."""
    B, N1 = Xbar.shape[:2]
    Xa = np.asarray(aux["Xa"]).reshape(B, N1, n, r)
    Ua = np.asarray(aux["Ua"]).reshape(B, N1, m, r)
    return np.einsum("bkir,bki->br", Xa, Xbar) + np.einsum("bkjr,bkj->br", Ua, Ubar)


def _cot(rng, B, N, n, m):
    return rng.normal(size=(B, N + 1, n)), rng.normal(size=(B, N + 1, m))


# ------------------------------------------------------------------------------------------------ unbounded models
@pytest.mark.parametrize("fix", list(CASES))
def test_adjoint_vs_forward_mode_and_oracle(fix):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = emu_oc(name, n_grid=N)
    n, m, r = oc.n_state, oc.n_control, oc.n_auxvar
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    Xbar, Ubar = _cot(np.random.default_rng(3), 1, N, n, m)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:1], fx["wp"][:1], sel, mode=DISC)
    assert int(adj["aux_status"][0]) == 0 and int(aux["aux_status"][0]) == 0
    e_th = _rel(adj["theta_bar"], forward_mode(aux, Xbar, Ubar, n, m, r))
    orc = AdjointOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    DX, DU = orc.dx0_discrete(oc._time_grid(T, N), X, U, Lam, th)
    e_x0 = _rel(adj["x0_bar"][0], contract(DX, DU, Xbar[0], Ubar[0]))
    print("%s: theta_bar vs forward mode %.2e, x0_bar vs dense oracle %.2e" % (fix, e_th, e_x0))
    assert e_th <= 1e-12
    assert e_x0 <= 1e-10


def test_x0_bar_matches_finite_differences_of_the_solve():
    """x0_bar = central differences of l(x0) = sum Xbar.X + Ubar.U over the trajectory re-solved at tol 1e-12 (pendulum)."""
    oc = emu_oc("pendulum")
    oc.tol = 1e-12
    fx = _fx("pendulum")
    x0, th = fx["x0"][:1].copy(), fx["theta"][0]
    Xbar, Ubar = _cot(np.random.default_rng(5), 1, oc.n_grid, 2, 1)

    def ell(x):
        s = oc.cocSolverBatch(x, 1.0, th)
        assert int(s["status"][0]) == 1
        return float((s["X"] * Xbar).sum() + (s["U"] * Ubar).sum())
    sol = oc.cocSolverBatch(x0, 1.0, th)
    g = oc.auxSysAdjointBatch(sol, Xbar, Ubar)["x0_bar"][0]
    fd = np.zeros(2)
    for i in range(2):
        h = 1e-5
        xp, xm = x0.copy(), x0.copy()
        xp[0, i] += h
        xm[0, i] -= h
        fd[i] = (ell(xp) - ell(xm)) / (2 * h)
    err = np.abs(g - fd).max() / np.abs(g).max()
    print("x0_bar vs finite differences: %.2e" % err)
    assert err <= 1e-6


def test_cotangent_on_last_control_folds_onto_the_one_before():
    """U_N = U_{N-1}: a cotangent on U_N alone gives the same bits as the same cotangent on U_{N-1}."""
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    sol = host_sol(oc, 1.0, fx["theta"][0], fx["X"][:1], fx["U"][:1], fx["Lam"][:1])
    N = oc.n_grid
    c = np.random.default_rng(9).normal(size=1)
    Ua, Ub = np.zeros((1, N + 1, 1)), np.zeros((1, N + 1, 1))
    Ua[0, N], Ub[0, N - 1] = c, c
    a, b = oc.auxSysAdjointBatch(sol, Ubar=Ua), oc.auxSysAdjointBatch(sol, Ubar=Ub)
    assert np.array_equal(a["theta_bar"], b["theta_bar"]) and np.array_equal(a["x0_bar"], b["x0_bar"])
    assert np.abs(a["theta_bar"]).max() > 0


def test_status_rows_and_rebatching():
    oc = emu_oc("pendulum")
    fx = _fx("pendulum")
    N = oc.n_grid
    # converged / solve NUMERIC (aux 3) / MAXITER (aux 0, not converged) / Quu not positive definite (aux 4)
    th = np.vstack([fx["theta"][0], fx["theta"][0], fx["theta"][0], [1.0, -50.0, -50.0]])
    idx = [0, 0, 0, 0]
    sol = host_sol(oc, 1.0, th, fx["X"][idx], fx["U"][idx], fx["Lam"][idx], status=[1, 4, 2, 1])
    Xbar, Ubar = _cot(np.random.default_rng(1), 4, N, 2, 1)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    assert list(adj["aux_status"]) == [0, 3, 0, 4]
    assert np.abs(adj["theta_bar"][0]).max() > 0 and np.abs(adj["x0_bar"][0]).max() > 0
    assert not adj["theta_bar"][1:].any() and not adj["x0_bar"][1:].any()
    # rows do not depend on the batch around them
    sol = oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"])
    assert (sol["status"] == 1).all()
    Xbar, Ubar = _cot(np.random.default_rng(2), 3, N, 2, 1)
    full = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    for b in range(3):
        one = host_sol(oc, 1.0, fx["theta"][b], sol["X"][b:b + 1], sol["U"][b:b + 1], sol["Lam"][b:b + 1], status=[1])
        a1 = oc.auxSysAdjointBatch(one, Xbar[b:b + 1], Ubar[b:b + 1])
        for k in ("theta_bar", "x0_bar", "aux_status"):
            assert np.array_equal(a1[k][0], full[k][b]), (k, b)
    # argument errors: no cotangent, no theta_bar
    with pytest.raises(ValueError):
        oc.auxSysAdjointBatch(sol)
    mem, ws = oc._device(), oc._workspace(3)
    L, p = oc._lib.L, mem.ptr
    out = np.zeros((3, 3))
    args = [p(ws), int(ws.shape[0]), 3, N, 4, 1.0, p(sol["theta"]), sol["theta_stride"], None, p(sol["X"]), p(sol["U"]),
            p(sol["Lam"]), p(sol["status"])]
    st = np.zeros(3, dtype=np.int32)
    assert L.cpdp_aux_adjoint(*args, None, None, p(out), None, p(st), None) == -1
    assert L.cpdp_aux_adjoint(*args, p(Xbar), None, None, None, p(st), None) == -1
    assert L.cpdp_aux_adjoint(*(args[:7] + [1] + args[8:]), p(Xbar), None, p(out), None, p(st), None) == -2
    assert L.cpdp_aux_adjoint(*(args[:1] + [16] + args[2:]), p(Xbar), None, p(out), None, p(st), None) == -3


# ------------------------------------------------------------------------------------------------ bounded models
# x0_bar against the dense perturbed-KKT oracle.  The active STATE bound of the robot arm puts Sigma ~ 1e12 into the Riccati value
# function, whose recursion keeps ~ 1e-16 * Sigma relative accuracy (DESIGN.md §3.8); the adjoint reads that recursion's gains.
X0_TOL = {"pendulum": 1e-10, "quadrotor": 1e-10, "robotarm": 1e-5}


@pytest.mark.parametrize("key", ["pendulum", "robotarm", "quadrotor"])
def test_bounded_adjoint_vs_forward_mode_and_oracle(key):
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved(key)
    n, m, r, N = oc.n_state, oc.n_control, oc.n_auxvar, oc.n_grid
    Xbar, Ubar = _cot(np.random.default_rng(11), nb, N, n, m)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=DISC)
    assert (adj["aux_status"] == 0).all()
    e_th = _rel(adj["theta_bar"], forward_mode(aux, Xbar, Ubar, n, m, r))
    ao = BoundedAdjointOracle(BCASES[key][2](), *bnd, n_grid=N)
    e_x0 = 0.0
    for b in range(nb):
        R = ref[b]
        if pd is not None:
            ao.pd = pd[b]
        DX, DU = ao.dx0_discrete_bounded(R["time_grid"], R["X"], R["U"], R["Lam"], R["Zl"], R["Zu"], fx["theta"][b])
        e_x0 = max(e_x0, _rel(adj["x0_bar"][b], contract(DX, DU, Xbar[b], Ubar[b])))
    print("bounded %s: theta_bar vs forward mode %.2e, x0_bar vs dense oracle %.2e" % (key, e_th, e_x0))
    assert e_th <= 1e-12
    assert e_x0 <= X0_TOL[key]


# ------------------------------------------------------------------------------------------------ the autograd layer
class TorchCpuMem:
    """Memory provider of COCSys on torch CPU tensors, so that the emulated library serves cpdp_layer."""

    _dt = {"f8": torch.float64, "i4": torch.int32, "u1": torch.uint8}

    def empty(self, shape, dtype="f8"):
        return torch.zeros(shape, dtype=self._dt[dtype])

    zeros = empty

    def from_host(self, a, dtype="f8"):
        if isinstance(a, torch.Tensor):
            return a.to(dtype=self._dt[dtype]).contiguous()
        return torch.tensor(np.asarray(a), dtype=self._dt[dtype])

    def to_host(self, x):
        return x.detach().numpy()

    def ptr(self, x):
        return 0 if x is None else x.data_ptr()

    def stream(self):
        return 0


def _torch_oc(name, **kw):
    oc = emu_oc(name, **kw)
    oc._mem = TorchCpuMem()
    return oc


def test_layer_gradcheck():
    """torch.autograd.gradcheck of cpdp_layer (pendulum, N = 10, float64) with respect to x0 and theta, shared and per problem,
    through random linear functionals of (X, U) (three backward passes each instead of one per trajectory entry)."""
    oc = _torch_oc("pendulum")
    oc.tol = 1e-12
    fx = _fx("pendulum")
    g = torch.Generator().manual_seed(0)
    P = torch.randn(3, 2, 11, 2, generator=g, dtype=torch.float64)
    Q = torch.randn(3, 2, 11, 1, generator=g, dtype=torch.float64)

    def f(x0, th):
        X, U, info = cpdp_layer(oc, x0, th, 1.0)
        assert (info["status"] == 1).all()
        return torch.einsum("pbki,bki->p", P, X) + torch.einsum("pbkj,bkj->p", Q, U)
    x0 = torch.tensor(fx["x0"][:2], dtype=torch.float64, requires_grad=True)
    for th in (torch.tensor(fx["theta"][0], dtype=torch.float64), torch.tensor(fx["theta"][:2], dtype=torch.float64)):
        th.requires_grad_(True)
        assert torch.autograd.gradcheck(f, (x0, th), eps=1e-6, atol=1e-6, rtol=1e-4)


def _interp_loss(X, taus, wp, sel, T):
    """0.5 sum ||y(tau) - wp||^2 with y the linear interpolant of the nodes X (scipy's interp1d index rule), in torch."""
    N = X.shape[1] - 1
    dt = T / N
    loss = X.new_zeros(())
    for b in range(X.shape[0]):
        for w, t in enumerate(taus[b]):
            lo = min(max(int(np.searchsorted(dt * np.arange(N + 1), t, "left")), 1), N) - 1
            y = X[b, lo, sel] + (X[b, lo + 1, sel] - X[b, lo, sel]) / dt * (t - dt * lo)
            loss = loss + 0.5 * ((y - X.new_tensor(wp[b, w])) ** 2).sum()
    return loss


def test_layer_waypoint_loss_matches_mode2():
    """A waypoint loss written in torch back-propagates to exactly mode 2's dtheta (the reference's dl_dy = y - wp convention is
    the gradient of 0.5 ||y - wp||^2): per-problem theta row by row, a shared theta to their sum; aux_status is filled in."""
    oc = _torch_oc("pendulum")
    fx = _fx("pendulum")
    aux = oc.auxSysSolverBatch(oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"]), fx["taus"], fx["wp"], [0], mode=DISC)
    th = torch.tensor(fx["theta"], dtype=torch.float64, requires_grad=True)
    X, U, info = cpdp_layer(oc, torch.tensor(fx["x0"]), th, 1.0)
    _interp_loss(X, fx["taus"], fx["wp"], [0], 1.0).backward()
    assert (info["aux_status"] == 0).all()
    e = _rel(th.grad.numpy(), aux["dtheta"].numpy())
    ths = torch.tensor(fx["theta"][0], dtype=torch.float64, requires_grad=True)
    sol = oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"][0])
    ref = oc.auxSysSolverBatch(sol, fx["taus"], fx["wp"], [0], mode=DISC)["dtheta"].numpy().sum(0)
    X, U, info = cpdp_layer(oc, torch.tensor(fx["x0"]), ths, 1.0)
    _interp_loss(X, fx["taus"], fx["wp"], [0], 1.0).backward()
    es = _rel(ths.grad.numpy(), ref)
    print("waypoint loss through the layer vs mode 2: per problem %.2e, shared %.2e" % (e, es))
    assert e <= 1e-12 and es <= 1e-12


def test_layer_rejects_differentiable_pdata():
    oc = _torch_oc("quadrotor", n_grid=4)
    from lfsd_b200 import synthetic
    qb = synthetic.quad_batch(1)
    with pytest.raises(NotImplementedError):
        cpdp_layer(oc, torch.tensor(qb["x0"]), torch.tensor(qb["theta"]), 1.0,
                   pdata=torch.tensor(qb["goal"], requires_grad=True))


# ------------------------------------------------------------------------------------------------ races
@pytest.mark.parametrize("model", ["pendulum", "quadrotor"])
def test_adjoint_kernel_is_race_free(model):
    """ThreadSanitizer over the emulated k_aux_adjoint (and the mode-2 phase 1 it runs first)."""
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from tests.emu.support import emu_oc\n"
            "from lfsd_b200 import synthetic\n"
            "oc = emu_oc(%r, tsan=True)\n"
            "if oc.n_state == 2:\n"
            "    sol = oc.cocSolverBatch(np.zeros((1, 2)), 1.0, np.array([1.0, 0.5, 1.5]))\n"
            "else:\n"
            "    qb = synthetic.quad_batch(1); oc.setIntegrator(n_grid=4)\n"
            "    sol = oc.cocSolverBatch(qb['x0'], 1.0, qb['theta'], pdata=qb['goal'])\n"
            "rng = np.random.default_rng(0)\n"
            "adj = oc.auxSysAdjointBatch(sol, rng.normal(size=sol['X'].shape), rng.normal(size=sol['U'].shape))\n"
            "print('adjoint run', adj['aux_status'], adj['theta_bar'][0])\n") % (ROOT, model)
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("adjoint run [0]") == 1, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
