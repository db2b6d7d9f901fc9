"""Box bounds on the states and controls: the barrier method of cpdp_solve and mode 2 through active bounds.  CPU tests: the
kernels run in the thread emulation of tests/emu/ through the same C ABI and COCSys host class as on the GPU, against the dense
barrier oracle of tests/bounded_oracle.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from lfsd_b200 import codegen, standard
from lfsd_b200.CPDP import COCSys
from tests.emu.support import emu_oc
from tests.emu.bounds_support import emu_bounded_oc, emu_from
from tests.bounded_oracle import BoundedOracle
from oracle.cpdp_oracle import Oracle, TIGHT
from oracle import models

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DISC = COCSys.MODE_DISCRETE
BIG = 1e20

# info["hash"] of the ten unbounded models' headers at the commit before bounds existed: their headers must not change
PARENT_HASHES = {"pendulum": "8060fa1dbf420866", "pendulum_tw2": "8b6c6ff18ab3310e", "robotarm": "3ef6a59ed973eded",
                 "rocket": "92262f39e2b65ed8", "quadrotor": "196c06251c2aa0e7", "cartpole": "d8a1960df124c1eb",
                 "robotarm_wd": "74bb0336cd353e80", "quadrotor_cost1": "444481be4fc5a54b",
                 "quadrotor_cost2": "900a79bf3cb6760a", "rocket_cost1": "081f3ca98c27ded5"}

# bounded model, fixture whose problems it solves, oracle model, observed states, (xlb, xub, ulb, uub), fixture problems used
# (those whose unbounded optimum leaves the box)
CASES = {
    "pendulum": ("pendulum_bounded", "pendulum", models.pendulum, [0],
                 ([-BIG] * 2, [BIG] * 2, [-5.0], [5.0]), [0, 1, 2]),
    "robotarm": ("robotarm_bounded", "robotarm", models.robotarm, [0, 1],
                 ([-BIG] * 3 + [-4.0], [BIG] * 3 + [4.0], [-3.0] * 2, [3.0] * 2), [2]),
    "quadrotor": ("quadrotor_bounded", "quadkat", models.quadrotor, [0, 1, 2],
                  ([-BIG] * 13, [BIG] * 13, [1.0] * 4, [4.0] * 4), [0]),
}


def _rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _fixture(fix, probs):
    """The fixture's arrays restricted to problems `probs` (per-problem arrays first), scalars as they are."""
    fx = np.load(os.path.join(HERE, "golden", "oracle_%s.npz" % fix))
    per = ("x0", "theta", "taus", "wp", "pdata", "X", "U", "Lam")
    return {k: (fx[k][probs] if k in per else fx[k]) for k in fx.files if k in per + ("n_grid", "T")}


def _case(key):
    name, fix, mk, sel, bnd, probs = CASES[key]
    fx = _fixture(fix, probs)
    nb = len(probs)
    N = int(fx["n_grid"])
    oc = emu_bounded_oc(name, n_grid=N)
    orc = BoundedOracle(mk(), *bnd, n_grid=N)
    pd = fx["pdata"] if "pdata" in fx else None
    return oc, orc, fx, pd, sel, bnd, nb


def _slacks(X, U, bnd):
    xlb, xub, ulb, uub = (np.asarray(v, dtype=float) for v in bnd)
    s = [X - xlb, xub - X, U - ulb, uub - U]
    fin = [np.abs(xlb) < 1e19, np.abs(xub) < 1e19, np.abs(ulb) < 1e19, np.abs(uub) < 1e19]
    return np.concatenate([si[..., f].ravel() for si, f in zip(s, fin)])


_SOLVED = {}


def _solved(key):
    """(emulated solve dict, [oracle result per problem]) of case `key`, cached over the module."""
    if key not in _SOLVED:
        oc, orc, fx, pd, sel, bnd, nb = _case(key)
        sol = oc.cocSolverBatch(fx["x0"][:nb], float(fx["T"]), fx["theta"][:nb], pdata=pd)
        ref = []
        for b in range(nb):
            if pd is not None:
                orc.pd = pd[b]
            ref.append(orc.solve_bounded(fx["x0"][b], float(fx["T"]), fx["theta"][b]))
        _SOLVED[key] = (oc, orc, fx, pd, sel, bnd, nb, sol, ref)
    return _SOLVED[key]


# ------------------------------------------------------------------------------------------------ code generation / host API
@pytest.mark.parametrize("name", sorted(PARENT_HASHES))
def test_unbounded_headers_unchanged(name):
    """A model without a finite bound generates the same header, byte for byte, as before bounds were supported."""
    oc = (standard.STANDARD.get(name) or standard.VARIANTS[name])()
    text, info = codegen.generate_model_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost,
                                               oc.pvar, time=getattr(oc, "time", None), bounds=oc._bounds())
    assert not oc.bounded and "HAS_BOUNDS" not in text
    assert info["hash"] == PARENT_HASHES[name]


def test_bounded_library_reports_its_bounds():
    oc = emu_bounded_oc("robotarm_bounded")
    assert oc.bounded and oc._lib.has_bounds
    assert oc._lib.lb == [-BIG, -BIG, -BIG, -4.0, -3.0, -3.0]
    assert oc._lib.ub == [BIG, BIG, BIG, 4.0, 3.0, 3.0]
    assert not emu_oc("pendulum")._lib.has_bounds


def test_setter_rejects_empty_boxes():
    oc = standard.pendulum_oc()
    with pytest.raises(ValueError):
        oc.setControlVariable(oc.env.U, [1.0], [1.0])          # fixed variable
    with pytest.raises(ValueError):
        oc.setControlVariable(oc.env.U, [2.0], [1.0])
    with pytest.raises(ValueError):
        oc.setStateVariable(oc.env.X, [0.0, float("nan")], [1.0, 1.0])
    oc.setControlVariable(oc.env.U, [-1.0], [float("inf")])    # one-sided, infinity = none
    assert oc.control_ub == [BIG] and oc.bounded


# ------------------------------------------------------------------------------------------------ the oracle itself
def test_oracle_matches_trust_constr():
    """The barrier oracle's optimum of the bounded pendulum = scipy's trust-constr on the same NLP (U within 1e-6); the bounds
    hold, the multipliers are non-negative and complementary."""
    from scipy.optimize import minimize, NonlinearConstraint, Bounds
    _, orc, fx, _, _, bnd, _, _, ref = _solved("pendulum")
    r = ref[0]
    x0, th, T = fx["x0"][0], fx["theta"][0], float(fx["T"])
    N, n = orc.N, orc.n
    DT = T / N / orc.S
    tg = np.array([T / N * k for k in range(N + 1)])
    zero = np.zeros((N + 1) * n)
    asm = lambda w, lam: orc._assemble(w, lam, th, x0, tg, DT)
    cons = NonlinearConstraint(lambda w: asm(w, zero)[1], 0.0, 0.0, jac=lambda w: asm(w, zero)[4],
                               hess=lambda w, v: asm(w, v)[3] - asm(w, zero)[3])
    res = minimize(lambda w: asm(w, zero)[0], orc.start(), jac=lambda w: asm(w, zero)[2], hess=lambda w: asm(w, zero)[3],
                   method="trust-constr", constraints=[cons], bounds=Bounds(orc.lb, orc.ub),
                   options=dict(gtol=1e-12, xtol=1e-14, barrier_tol=1e-12, maxiter=3000))
    nz = orc.n + orc.m
    Ut = np.concatenate([res.x, np.zeros(orc.m)]).reshape(N + 1, nz)[:N, n:]
    assert r["status"] == "converged"
    assert np.abs(Ut - r["U"][:N]).max() < 1e-6
    s = _slacks(r["X"], r["U"][:N], bnd)
    assert s.min() > 0 and s.min() < 1e-6                     # feasible, and the torque bound is active
    Zl, Zu = r["Zl"][:, n:][:N, 0], r["Zu"][:, n:][:N, 0]
    assert Zl.min() > 0 and Zu.min() > 0
    assert np.abs((r["U"][:N, 0] + 5.0) * Zl).max() < 1e-9 and np.abs((5.0 - r["U"][:N, 0]) * Zu).max() < 1e-9
    assert Zu.max() > 1e-3                                     # the active upper bound carries a multiplier


# ------------------------------------------------------------------------------------------------ kernels against the oracle
@pytest.mark.parametrize("key", ["pendulum", "robotarm", "quadrotor"])
def test_bounded_solve_matches_oracle(key):
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved(key)
    n = orc.n
    for b in range(nb):
        r = ref[b]
        assert r["status"] == "converged" and int(sol["status"][b]) == 1
        assert int(sol["iters"][b]) == r["iters"], (b, sol["iters"][b], r["iters"])
        for k in ("X", "U", "Lam", "Zl", "Zu"):
            assert _rel(sol[k][b], r[k]) < 1e-6, (k, b, _rel(sol[k][b], r[k]))
        s = _slacks(sol["X"][b], sol["U"][b][:-1], bnd)
        assert s.min() > 0.0
        assert s.min() < 1e-6, "no bound is active in case %s/%d" % (key, b)
        assert abs(float(sol["mu"][b]) - r["mu"]) <= 1e-15
        assert float(sol["kkt"][b]) < oc.tol
    assert n == oc.n_state


def test_every_iterate_is_strictly_inside():
    """Fixed round counts stop the solver after each iteration: every iterate lies strictly inside the box."""
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved("pendulum")
    T = float(fx["T"])
    for rounds in range(1, int(sol["iters"].max()) + 1):
        s = oc.cocSolverBatch(fx["x0"][:nb], T, fx["theta"][:nb], rounds=rounds)
        assert _slacks(s["X"], s["U"][:, :-1], bnd).min() > 0.0, rounds
        assert (s["Zl"][:, :-1, 2] > 0).all() and (s["Zu"][:, :-1, 2] > 0).all()


def test_inactive_bounds_reproduce_unbounded():
    """|u| <= 1e3 never binds: the barrier method returns the unbounded solution to 1e-8."""
    fx = np.load(os.path.join(HERE, "golden", "oracle_pendulum.npz"))
    T = float(fx["T"])
    ob = standard.pendulum_oc()
    ob.setControlVariable(ob.env.U, [-1e3], [1e3])
    ob = emu_from(ob, "pendulum_wide")
    sb = ob.cocSolverBatch(fx["x0"], T, fx["theta"])
    su = emu_oc("pendulum").cocSolverBatch(fx["x0"], T, fx["theta"])
    assert (sb["status"] == 1).all()
    for k in ("X", "U", "Lam"):
        assert _rel(sb[k], su[k]) < 1e-8, (k, _rel(sb[k], su[k]))


def test_rebatching_does_not_change_rows():
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved("pendulum")
    T = float(fx["T"])
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=DISC)
    for b in range(nb):
        s1 = oc.cocSolverBatch(fx["x0"][b:b + 1], T, fx["theta"][b:b + 1])
        a1 = oc.auxSysSolverBatch(s1, fx["taus"][b:b + 1], fx["wp"][b:b + 1], sel, mode=DISC)
        for k in ("X", "U", "Lam", "Zl", "Zu", "mu", "iters"):
            assert np.array_equal(s1[k][0], sol[k][b]), k
        for k in ("Xa", "Ua", "loss", "dtheta"):
            assert np.array_equal(a1[k][0], aux[k][b]), k


# ------------------------------------------------------------------------------------------------ mode 2 through active bounds
# Agreement of mode 2 with the dense perturbed-KKT oracle.  An active STATE bound puts Sigma ~ z/s ~ 1e12 on a diagonal entry of
# the Riccati value function, and V = Qxx + Qxu K then cancels terms of that size: the recursion keeps ~ 1e-16 * Sigma of relative
# accuracy (2e-6 measured on the robot arm), while control bounds only enter Quu (DESIGN.md §3.8).
MODE2_TOL = {"pendulum": 1e-10, "quadrotor": 1e-10, "robotarm": 1e-5}


@pytest.mark.parametrize("key", ["pendulum", "robotarm", "quadrotor"])
def test_mode2_matches_perturbed_kkt_oracle(key):
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved(key)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=DISC)
    assert (aux["aux_status"] == 0).all()
    m, r = orc.m, orc.r
    for b in range(nb):
        R = ref[b]
        if pd is not None:
            orc.pd = pd[b]
        Xa, Ua = orc.aux_discrete_bounded(R["time_grid"], R["X"], R["U"], R["Lam"], R["Zl"], R["Zu"], fx["theta"][b])
        errs = (_rel(aux["Xa"][b], Xa), _rel(aux["Ua"][b], Ua))
        assert max(errs) < MODE2_TOL[key], errs
        # components pinned at a bound do not move with theta
        U = sol["U"][b][:-1]
        act = (U - np.asarray(bnd[2]) < 1e-6) | (np.asarray(bnd[3]) - U < 1e-6)
        assert act.any()
        dU = aux["Ua"][b][:-1].reshape(-1, m, r)
        print("%s/%d: max |du/dtheta| %.3g on active components, %.3g overall" % (key, b, np.abs(dU[act]).max(), np.abs(dU).max()))
        assert np.abs(dU[act]).max() < 1e-6 * max(1.0, np.abs(dU).max())


def test_mode2_gradient_matches_finite_differences():
    """dL/dtheta of mode 2 = central differences of the re-solved bounded loss (the active set does not change)."""
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved("pendulum")
    T = float(fx["T"])
    b = 0
    th = np.array(fx["theta"][b], dtype=float)
    taus, wp = fx["taus"][b:b + 1], fx["wp"][b:b + 1]
    aux = oc.auxSysSolverBatch(oc.cocSolverBatch(fx["x0"][b:b + 1], T, th), taus, wp, sel, mode=DISC)

    def loss(t):
        s = oc.cocSolverBatch(fx["x0"][b:b + 1], T, t)
        return float(oc.auxSysSolverBatch(s, taus, wp, sel, mode=DISC)["loss"][0])
    for i in range(len(th)):
        h = 1e-5 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += h
        tm[i] -= h
        fd = (loss(tp) - loss(tm)) / (2 * h) / 2               # reference convention: dl_dy = y - wp (half the gradient)
        assert abs(fd - aux["dtheta"][0][i]) < 1e-6 * max(1.0, abs(fd)), (i, fd, aux["dtheta"][0][i])


def test_bound_multipliers_round_trip():
    """cpdp_get/set_bound_multipliers: mode 2 on a solution handed in from the host gives the same bits."""
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved("pendulum")
    mem = oc._device()
    a1 = oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=DISC)
    host = {k: np.array(sol[k]) for k in ("X", "U", "Lam", "Zl", "Zu", "mu")}
    ws = oc._workspace(nb)
    zeros = np.zeros_like(host["Zl"])
    oc._lib.set_bound_multipliers(mem.ptr(ws), int(ws.shape[0]), nb, oc.n_grid, oc.steps_per_grid, mem.ptr(zeros),
                                  mem.ptr(zeros), mem.ptr(np.zeros(nb)), 0)
    got = {k: np.empty_like(host[k]) for k in ("Zl", "Zu", "mu")}
    oc._lib.get_bound_multipliers(mem.ptr(ws), int(ws.shape[0]), nb, oc.n_grid, oc.steps_per_grid, mem.ptr(got["Zl"]),
                                  mem.ptr(got["Zu"]), mem.ptr(got["mu"]), 0)
    assert not got["Zl"].any() and not got["mu"].any()
    s2 = dict(sol, **{k: mem.from_host(v) for k, v in host.items()})
    a2 = oc.auxSysSolverBatch(s2, fx["taus"][:nb], fx["wp"][:nb], sel, mode=DISC)
    for k in ("Xa", "Ua", "loss", "dtheta"):
        assert np.array_equal(a1[k], a2[k]), k
    with pytest.raises(ValueError):
        oc.auxSysSolverBatch({k: v for k, v in sol.items() if k not in ("Zl", "Zu", "mu")}, fx["taus"][:nb], fx["wp"][:nb],
                             sel, mode=DISC)


def test_modes01_ignore_bounds():
    """Modes 0/1 restate the reference's auxiliary system, which knows no bounds: on a bounded solution mode 0 equals
    Oracle.aux on it."""
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved("pendulum")
    oc.rtol_back, oc.atol_back = TIGHT["rtol"], TIGHT["atol"]
    oc.rtol_fwd, oc.atol_fwd = TIGHT["rtol"], TIGHT["atol"]
    sol = oc.cocSolverBatch(fx["x0"][:1], float(fx["T"]), fx["theta"][:1])
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:1], fx["wp"][:1], sel, mode=COCSys.MODE_RK45)
    plain = Oracle(models.pendulum(), n_grid=orc.N)
    Xa, Ua, _ = plain.aux(sol["time_grid"], sol["X"][0], sol["U"][0], sol["Lam"][0], fx["theta"][0], back=dict(TIGHT),
                          fwd=dict(TIGHT))
    assert _rel(aux["Xa"][0], Xa) < 1e-6 and _rel(aux["Ua"][0], Ua) < 1e-6


# ------------------------------------------------------------------------------------------------ status and errors
def test_x0_outside_a_state_bound_is_infeasible():
    oc = emu_bounded_oc("robotarm_bounded", n_grid=10)
    x0 = np.array([[-np.pi / 2, 0.0, 0.0, 0.0], [-np.pi / 2, 0.0, 0.0, 4.5], [-np.pi / 2, 0.0, 0.0, -4.0]])
    th = np.array([3.0, 1.0, 1.0, 1.0, 1.0])
    sol = oc.cocSolverBatch(x0, 1.0, th)
    assert list(sol["status"]) == [1, 5, 5]
    assert sol["iters"][1] == 0 and sol["iters"][2] == 0
    aux = oc.auxSysSolverBatch(sol, [0.3], np.tile([[[-np.pi / 4, 2.0]]], (3, 1, 1)), [0, 1], mode=DISC)
    assert list(aux["aux_status"]) == [0, 3, 3]
    full = oc.reduceRows(oc.packRows(sol, aux))
    assert full[-1] == 2.0                                     # both infeasible rows count as failed


def test_bounded_newton_step_is_race_free():
    """ThreadSanitizer over the emulated barrier Newton step (and mode 2 of the bounded model)."""
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from tests.emu.bounds_support import emu_bounded_oc\n"
            "oc = emu_bounded_oc('pendulum_bounded', tsan=True)\n"
            "sol = oc.cocSolverBatch(np.zeros((1, 2)), 1.0, np.array([2.0, 1.0, 1.0]))\n"
            "aux = oc.auxSysSolverBatch(sol, [0.4], np.array([[[1.0]]]), [0], mode=2)\n"
            "print('bounded run', sol['status'], sol['iters'], aux['aux_status'])\n") % ROOT
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("bounded run [1]") == 1, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
