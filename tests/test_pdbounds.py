"""Bounds that are expressions of the per-problem constants pdata (DESIGN.md §3.12): code generation, the per-problem barrier solve,
mode 2 and the pdata adjoint's bound term.  CPU tests: the kernels run in the thread emulation of tests/emu/ (built with the
companion header) through the same C ABI and COCSys host class as on the GPU, against tests/bounded_oracle.py and
tests/pdbounds_oracle.py."""
import os
import subprocess
import sys

import numpy as np
import pytest
import sympy as sp
import torch

from lfsd_b200 import codegen, standard
from lfsd_b200.autograd import cpdp_layer
from lfsd_b200.CPDP import COCSys, COCSys_TimeVarying
from lfsd_b200.sx import SX
from tests.adjoint_oracle import contract
from tests.bounded_oracle import BoundedOracle
from tests.emu.bounds_support import emu_bounded_oc
from tests.emu.pdbounds_support import emu_pdb_oc, emu_pdb_from
from tests.emu.support import emu_oc
from tests.pdbounds_oracle import PdBoundedOracle
from tests.test_adjoint import TorchCpuMem
from tests.test_bounds import CASES as BCASES, _fixture, _rel
from oracle import models

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DISC = COCSys.MODE_DISCRETE
BIG = 1e20

# (model header hash, companion header hash) of the thirteen standard libraries at the parent commit: unchanged
PARENT_HASHES = {
    'pendulum': ('8060fa1dbf420866', '7a26b781d97ed07c'), 'pendulum_tw2': ('8b6c6ff18ab3310e', '9beed08ea8cc3a2a'),
    'robotarm': ('3ef6a59ed973eded', 'e316644573b8c31d'), 'rocket': ('92262f39e2b65ed8', '155e53af74049621'),
    'quadrotor': ('196c06251c2aa0e7', 'e25fae2796766421'), 'cartpole': ('d8a1960df124c1eb', '8a538fd6e346527e'),
    'robotarm_wd': ('74bb0336cd353e80', '4fd3b0ba97f3330a'), 'quadrotor_cost1': ('444481be4fc5a54b', '8335808ae1ce945c'),
    'quadrotor_cost2': ('900a79bf3cb6760a', '3cf49de532ee416b'), 'rocket_cost1': ('081f3ca98c27ded5', '096281a78f9fef66'),
    'pendulum_bounded': ('72ca55267021e414', 'ee04bc741725f393'), 'robotarm_bounded': ('32302235f7f6ce59', 'f41bd38c741e6970'),
    'quadrotor_bounded': ('9f50d3d5569e4fbf', 'bc5edef539cf77d5')}

# pdata-bounded model -> (constant-bound twin, case of tests/test_bounds.py, the limits' pdata that reproduce the twin)
TWINS = {"pendulum_pdbounded": ("pendulum_bounded", "pendulum", [5.0]),
         "pendulum_pdbounded_ab": ("pendulum_bounded", "pendulum", [1.0, 2.0]),
         "robotarm_pdbounded": ("robotarm_bounded", "robotarm", [4.0]),
         "quadrotor_pdbounded": ("quadrotor_bounded", "quadrotor", [4.0])}


def _pend_bnd(pd):
    return [-BIG] * 2, [BIG] * 2, [-pd[0]], [pd[0]]


def _arm_bnd(pd):
    return [-BIG] * 3 + [-pd[0]], [BIG] * 3 + [pd[0]], [-3.0] * 2, [3.0] * 2


def _model_with_pd(mk, names):
    """An oracle model with extra per-problem constants that only the bounds use."""
    mdl = mk()
    mdl.pdata = list(mdl.pdata) + [sp.Symbol(s, real=True) for s in names]
    return mdl


def _pend(n_grid=10):
    return emu_pdb_oc("pendulum_pdbounded", n_grid=n_grid)


def _pfix():
    fx = _fixture("pendulum", [0, 1, 2])
    return fx, float(fx["T"])


def _cot(rng, B, N, n, m):
    return rng.normal(size=(B, N + 1, n)), rng.normal(size=(B, N + 1, m))


# ------------------------------------------------------------------------------------------------ code generation / host API
@pytest.mark.parametrize("name", sorted(PARENT_HASHES))
def test_standard_headers_unchanged(name):
    """Model and companion headers of the thirteen standard libraries are byte-identical to the parent's."""
    oc = (standard.STANDARD.get(name) or standard.VARIANTS.get(name) or standard.BOUNDED[name])()
    args = (oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar)
    tv = getattr(oc, "time", None)
    text, info = codegen.generate_model_header(oc.lib_name, *args, time=tv, bounds=oc._bounds())
    pd_text, pinfo = codegen.generate_pdata_header(oc.lib_name, *args, time=tv, bounds=oc._bounds())
    assert (info["hash"], pinfo["hash"]) == PARENT_HASHES[name]
    assert "BOUNDS_PD" not in text + pd_text and not oc.bounds_depend_on_pdata


def _exec_c(body, env):
    """Runs the generated C statements of a bound function body as Python (they are plain arithmetic on pd[])."""
    for line in body.strip().split("\n"):
        line = line.strip().rstrip(";")
        if not line or line.startswith("(void)"):
            continue
        exec(line.replace("const double ", ""), {}, env)


def test_generated_bounds_and_jacobians_match_sympy():
    """The generated XLB/XUB/ULB/UUB(i, pd) of the nonlinear model and its dbounds Jacobians against sympy at random pd; the
    library evaluates the same values (cpdp_eval_bounds)."""
    oc = standard.pendulum_pdbounded_ab_oc()
    args = (oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar)
    text, _ = codegen.generate_model_header("ab", *args, bounds=oc._bounds())
    pd_text, _ = codegen.generate_pdata_header("ab", *args, bounds=oc._bounds())
    assert "BOUNDS_PD = 1" in text and "BOUNDS_PD = 1" in pd_text
    a, b = sp.symbols("a b", real=True)
    lo, hi = -a * (1 + b ** 2), a + b ** 2
    body = pd_text[pd_text.index("static void dbounds"):]
    body = body[body.index("{") + 1:body.index("\n    }")]
    lib = emu_pdb_from(standard.pendulum_pdbounded_ab_oc(), "pendulum_pdbounded_ab")
    assert lib._lib.bounds_pd and np.isnan(lib._lib.lb[2]) and lib._lib.lb[:2] == [-BIG, -BIG]
    rng = np.random.default_rng(0)
    P = rng.uniform(-3, 3, size=(5, 2))
    lb, ub = lib.boundsBatch(P)
    for k, pd in enumerate(P):
        env = dict(pd=list(pd), dlb=[0.0] * 6, dub=[0.0] * 6)
        _exec_c(body, env)
        sub = {a: pd[0], b: pd[1]}
        for j, e in enumerate((lo, hi)):
            d = env["dlb" if j == 0 else "dub"]
            assert d[:4] == [0.0] * 4
            for q, s in enumerate((a, b)):
                assert abs(d[4 + q] - float(sp.diff(e, s).subs(sub))) <= 1e-14 * max(1.0, abs(d[4 + q]))
        assert abs(lb[k, 2] - float(lo.subs(sub))) <= 1e-14 * abs(lb[k, 2]) and abs(ub[k, 2] - float(hi.subs(sub))) <= 1e-14 * abs(ub[k, 2])
        assert list(lb[k, :2]) == [-BIG, -BIG] and list(ub[k, :2]) == [BIG, BIG]


def test_codegen_rejects_bounds_on_state_control_theta_time():
    oc = standard.pendulum_pdbounded_oc()
    for bad in (oc.env.X[0] if hasattr(oc.env.X, "__getitem__") else None, oc.env.U, SX.sym("beta")):
        oc.setControlVariable(oc.env.U, [-5.0], [bad])
        with pytest.raises(ValueError, match="bound may use only the problem variables"):
            oc.build(name="pdb_reject")
    tv = COCSys_TimeVarying("pdb_tv")
    t, x, u, g = SX.sym("t"), SX.sym("x"), SX.sym("u"), SX.sym("g")
    tv.setTimeVariable(t)
    tv.setAuxvarVariable(SX.sym("k"))
    tv.setStateVariable(x)
    tv.setControlVariable(u, [-1.0], [1.0 + t])
    tv.setProblemVariable(g)
    tv.setDyn(u)
    tv.setPathCost(u * u + (x - g) ** 2)
    tv.setFinalCost(x * x)
    with pytest.raises(ValueError, match="time"):
        tv.build(name="pdb_tv")
    # a numeric empty box still raises in the setter; a symbolic pair is checked per problem at run time
    with pytest.raises(ValueError):
        oc.setControlVariable(oc.env.U, [2.0], [1.0])
    umax = SX.sym("umax")
    oc.setControlVariable(oc.env.U, [umax], [-umax])
    assert oc.bounded and oc.bounds_depend_on_pdata


def test_eval_bounds_and_error_codes():
    """cpdp_eval_bounds for a pdata-bounded, a constant-bounded and an unbounded library; -1 and -8."""
    oc = _pend()
    P = np.array([[3.0], [7.5]])
    lb, ub = oc.boundsBatch(P)
    assert np.array_equal(lb, [[-BIG, -BIG, -3.0], [-BIG, -BIG, -7.5]]) and np.array_equal(ub, [[BIG, BIG, 3.0], [BIG, BIG, 7.5]])
    assert oc._lib.has_bounds and oc._lib.bounds_pd and oc.bounded and oc.bounds_depend_on_pdata
    with pytest.raises(ValueError):
        oc.boundsBatch()
    p = oc._device().ptr
    out = np.zeros((2, 3))
    assert oc._lib.L.cpdp_eval_bounds(None, 2, p(out), p(out), None) == -8
    assert oc._lib.L.cpdp_eval_bounds(p(P), 0, p(out), p(out), None) == -1
    assert oc._lib.L.cpdp_eval_bounds(p(P), 2, None, p(out), None) == -1
    cb = emu_bounded_oc("robotarm_bounded")
    lb, ub = cb.boundsBatch()
    assert lb.shape == (1, 6) and list(lb[0]) == [-BIG] * 3 + [-4.0, -3.0, -3.0] and list(ub[0]) == [BIG] * 3 + [4.0, 3.0, 3.0]
    assert not cb._lib.bounds_pd
    un = emu_oc("pendulum")
    lb, ub = un.boundsBatch()
    assert list(lb[0]) == [-BIG] * 3 and list(ub[0]) == [BIG] * 3


# ------------------------------------------------------------------------------------------------ the solve
@pytest.mark.parametrize("name", sorted(TWINS))
def test_equivalent_to_constant_twin(name):
    """At the constants of its BOUNDED twin, a PD_BOUNDED model gives the same statuses and iteration counts, and X, U, Lam, z to
    1e-12 (whether the rows are bit-identical is printed: the compiler may fold constant bounds differently)."""
    twin, case, lim = TWINS[name]
    _, fix, _, _, _, probs = BCASES[case]
    fx = _fixture(fix, probs)
    N = int(fx["n_grid"])
    ot = emu_bounded_oc(twin, n_grid=N)
    op = emu_pdb_oc(name, n_grid=N)
    nb = len(probs)
    base = fx["pdata"] if "pdata" in fx else np.zeros((nb, 0))
    pd_t = fx["pdata"] if "pdata" in fx else None
    pd_p = np.hstack([base, np.tile(lim, (nb, 1))])
    T = float(fx["T"])
    st = ot.cocSolverBatch(fx["x0"], T, fx["theta"], pdata=pd_t)
    sp_ = op.cocSolverBatch(fx["x0"], T, fx["theta"], pdata=pd_p)
    assert np.array_equal(st["status"], sp_["status"]) and np.array_equal(st["iters"], sp_["iters"])
    assert (st["status"] == 1).all()
    same = True
    for k in ("X", "U", "Lam", "Zl", "Zu", "mu"):
        e = np.abs(np.asarray(sp_[k]) - np.asarray(st[k])).max() / max(1.0, np.abs(st[k]).max())
        assert e <= 1e-12, (k, e)
        same &= np.array_equal(sp_[k], st[k])
    print("%s vs %s: bit-identical %s" % (name, twin, same))


def _per_problem(nlim=(3.5, 4.5, 5.5, 6.5)):
    """One pendulum problem of the fixture under a different torque limit per problem (all active: the unbounded peak is 9.95)."""
    fx, T = _pfix()
    B = len(nlim)
    x0, th = np.tile(fx["x0"][:1], (B, 1)), np.tile(fx["theta"][:1], (B, 1))
    return fx, T, x0, th, np.array(nlim).reshape(B, 1)


def test_per_problem_limits_match_oracle_and_rebatching():
    """Each row equals BoundedOracle run at that problem's limit (iteration counts equal); rows are bit-identical when the batch
    is cut or reordered, cold and warm; a converged guess takes 0 iterations."""
    fx, T, x0, th, P = _per_problem()
    oc = _pend()
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    assert (sol["status"] == 1).all()
    for b in range(len(P)):
        r = BoundedOracle(models.pendulum(), *_pend_bnd(P[b]), n_grid=oc.n_grid).solve_bounded(x0[b], T, th[b])
        assert r["status"] == "converged" and int(sol["iters"][b]) == r["iters"], (b, sol["iters"][b], r["iters"])
        for k in ("X", "U", "Lam", "Zl", "Zu"):
            assert _rel(sol[k][b], r[k]) < 1e-6, (k, b)
        assert abs(np.abs(sol["U"][b]).max() - P[b, 0]) < 1e-6          # the limit of this problem is active
    perm = [2, 0, 3, 1]
    s2 = oc.cocSolverBatch(x0[perm], T, th[perm], pdata=P[perm])
    for i, b in enumerate(perm):
        s1 = oc.cocSolverBatch(x0[b:b + 1], T, th[b:b + 1], pdata=P[b:b + 1])
        for k in ("X", "U", "Lam", "Zl", "Zu", "mu", "iters", "status"):
            assert np.array_equal(s1[k][0], sol[k][b]) and np.array_equal(s2[k][i], sol[k][b]), (k, b)
    # (a bounded model's warm start pushes the guess into the interior and restarts mu at mu_init: a few iterations, DESIGN.md §3.10)
    w = oc.cocSolverBatch(x0, T, th, pdata=P, init=sol)
    assert (w["status"] == 1).all() and (w["iters"] < sol["iters"]).all()
    guess = {k: np.asarray(sol[k])[perm] for k in ("X", "U", "Lam", "Zl", "Zu", "status")}
    for shift in (0, 1):
        wp = oc.cocSolverBatch(x0[perm], T, th[perm], pdata=P[perm], init=guess, shift=shift)
        w1 = oc.cocSolverBatch(x0, T, th, pdata=P, init=sol, shift=shift)
        for i, b in enumerate(perm):
            for k in ("X", "U", "Lam", "Zl", "Zu", "iters", "status"):
                assert np.array_equal(wp[k][i], w1[k][b]), (shift, k, b)


def test_infeasible_problems_alone_get_status_5():
    """lb(pd) >= ub(pd), a NaN limit, or x0 outside the problem's own state bound: status 5 at the start, cold and warm; the
    neighbours' rows do not change a bit; mode 2 skips them and pack_rows counts them as failed."""
    fx, T, x0, th, P = _per_problem((5.0, -1.0, 6.0, np.nan))
    oc = _pend()
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    assert list(sol["status"]) == [1, 5, 1, 5] and sol["iters"][1] == 0 and sol["iters"][3] == 0
    ok = oc.cocSolverBatch(x0[[0, 2]], T, th[[0, 2]], pdata=P[[0, 2]])
    for k in ("X", "U", "Lam", "Zl", "Zu", "mu", "iters"):
        assert np.array_equal(ok[k], np.asarray(sol[k])[[0, 2]]), k
    w = oc.cocSolverBatch(x0, T, th, pdata=P, init=dict(sol, status=np.ones(4, dtype=np.int32)))
    assert list(w["status"]) == [1, 5, 1, 5]
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:1].repeat(4, 0), fx["wp"][:1].repeat(4, 0), [0], mode=DISC)
    assert list(aux["aux_status"]) == [0, 3, 0, 3]
    assert oc.reduceRows(oc.packRows(sol, aux))[-1] == 2.0
    # the robot arm's state bound per problem: x0 = 4.5 is inside |dq2| <= 5, outside |dq2| <= 4
    arm = emu_pdb_oc("robotarm_pdbounded", n_grid=10)
    xa = np.array([[-np.pi / 2, 0.0, 0.0, 4.5]] * 2)
    s = arm.cocSolverBatch(xa, 1.0, np.array([3.0, 1.0, 1.0, 1.0, 1.0]), pdata=np.array([[5.0], [4.0]]))
    assert list(s["status"]) == [1, 5]


# ------------------------------------------------------------------------------------------------ mode 2 and the adjoint
def test_mode2_theta_gradient_with_per_problem_bounds():
    fx, T, x0, th, P = _per_problem((4.0, 6.5))
    oc = _pend()
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:1].repeat(2, 0), fx["wp"][:1].repeat(2, 0), [0], mode=DISC)
    assert (aux["aux_status"] == 0).all()
    for b in range(2):
        orc = BoundedOracle(models.pendulum(), *_pend_bnd(P[b]), n_grid=oc.n_grid)
        Xa, Ua = orc.aux_discrete_bounded(sol["time_grid"], sol["X"][b], sol["U"][b], sol["Lam"][b], sol["Zl"][b], sol["Zu"][b],
                                          th[b])
        assert max(_rel(aux["Xa"][b], Xa), _rel(aux["Ua"][b], Ua)) < 1e-10


def _pdbar_vs_oracle(oc, mdl, bnd, sol, b, Xbar, Ubar, adj, th):
    orc = PdBoundedOracle(mdl, bnd, np.asarray(sol["pdata"][b]), n_grid=oc.n_grid)
    DX, DU = orc.dpd_discrete_pdbounded(sol["time_grid"], sol["X"][b], sol["U"][b], sol["Lam"][b], sol["Zl"][b], sol["Zu"][b], th)
    return _rel(adj["pdata_bar"][b], contract(DX, DU, Xbar[b], Ubar[b])), DU


def test_pendulum_pdata_bar_vs_oracle():
    """Control-bound limit: pdata_bar against the dense implicit differentiation of the perturbed KKT system to 1e-11; on the
    intervals where |u| = umax is active dU/dumax = +-1; theta_bar and x0_bar are cpdp_aux_adjoint's, bit for bit."""
    fx, T, x0, th, P = _per_problem((4.0, 6.5, 30.0))
    oc = _pend()
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    assert (sol["status"] == 1).all()
    Xbar, Ubar = _cot(np.random.default_rng(1), 3, oc.n_grid, 2, 1)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    ref = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    assert (adj["aux_status"] == 0).all()
    assert np.array_equal(adj["theta_bar"], ref["theta_bar"]) and np.array_equal(adj["x0_bar"], ref["x0_bar"])
    mdl = _model_with_pd(models.pendulum, ["umax"])
    for b in range(2):
        e, DU = _pdbar_vs_oracle(oc, mdl, _pend_bnd, sol, b, Xbar, Ubar, adj, th[b])
        print("pendulum umax=%g: pdata_bar vs dense oracle %.2e" % (P[b, 0], e))
        assert e <= 1e-11
        U = sol["U"][b][:-1, 0]
        act = np.abs(np.abs(U) - P[b, 0]) < 1e-6
        assert act.any()
        assert np.abs(DU[:-1, 0, 0][act] - np.sign(U[act])).max() < 1e-6
    # a limit that binds nowhere has (almost) no gradient
    assert np.abs(np.asarray(sol["U"][2])).max() < 29.0
    assert abs(adj["pdata_bar"][2, 0]) < 1e-6 * np.abs(adj["theta_bar"][2]).max()


def test_nonlinear_limits_pdata_bar_vs_oracle():
    """ub = a + b^2, lb = -a (1 + b^2): the Jacobians' entries beyond +-1 enter pdata_bar."""
    fx, T, x0, th, _ = _per_problem((0.0, 0.0))
    P = np.array([[1.0, 1.8], [2.0, 0.9]])
    oc = emu_pdb_oc("pendulum_pdbounded_ab")
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    assert (sol["status"] == 1).all()
    Xbar, Ubar = _cot(np.random.default_rng(2), 2, oc.n_grid, 2, 1)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    mdl = _model_with_pd(models.pendulum, ["a", "b"])
    bnd = lambda pd: ([-BIG] * 2, [BIG] * 2, [-pd[0] * (1 + pd[1] ** 2)], [pd[0] + pd[1] ** 2])
    for b in range(2):
        e, _ = _pdbar_vs_oracle(oc, mdl, bnd, sol, b, Xbar, Ubar, adj, th[b])
        print("pendulum a, b = %s: pdata_bar vs dense oracle %.2e" % (P[b], e))
        assert e <= 1e-11


def test_robotarm_state_bound_pdata_bar_vs_oracle():
    """Active state bound |dq2| <= vmax: the recursion keeps ~1e-16 Sigma of relative accuracy (DESIGN.md §3.8), and the bound
    term enters the pdata column at the size of Sigma itself (DESIGN.md §3.12)."""
    _, fix, _, _, _, probs = BCASES["robotarm"]
    fx = _fixture(fix, probs)
    N = int(fx["n_grid"])
    oc = emu_pdb_oc("robotarm_pdbounded", n_grid=N)
    P = np.array([[4.0]])
    sol = oc.cocSolverBatch(fx["x0"], float(fx["T"]), fx["theta"], pdata=P)
    assert int(sol["status"][0]) == 1
    assert np.abs(np.abs(sol["X"][0][:, 3]) - 4.0).min() < 1e-6, "the state bound is not active"
    Xbar, Ubar = _cot(np.random.default_rng(3), 1, N, 4, 2)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    e, _ = _pdbar_vs_oracle(oc, _model_with_pd(models.robotarm, ["vmax"]), _arm_bnd, sol, 0, Xbar, Ubar, adj, fx["theta"][0])
    X = sol["X"][0][:, 3]
    sig = max((sol["Zl"][0][:, 3] / (X + 4.0)).max(), (sol["Zu"][0][:, 3] / (4.0 - X)).max())
    print("robotarm vmax: pdata_bar vs dense oracle %.2e, largest Sigma of the state bound %.2e" % (e, sig))
    assert e <= 1e-16 * sig


def test_quadrotor_goal_pdata_bar_unaffected_where_no_bound_is_active():
    """f_max far above the thrusts: goal columns of pdata_bar, theta_bar, x0_bar equal those of quadrotor_bounded with its lower
    bound 1 <= f_i only active nowhere either -- compared here with the quadrotor whose f_max column reads ~0."""
    _, fix, _, _, _, probs = BCASES["quadrotor"]
    fx = _fixture(fix, probs)
    N = int(fx["n_grid"])
    oc = emu_pdb_oc("quadrotor_pdbounded", n_grid=N)
    T = float(fx["T"])
    P = np.hstack([fx["pdata"], [[40.0]]])
    sol = oc.cocSolverBatch(fx["x0"], T, fx["theta"], pdata=P)
    assert int(sol["status"][0]) == 1
    Xbar, Ubar = _cot(np.random.default_rng(4), 1, N, 13, 4)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    mdl = _model_with_pd(lambda: models.quadrotor(), ["f_max"])
    bnd = lambda pd: ([-BIG] * 13, [BIG] * 13, [1.0] * 4, [pd[3]] * 4)
    e, _ = _pdbar_vs_oracle(oc, mdl, bnd, sol, 0, Xbar, Ubar, adj, fx["theta"][0])
    print("quadrotor f_max = 40: pdata_bar vs dense oracle %.2e, f_max column %.2e" % (e, adj["pdata_bar"][0, 3]))
    assert e <= 1e-9
    assert abs(adj["pdata_bar"][0, 3]) < 1e-6 * np.abs(adj["pdata_bar"][0, :3]).max()


def test_pdata_bar_matches_finite_differences_of_the_solve():
    """pdata_bar = central differences of l(umax) = sum Xbar.X + Ubar.U over the trajectory re-solved at tol 1e-12."""
    fx, T, x0, th, P = _per_problem((6.0,))
    oc = _pend()
    oc.tol = 1e-12
    Xbar, Ubar = _cot(np.random.default_rng(6), 1, oc.n_grid, 2, 1)

    def ell(p):
        s = oc.cocSolverBatch(x0, T, th, pdata=p)
        assert int(s["status"][0]) == 1
        return float((s["X"] * Xbar).sum() + (s["U"] * Ubar).sum())
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    g = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)["pdata_bar"][0, 0]
    h = 1e-5
    fd = (ell(P + h) - ell(P - h)) / (2 * h)
    err = abs(g - fd) / abs(g)
    print("pdata_bar (umax) vs finite differences: %.2e" % err)
    assert err <= 1e-5


def test_layer_gradcheck_with_active_limit():
    """gradcheck of cpdp_layer(pdata_grad=True) with respect to the torque limit (active) and x0 (float64)."""
    fx, T, x0, th, P = _per_problem((5.0, 6.0))
    oc = _pend()
    oc._mem = TorchCpuMem()
    oc.tol = 1e-12
    g = torch.Generator().manual_seed(0)
    N = oc.n_grid
    Pc = torch.randn(3, 2, N + 1, 2, generator=g, dtype=torch.float64)
    Qc = torch.randn(3, 2, N + 1, 1, generator=g, dtype=torch.float64)
    tht = torch.tensor(th[0], dtype=torch.float64)

    def f(x, pd):
        X, U, info = cpdp_layer(oc, x, tht, T, pdata=pd, pdata_grad=True)
        assert (info["status"] == 1).all()
        return torch.einsum("pbki,bki->p", Pc, X) + torch.einsum("pbkj,bkj->p", Qc, U)
    x = torch.tensor(x0, dtype=torch.float64, requires_grad=True)
    pd = torch.tensor(P, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(f, (x, pd), eps=1e-6, atol=1e-6, rtol=1e-4)


# ------------------------------------------------------------------------------------------------ races
def test_pdata_bound_kernels_are_race_free():
    """ThreadSanitizer over the emulated solve (per-problem bounds), mode 2 and the pdata adjoint with the bound term."""
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
            "from tests.emu.pdbounds_support import emu_pdb_oc\n"
            "oc = emu_pdb_oc('pendulum_pdbounded_ab', tsan=True)\n"
            "sol = oc.cocSolverBatch(np.zeros((2, 2)), 1.0, np.array([2.0, 1.0, 1.0]), pdata=np.array([[1.0, 1.5], [1.0, -1.0]]))\n"
            "w = oc.cocSolverBatch(np.zeros((2, 2)), 1.0, np.array([2.0, 1.0, 1.0]), pdata=np.array([[1.0, 1.5], [1.0, -1.0]]), init=sol)\n"
            "aux = oc.auxSysSolverBatch(sol, [0.4], np.array([[[1.0]], [[1.0]]]), [0], mode=2)\n"
            "rng = np.random.default_rng(0)\n"
            "adj = oc.auxSysAdjointBatch(sol, rng.normal(size=sol['X'].shape), rng.normal(size=sol['U'].shape), pdata_bar=True)\n"
            "print('pdbounds run', sol['status'], w['iters'], aux['aux_status'], adj['aux_status'])\n") % ROOT
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("pdbounds run [1 1] ") == 1 and "[0 0] [0 0]\n" in out, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
