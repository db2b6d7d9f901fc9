"""Warm-started batched solve through the CUDA library on the device: the oracle checks of test_warm.py, the full-size batch with
sharding / chunking invariance, a receding-horizon loop and the warm-started device learner."""
import numpy as np
import pytest

from tests.test_bounds import CASES as BCASES, _fixture, _slacks
from tests.test_discrete_grad import CASES, _fx, _rel
from tests.test_warm import perturbed
from tests.warm_oracle import WarmBoundedOracle, WarmOracle, warm_point

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _oc(name, n_grid, bounded=False):
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard
    oc = (standard.BOUNDED if bounded else standard.STANDARD)[name](n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


@pytest.mark.parametrize("fix", list(CASES))
def test_warm_solve_matches_oracle_gpu(torch_mod, fix):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    from lfsd_b200 import standard
    oc = (standard.STANDARD.get(name) or standard.VARIANTS[name])(n_grid=N)
    oc.build(name=oc.lib_name)
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    x0, th, T = fx["x0"][:1], fx["theta"][0], float(fx["T"])
    th2 = perturbed(th)
    s0 = oc.cocSolverBatch(x0, T, th, pdata=pd)
    warm = oc.cocSolverBatch(x0, T, th2, pdata=pd, init=s0)
    cold = oc.cocSolverBatch(x0, T, th2, pdata=pd)
    orc = WarmOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    w0, lam0 = warm_point(x0[0], _np(s0["X"])[0], _np(s0["U"])[0], _np(s0["Lam"])[0])
    _, X, U, Lam, info = orc.solve_warm(x0[0], T, th2, w0, lam0)
    e = max(_rel(_np(warm["X"])[0], X), _rel(_np(warm["U"])[0], U), _rel(_np(warm["Lam"])[0], Lam))
    ec = max(_rel(_np(warm["X"])[0], _np(cold["X"])[0]), _rel(_np(warm["U"])[0], _np(cold["U"])[0]))
    print("%s (GPU): iterations cold %d, warm %d (oracle %d); warm vs oracle %.2e, warm vs cold %.2e"
          % (fix, _np(cold["iters"])[0], _np(warm["iters"])[0], info["iters"], e, ec))
    assert int(_np(warm["status"])[0]) == 1 and int(_np(warm["iters"])[0]) == info["iters"]
    assert e <= 1e-11 and ec <= 1e-6


@pytest.mark.parametrize("key", list(BCASES))
def test_bounded_warm_solve_matches_oracle_gpu(torch_mod, key):
    name, fix, mk, sel, bnd, probs = BCASES[key]
    fx = _fixture(fix, probs)
    nb, T, N = len(probs), float(fx["T"]), int(fx["n_grid"])
    oc = _oc(name, N, bounded=True)
    pd = fx["pdata"] if "pdata" in fx else None
    s0 = oc.cocSolverBatch(fx["x0"], T, fx["theta"], pdata=pd)
    th2 = perturbed(fx["theta"])
    warm = oc.cocSolverBatch(fx["x0"], T, th2, pdata=pd, init=s0)
    worc = WarmBoundedOracle(mk(), *bnd, n_grid=N)
    h = {k: _np(v) for k, v in s0.items() if k in ("X", "U", "Lam", "Zl", "Zu")}
    w = {k: _np(v) for k, v in warm.items() if k in ("X", "U", "Lam", "Zl", "Zu", "iters", "status")}
    for b in range(nb):
        if pd is not None:
            worc.pd = pd[b]
        r = worc.solve_warm(fx["x0"][b], T, th2[b], h["X"][b], h["U"][b], h["Lam"][b], h["Zl"][b], h["Zu"][b],
                            mu_init=oc.warm_mu_init)
        print("%s/%d (GPU): warm iterations %d (oracle %d)" % (key, b, w["iters"][b], r["iters"]))
        assert int(w["status"][b]) == 1 and int(w["iters"][b]) == r["iters"]
        for k in ("X", "U", "Lam", "Zl", "Zu"):
            assert _rel(w[k][b], r[k]) < 1e-6, (k, b)
        assert _slacks(w["X"][b], w["U"][b][:-1], bnd).min() > 0.0


@pytest.mark.parametrize("bounded", [False, True])
def test_full_size_warm_start_sharding_and_chunks(torch_mod, bounded):
    """4096 quadrotor OCPs, N = 50 (thrust-bounded: 1 <= f_i <= 4): warm-started at theta' from the solution at theta, every
    problem converges; rows are bit-identical for 1/2/4/8-way splits and for chunks = 2 against 1."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc("quadrotor_bounded" if bounded else "quadrotor", 50, bounded=bounded)
    B = 4096
    qb = synthetic.quad_batch(B)
    th2 = perturbed(qb["theta"])
    s0 = oc.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])
    assert (_np(s0["status"]) == 1).all()
    keys = ("X", "U", "Lam", "status", "iters", "kkt", "cost") + (("Zl", "Zu", "mu") if bounded else ())
    full = oc.cocSolverBatch(qb["x0"], 1.0, th2, pdata=qb["goal"], init=s0)
    it = _np(full["iters"])
    print("4096 quadrotor OCPs%s: warm iterations mean %.2f max %d (cold at theta: mean %.2f)"
          % (" (thrust-bounded)" if bounded else "", it.mean(), it.max(), _np(s0["iters"]).mean()))
    assert (_np(full["status"]) == 1).all()
    for G in (2, 4, 8):
        for g in range(G):
            lo, hi = synthetic.shard_bounds(B, G, g)
            part = oc.cocSolverBatch(qb["x0"][lo:hi], 1.0, th2, pdata=qb["goal"][lo:hi],
                                     init={k: s0[k][lo:hi] for k in ("X", "U", "Lam", "Zl", "Zu", "status") if k in s0})
            for k in keys:
                assert torch.equal(part[k], full[k][lo:hi]), (G, g, k)
    args = (qb["x0"], 1.0, th2, qb["taus"], qb["wp"], qb["sel"])
    r = int(it.max()) + 1
    red1, sol1, aux1 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=r, init=s0)
    red2, sol2, aux2 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=r, chunks=2, init=s0)
    torch.cuda.synchronize()
    assert torch.equal(red1, red2)
    for k in keys:
        assert torch.equal(sol1[k], sol2[k]), k


def test_receding_horizon_loop(torch_mod):
    """20 receding-horizon steps on 4096 quadrotors (N = 50): x <- X[:, 1] of the last solve; shift = 1 warm starts against cold
    starts from the same states.  Every solve converges and the applied controls U[:, 0] agree to 1e-6 (relative to their
    scale): both solves stop at a KKT error below tol = 1e-10 on the same NLP."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc("quadrotor", 50)
    qb = synthetic.quad_batch(4096)
    goal = torch.from_numpy(qb["goal"]).cuda()
    x = torch.from_numpy(qb["x0"]).cuda()
    prev = None
    worst, its_w, its_c = 0.0, [], []
    for step in range(20):
        warm = oc.cocSolverBatch(x, 1.0, qb["theta"], pdata=goal, init=prev, shift=1)
        cold = oc.cocSolverBatch(x, 1.0, qb["theta"], pdata=goal)
        assert (_np(warm["status"]) == 1).all() and (_np(cold["status"]) == 1).all(), step
        du = (warm["U"][:, 0] - cold["U"][:, 0]).abs().max().item() / cold["U"][:, 0].abs().max().item()
        worst = max(worst, du)
        its_w.append(_np(warm["iters"]).mean())
        its_c.append(_np(cold["iters"]).mean())
        prev = warm
        x = warm["X"][:, 1].contiguous()
    print("receding horizon, 20 steps: mean iterations warm %.2f, cold %.2f; applied controls agree to %.2e"
          % (np.mean(its_w[1:]), np.mean(its_c), worst))
    assert worst <= 1e-6


def test_device_learner_warm_start_quad_example(torch_mod):
    """DeviceLearner(mode=2, warm_start=True) on the Examples/quad_example.py configuration stops by its rule at the same iteration
    as the cold run, and its loss trace agrees with the cold run's to 1e-6 relative (the solutions differ at the solver
    tolerance, and the learner amplifies that over its iterations)."""
    from lfsd_b200.optim import DeviceLearner
    fx = _fx("quadexample")
    oc = _oc("quadrotor", 25)
    para = {"learning_rate": 0.01, "iter_num": 50, "method": "Nesterov", "mu": 0.9, "true_loss_print_flag": True}
    runs = {}
    for warm in (False, True):
        D = DeviceLearner(oc, fx["x0"], 1.0, fx["taus"][0], fx["wp"], [0, 1, 2], pdata=fx["pdata"], mode=oc.MODE_DISCRETE,
                          warm_start=warm)
        D.load_optimization_function(para)
        D.run(fx["theta"][0])
        runs[warm] = (np.array(D.loss_trace), D.stopped_early)
    (lc, sc), (lw, sw) = runs[False], runs[True]
    e = np.abs(lw - lc).max() / np.abs(lc).max() if len(lw) == len(lc) else np.inf
    print("quad_example, mode 2: %d iterations cold, %d warm; loss traces agree to %.2e" % (len(lc), len(lw), e))
    assert len(lw) == len(lc) and sw == sc
    assert e <= 1e-6
