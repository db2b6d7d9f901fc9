"""Box bounds through the CUDA library on the device: the oracle checks of test_bounds.py, the full-size bounded batch with
sharding / chunking invariance, and the device learner on a thrust-bounded quadrotor."""
import os

import numpy as np
import pytest

from tests.bounded_oracle import BoundedOracle
from tests.test_bounds import CASES, MODE2_TOL, _fixture, _rel, _slacks

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _np(t):
    return t.detach().cpu().numpy()


def _oc(name, n_grid):
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard
    oc = standard.BOUNDED[name](n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


@pytest.mark.parametrize("key", ["pendulum", "robotarm", "quadrotor"])
def test_bounded_solve_and_mode2_vs_oracle_gpu(torch_mod, key):
    from oracle.cpdp_oracle import Oracle, TIGHT
    name, fix, mk, sel, bnd, probs = CASES[key]
    fx = _fixture(fix, probs)
    nb = len(probs)
    N, T = int(fx["n_grid"]), float(fx["T"])
    oc = _oc(name, N)
    orc = BoundedOracle(mk(), *bnd, n_grid=N)
    pd = fx["pdata"] if "pdata" in fx else None
    sol = oc.cocSolverBatch(fx["x0"][:nb], T, fx["theta"][:nb], pdata=pd)
    aux = oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=oc.MODE_DISCRETE)
    h = {k: _np(sol[k]) for k in ("X", "U", "Lam", "Zl", "Zu", "status", "iters")}
    a = {k: _np(aux[k]) for k in ("Xa", "Ua", "aux_status")}
    for b in range(nb):
        if pd is not None:
            orc.pd = pd[b]
        r = orc.solve_bounded(fx["x0"][b], T, fx["theta"][b])
        errs = {k: _rel(h[k][b], r[k]) for k in ("X", "U", "Lam", "Zl", "Zu")}
        print("%s/%d (GPU): iterations %d (oracle %d), errors %s" % (key, b, h["iters"][b], r["iters"], errs))
        assert h["status"][b] == 1 and r["status"] == "converged" and h["iters"][b] == r["iters"]
        assert max(errs.values()) < 1e-6
        assert 0.0 < _slacks(h["X"][b], h["U"][b][:-1], bnd).min() < 1e-6
        assert a["aux_status"][b] == 0
        Xa, Ua = orc.aux_discrete_bounded(r["time_grid"], r["X"], r["U"], r["Lam"], r["Zl"], r["Zu"], fx["theta"][b])
        e2 = (_rel(a["Xa"][b], Xa), _rel(a["Ua"][b], Ua))
        print("  mode 2 vs dense perturbed-KKT oracle: Xa %.2e Ua %.2e" % e2)
        assert max(e2) < MODE2_TOL[key], e2
    if key == "pendulum":                 # modes 0/1 ignore the bounds: mode 0 = Oracle.aux at the bounded solution
        oc.rtol_back, oc.atol_back, oc.rtol_fwd, oc.atol_fwd = TIGHT["rtol"], TIGHT["atol"], TIGHT["rtol"], TIGHT["atol"]
        s1 = oc.cocSolverBatch(fx["x0"][:1], T, fx["theta"][:1], pdata=pd)
        a0 = oc.auxSysSolverBatch(s1, fx["taus"][:1], fx["wp"][:1], sel, mode=oc.MODE_RK45)
        Xa, Ua, _ = Oracle(mk(), n_grid=N).aux(sol["time_grid"], h["X"][0], h["U"][0], h["Lam"][0], fx["theta"][0],
                                               back=dict(TIGHT), fwd=dict(TIGHT))
        assert _rel(_np(a0["Xa"])[0], Xa) < 1e-6 and _rel(_np(a0["Ua"])[0], Ua) < 1e-6


def test_full_size_bounded_sharding_and_chunks(torch_mod):
    """4096 thrust-bounded quadrotor OCPs, N = 50: status counts of the adaptive solve (observed on a B200: see the assertion),
    then rows bit-identical for 1/2/4/8-way sharding of the batch and for chunks = 2 against chunks = 1 at a fixed round count."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc("quadrotor_bounded", 50)
    B = 4096
    qb = synthetic.quad_batch(B)
    sol = oc.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])
    st, it = _np(sol["status"]), _np(sol["iters"])
    counts = np.bincount(st, minlength=6).tolist()
    print("4096 bounded quadrotor OCPs: solver status", counts, "Newton iterations min/median/max", it.min(), np.median(it),
          it.max(), "rounds", oc._lib.last_rounds())
    assert counts[1] >= B - 8 and counts[4] == 0 and counts[5] == 0
    rounds = int(it.max()) + 1
    args = (qb["x0"], 1.0, qb["theta"], qb["taus"], qb["wp"], qb["sel"])
    red1, sol1, aux1 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds)
    assert np.array_equal(_np(sol1["status"]), st) and np.array_equal(_np(sol1["iters"]), it)
    ast = _np(aux1["aux_status"])
    assert (ast[st == 1] == 0).all() and np.isfinite(_np(aux1["dtheta"])).all()
    red2, sol2, aux2 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds, chunks=2)
    torch.cuda.synchronize()
    assert torch.equal(red1, red2)
    for k in ("Zl", "Zu", "mu"):
        assert torch.equal(sol1[k], sol2[k]), k
    for k in ("Xa", "Ua", "loss", "dtheta", "aux_status"):
        assert torch.equal(aux1[k], aux2[k]), k
    rows = _np(oc.packRows(sol1, aux1))
    for G in (2, 4, 8):
        parts = []
        for g in range(G):
            lo, hi = synthetic.shard_bounds(B, G, g)
            _, s, a = oc.gradIterBatch(qb["x0"][lo:hi], 1.0, qb["theta"], qb["taus"], qb["wp"][lo:hi], qb["sel"],
                                       pdata=qb["goal"][lo:hi], mode=oc.MODE_DISCRETE, rounds=rounds)
            parts.append(_np(oc.packRows(s, a)))
        assert np.array_equal(np.concatenate(parts), rows), G


def test_device_learner_mode2_bounded_quad_example(torch_mod):
    """DeviceLearner(mode=2) on the Examples/quad_example.py configuration with the thrusts bounded (1 <= f_i <= 4) runs to its
    stop rule with every OCP converged."""
    from lfsd_b200.optim import DeviceLearner
    fx = np.load(os.path.join(HERE, "golden", "oracle_quadexample.npz"))
    oc = _oc("quadrotor_bounded", 25)
    para = {"learning_rate": 0.01, "iter_num": 50, "method": "Nesterov", "mu": 0.9, "true_loss_print_flag": True}
    D = DeviceLearner(oc, fx["x0"], 1.0, fx["taus"][0], fx["wp"], [0, 1, 2], pdata=fx["pdata"], mode=oc.MODE_DISCRETE)
    D.load_optimization_function(para)
    th = D.run(fx["theta"][0])
    n = len(D.loss_trace)
    print("quad_example with thrust bounds, mode 2: %d iterations, loss %.4f -> %.4f, stopped early %s"
          % (n, D.loss_trace[0], D.loss_trace[-1], D.stopped_early))
    assert n >= 2 and np.isfinite(th).all() and np.isfinite(D.loss_trace).all()
