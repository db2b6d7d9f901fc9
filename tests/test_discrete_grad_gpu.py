"""Discrete auxiliary mode (cpdp_aux mode 2) through the CUDA library on the device: the oracle and finite-difference checks of
test_discrete_grad.py, the full-size batch, sharding / chunking invariance and the device learner."""
import os

import numpy as np
import pytest

from tests.discrete_oracle import DiscreteOracle
from tests.test_discrete_grad import CASES, host_sol, _fx, _rel

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
    oc = standard.STANDARD[name](n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


@pytest.mark.parametrize("fix", list(CASES))
def test_mode2_vs_dense_oracle_gpu(torch_mod, fix):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = _oc(name, N)
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    orc = DiscreteOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    aux = oc.auxSysSolverBatch(host_sol(oc, T, th, X[None], U[None], Lam[None], pd), fx["taus"][:1], fx["wp"][:1], sel,
                               mode=oc.MODE_DISCRETE)
    assert int(_np(aux["aux_status"])[0]) == 0 and not _np(aux["counters"]).any()
    tg = oc._time_grid(T, N)
    Xa, Ua = orc.aux_discrete(tg, X, U, Lam, th)
    loss, dl = orc.loss_grad(fx["taus"][0], fx["wp"][0], tg, X, Xa, sel=sel)
    errs = (_rel(_np(aux["Xa"])[0], Xa), _rel(_np(aux["Ua"])[0], Ua), abs(_np(aux["loss"])[0] - loss) / max(abs(loss), 1e-300),
            _rel(_np(aux["dtheta"])[0], dl))
    print("%s (GPU): Xa %.2e Ua %.2e loss %.2e dL/dtheta %.2e" % ((fix,) + errs))
    assert max(errs) < 1e-8, errs


def test_gradient_matches_finite_differences_gpu(torch_mod):
    """dL/dtheta of mode 2 = central differences of the end-to-end loss re-solved at tol 1e-12 (quadrotor, N = 25, stored run)."""
    g = np.load(os.path.join(HERE, "golden", "quad_run.npz"))
    oc = _oc("quadrotor", 25)
    oc.tol = 1e-12
    th = g["parameter_trace"][0].astype(float)
    x0, pd, taus, wp = g["ini_state"].reshape(1, 13), g["goal_position"].reshape(1, 3), g["time_grid"], g["waypoints"].reshape(1, -1, 3)

    def run(t, mode=oc.MODE_DISCRETE):
        sol = oc.cocSolverBatch(x0, 1.0, t, pdata=pd)
        assert int(_np(sol["status"])[0]) == 1
        return oc.auxSysSolverBatch(sol, taus, wp, [0, 1, 2], mode=mode)

    gr = _np(run(th)["dtheta"])[0].copy()
    fd = np.zeros_like(gr)
    for i in range(len(th)):
        h = 1e-5 * max(1.0, abs(th[i]))
        tp, tm = th.copy(), th.copy()
        tp[i] += h
        tm[i] -= h
        fd[i] = 0.5 * (_np(run(tp)["loss"])[0] - _np(run(tm)["loss"])[0]) / (2 * h)
    err = np.abs(gr - fd).max() / np.abs(gr).max()
    gap = np.abs(_np(run(th, mode=oc.MODE_BDF)["dtheta"])[0] - gr).max() / np.abs(gr).max()
    print("quadrotor N=25 (GPU): finite differences vs mode 2 %.2e; mode 1 vs mode 2 (information only) %.2e" % (err, gap))
    assert err < 1e-6


def test_full_size_sharding_and_chunks(torch_mod):
    """4096 quadrotor OCPs, N = 50: every converged problem gets aux_status 0; per-problem rows are bit-identical for 1/2/4/8-way
    sharding of the batch and for chunks = 2 against chunks = 1."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc("quadrotor", 50)
    B = 4096
    qb = synthetic.quad_batch(B)
    args = (qb["x0"], 1.0, qb["theta"], qb["taus"], qb["wp"], qb["sel"])
    red1, sol1, aux1 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=8)
    st, ast = _np(sol1["status"]), _np(aux1["aux_status"])
    print("4096 quadrotor OCPs, mode 2: solver status", np.bincount(st, minlength=5).tolist(), "aux status",
          np.bincount(ast, minlength=6).tolist())
    conv = st == 1
    assert conv.any() and (ast[conv] == 0).all()
    assert np.isfinite(_np(aux1["dtheta"])).all()
    red2, sol2, aux2 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=8, chunks=2)
    torch.cuda.synchronize()
    assert torch.equal(red1, red2)
    for k in ("Xa", "Ua", "loss", "dtheta", "aux_status"):
        assert torch.equal(aux1[k], aux2[k]), k
    rows = _np(oc.packRows(sol1, aux1))
    for G in (2, 4, 8):
        parts = []
        for g in range(G):
            lo, hi = synthetic.shard_bounds(B, G, g)
            _, s, a = oc.gradIterBatch(qb["x0"][lo:hi], 1.0, qb["theta"], qb["taus"], qb["wp"][lo:hi], qb["sel"],
                                       pdata=qb["goal"][lo:hi], mode=oc.MODE_DISCRETE, rounds=8)
            parts.append(_np(oc.packRows(s, a)))
        assert np.array_equal(np.concatenate(parts), rows), G


def test_device_learner_mode2_quad_example(torch_mod):
    """DeviceLearner(mode=2) on the Examples/quad_example.py configuration (n_grid 25, Nesterov lr 0.01 mu 0.9 with the second
    evaluation per iteration, 50 iterations at most) runs to its stop rule and its loss decreases."""
    from lfsd_b200.optim import DeviceLearner
    fx = _fx("quadexample")
    oc = _oc("quadrotor", 25)
    para = {"learning_rate": 0.01, "iter_num": 50, "method": "Nesterov", "mu": 0.9, "true_loss_print_flag": True}
    D = DeviceLearner(oc, fx["x0"], 1.0, fx["taus"][0], fx["wp"], [0, 1, 2], pdata=fx["pdata"], mode=oc.MODE_DISCRETE)
    D.load_optimization_function(para)
    th = D.run(fx["theta"][0])
    n = len(D.loss_trace)
    print("quad_example, mode 2: %d iterations, loss %.4f -> %.4f, stopped early %s" % (n, D.loss_trace[0], D.loss_trace[-1],
                                                                                     D.stopped_early))
    assert n >= 2 and np.isfinite(th).all()
    assert D.loss_trace[-1] < D.loss_trace[0]
