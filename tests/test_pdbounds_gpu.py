"""Bounds that depend on pdata through the CUDA library on the device (DESIGN.md §3.12): the oracle checks of test_pdbounds.py, the
full-size batch with a per-problem thrust limit (batching / chunking invariance, theta_bar and x0_bar equal to cpdp_aux_adjoint's),
the same statuses and iterations as the compiled-in limit, and torque-limit recovery with torch.optim.Adam through cpdp_layer."""
import numpy as np
import pytest

from tests.adjoint_oracle import contract
from tests.bounded_oracle import BoundedOracle
from tests.pdbounds_oracle import PdBoundedOracle
from tests.test_bounds import _fixture, _rel
from tests.test_pdbounds import _model_with_pd, _pend_bnd
from oracle import models

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
    oc = (standard.PD_BOUNDED.get(name) or standard.BOUNDED[name])(n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


def test_pendulum_per_problem_limits_vs_oracles_gpu(torch_mod):
    """Per-problem torque limits: each row against BoundedOracle at its limit (equal iteration counts), pdata_bar against the
    dense perturbed-KKT oracle to 1e-11."""
    fx = _fixture("pendulum", [0])
    T = float(fx["T"])
    oc = _oc("pendulum_pdbounded", 10)
    P = np.array([[3.5], [5.0], [6.5]])
    x0, th = np.tile(fx["x0"], (3, 1)), np.tile(fx["theta"], (3, 1))
    sol = oc.cocSolverBatch(x0, T, th, pdata=P)
    h = {k: _np(sol[k]) for k in ("X", "U", "Lam", "Zl", "Zu", "status", "iters")}
    assert (h["status"] == 1).all()
    rng = np.random.default_rng(1)
    Xbar, Ubar = rng.normal(size=(3, 11, 2)), rng.normal(size=(3, 11, 1))
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    pb = _np(adj["pdata_bar"])
    mdl = _model_with_pd(models.pendulum, ["umax"])
    for b in range(3):
        r = BoundedOracle(models.pendulum(), *_pend_bnd(P[b]), n_grid=10).solve_bounded(x0[b], T, th[b])
        assert int(h["iters"][b]) == r["iters"]
        assert _rel(h["U"][b], r["U"]) < 1e-6
        orc = PdBoundedOracle(mdl, _pend_bnd, P[b], n_grid=10)
        DX, DU = orc.dpd_discrete_pdbounded(sol["time_grid"], h["X"][b], h["U"][b], h["Lam"][b], h["Zl"][b], h["Zu"][b], th[b])
        e = _rel(pb[b], contract(DX, DU, Xbar[b], Ubar[b]))
        print("umax %g on the device: pdata_bar vs dense oracle %.2e" % (P[b, 0], e))
        assert e <= 1e-11


def _quad_full(torch, fmax):
    from lfsd_b200 import synthetic
    B = 4096
    qb = synthetic.quad_batch(B)
    return qb, np.hstack([qb["goal"], np.broadcast_to(np.asarray(fmax, dtype=float).reshape(-1, 1), (B, 1))])


def test_full_size_per_problem_limits(torch_mod):
    """4096 quadrotor OCPs, N = 50, f_max uniform in [3.5, 5] per problem: solve rows, mode-2 rows and pdata_bar rows bit-identical
    for 1/2/4/8-way splits and gradIterBatch(chunks=2); theta_bar and x0_bar of cpdp_aux_adjoint_pd bit-identical to
    cpdp_aux_adjoint's."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    qb, P = _quad_full(torch, np.random.default_rng(7).uniform(3.5, 5.0, size=4096))
    oc = _oc("quadrotor_pdbounded", 50)
    B, N = 4096, 50
    args = (qb["x0"], 1.0, qb["theta"], qb["taus"], qb["wp"], qb["sel"])
    _, sol1, aux1 = oc.gradIterBatch(*args, pdata=P, mode=oc.MODE_DISCRETE)
    st = _np(sol1["status"])
    print("quadrotor_pdbounded, 4096 OCPs, per-problem f_max: solver status %s, iterations mean %.2f max %d"
          % (np.bincount(st, minlength=6).tolist(), _np(sol1["iters"])[st == 1].mean(), _np(sol1["iters"]).max()))
    assert (st == 1).sum() >= B - 8
    dev = sol1["X"].device
    g = torch.Generator(device=dev).manual_seed(0)
    Xbar = torch.randn(B, N + 1, 13, generator=g, device=dev, dtype=torch.float64)
    Ubar = torch.randn(B, N + 1, 4, generator=g, device=dev, dtype=torch.float64)
    adj = oc.auxSysAdjointBatch(sol1, Xbar, Ubar, pdata_bar=True)
    ref = oc.auxSysAdjointBatch(sol1, Xbar, Ubar)
    torch.cuda.synchronize()
    assert torch.equal(adj["theta_bar"], ref["theta_bar"]) and torch.equal(adj["x0_bar"], ref["x0_bar"])
    pb = _np(adj["pdata_bar"])
    assert np.abs(pb[:, 3]).max() > 0
    pdd = torch.from_numpy(P).to(dev)
    for G in (2, 4, 8):
        for gi in range(G):
            lo, hi = synthetic.shard_bounds(B, G, gi)
            s = oc.cocSolverBatch(qb["x0"][lo:hi], 1.0, qb["theta"], pdata=pdd[lo:hi])
            for k in ("X", "U", "Lam", "Zl", "Zu", "iters", "status"):
                assert torch.equal(s[k], sol1[k][lo:hi]), (G, gi, k)
            a = oc.auxSysSolverBatch(s, qb["taus"], qb["wp"][lo:hi], qb["sel"], mode=oc.MODE_DISCRETE)
            for k in ("Xa", "Ua", "loss", "dtheta"):
                assert torch.equal(a[k], aux1[k][lo:hi]), (G, gi, k)
            p = oc.auxSysAdjointBatch(s, Xbar[lo:hi], Ubar[lo:hi], pdata_bar=True)["pdata_bar"]
            assert np.array_equal(_np(p), pb[lo:hi]), (G, gi)
    rounds = int(_np(sol1["iters"]).max()) + 1                 # (chunks > 1 runs a fixed number of Newton rounds)
    _, sol2, aux2 = oc.gradIterBatch(*args, pdata=P, mode=oc.MODE_DISCRETE, rounds=rounds, chunks=2)
    sol2.update(theta=sol1["theta"], theta_stride=sol1["theta_stride"], pdata=sol1["pdata"])
    adj2 = oc.auxSysAdjointBatch(sol2, Xbar, Ubar, pdata_bar=True)
    torch.cuda.synchronize()
    for k in ("X", "U", "status", "iters"):
        assert torch.equal(sol1[k], sol2[k]), k
    for k in ("Xa", "loss", "dtheta"):
        assert torch.equal(aux1[k], aux2[k]), k
    for k in ("pdata_bar", "theta_bar", "x0_bar", "aux_status"):
        assert torch.equal(adj[k], adj2[k]), k


def test_full_size_same_limit_as_compiled_in(torch_mod):
    """f_max = 4 for every problem: the statuses and iteration counts of quadrotor_bounded (1 <= f_i <= 4 compiled in)."""
    torch = torch_mod
    qb, P = _quad_full(torch, 4.0)
    ob, op = _oc("quadrotor_bounded", 50), _oc("quadrotor_pdbounded", 50)
    sb = ob.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])
    sp_ = op.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=P)
    torch.cuda.synchronize()
    assert torch.equal(sb["status"], sp_["status"]) and torch.equal(sb["iters"], sp_["iters"])
    same = all(torch.equal(sb[k], sp_[k]) for k in ("X", "U", "Lam", "Zl", "Zu"))
    d = max(float((sb[k] - sp_[k]).abs().max()) for k in ("X", "U", "Lam"))
    print("f_max = 4 vs compiled-in limit: statuses %s, bit-identical %s, max |diff| %.2e"
          % (np.bincount(_np(sb["status"]), minlength=6).tolist(), same, d))


def test_limit_recovery_with_adam(torch_mod):
    """64 pendulums whose demonstrations saturate true torque limits in [4, 7]; the limits start perturbed by N(0, 0.4^2) (below
    the unbounded peak, so they stay active); 40 Adam steps (lr 0.05) on the limits alone through cpdp_layer(pdata_grad=True) with
    a trajectory loss written in torch.  The mean limit error falls below 35 % of its start (first measured run on a B200: 0.356 ->
    0.0257, 7.2 %, DESIGN.md §3.12)."""
    torch = torch_mod
    from lfsd_b200.autograd import cpdp_layer
    oc = _oc("pendulum_pdbounded", 10)
    dev = torch.device("cuda", torch.cuda.current_device())
    fx = _fixture("pendulum", [0])
    B = 64
    rng = np.random.default_rng(3)
    x0 = torch.tensor(np.tile(fx["x0"], (B, 1)), dtype=torch.float64, device=dev)
    th = torch.tensor(fx["theta"][0], dtype=torch.float64, device=dev)
    true = torch.tensor(rng.uniform(4.0, 7.0, size=(B, 1)), dtype=torch.float64, device=dev)
    with torch.no_grad():
        Xd, Ud, info = cpdp_layer(oc, x0, th, float(fx["T"]), pdata=true)
        assert (_np(info["status"]) == 1).all()
        assert ((Ud.abs().amax(dim=(1, 2)) - true[:, 0]).abs() < 1e-6).all(), "every demonstration saturates its limit"
    start = np.clip(_np(true) + rng.normal(0.0, 0.4, size=(B, 1)), 3.5, 7.5)
    lim = torch.tensor(start, dtype=torch.float64, device=dev, requires_grad=True)
    opt = torch.optim.Adam([lim], lr=0.05)
    losses, errs = [], []
    for _ in range(40):
        opt.zero_grad()
        X, U, info = cpdp_layer(oc, x0, th, float(fx["T"]), pdata=lim, pdata_grad=True)
        loss = (((X - Xd) ** 2).sum() + ((U - Ud) ** 2).sum()) / B
        loss.backward()
        assert (_np(info["status"]) == 1).all() and (_np(info["aux_status"]) == 0).all()
        losses.append(float(loss.detach()))
        errs.append(float((lim.detach() - true).abs().mean()))
        opt.step()
    print("limit recovery: loss %.3e -> %.3e, mean limit error %.3e -> %.3e" % (losses[0], losses[-1], errs[0], errs[-1]))
    print("  errors %s" % ["%.3e" % v for v in errs[::5]])
    assert errs[-1] < 0.35 * errs[0]
