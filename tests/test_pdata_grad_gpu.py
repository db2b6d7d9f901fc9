"""Adjoint with respect to the per-problem constants through the CUDA library on the device: the oracle checks of
test_pdata_grad.py, the full-size batch (unbounded and thrust-bounded) with batching / chunking invariance and theta_bar, x0_bar
equal to cpdp_aux_adjoint's, and goal recovery from noise-free demonstrations with torch.optim.Adam through cpdp_layer."""
import os

import numpy as np
import pytest

from tests.adjoint_oracle import contract
from tests.pdata_oracle import BoundedPdataOracle, PdataOracle
from tests.test_bounds import CASES as BCASES
from tests.test_discrete_grad import host_sol, _fx, _rel
from oracle import models

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
    oc = (standard.STANDARD.get(name) or standard.BOUNDED[name])(n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


def _cot(rng, B, N, n, m):
    return rng.normal(size=(B, N + 1, n)), rng.normal(size=(B, N + 1, m))


def test_quadrotor_pdata_bar_vs_oracle_gpu(torch_mod):
    fx = _fx("quadkat")
    N = int(fx["n_grid"])
    oc = _oc("quadrotor", N)
    pd = fx["pdata"][:1]
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    Xbar, Ubar = _cot(np.random.default_rng(3), 1, N, 13, 4)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    ref = oc.auxSysAdjointBatch(sol, Xbar, Ubar)
    assert int(_np(adj["aux_status"])[0]) == 0
    orc = PdataOracle(models.quadrotor(), n_grid=N)
    orc.pd = pd[0]
    DX, DU = orc.dpd_discrete(oc._time_grid(T, N), X, U, Lam, th)
    e = _rel(_np(adj["pdata_bar"])[0], contract(DX, DU, Xbar[0], Ubar[0]))
    d_th = _rel(_np(adj["theta_bar"]), _np(ref["theta_bar"]))
    d_x0 = _rel(_np(adj["x0_bar"]), _np(ref["x0_bar"]))
    print("quadrotor on the device: pdata_bar vs dense oracle %.2e; theta_bar, x0_bar vs cpdp_aux_adjoint %.2e, %.2e"
          % (e, d_th, d_x0))
    assert e <= 1e-9 and d_th <= 1e-14 and d_x0 <= 1e-14


def test_bounded_quadrotor_pdata_bar_vs_oracle_gpu(torch_mod):
    _, fix, mk, sel, bnd, _ = BCASES["quadrotor"]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = _oc("quadrotor_bounded", N)
    pd = fx["pdata"][:1]
    T = float(fx["T"])
    sol = oc.cocSolverBatch(fx["x0"][:1], T, fx["theta"][:1], pdata=pd)
    assert int(_np(sol["status"])[0]) == 1
    Xbar, Ubar = _cot(np.random.default_rng(4), 1, N, 13, 4)
    adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True)
    orc = BoundedPdataOracle(mk(), *bnd, n_grid=N)
    orc.pd = pd[0]
    h = {k: _np(sol[k])[0] for k in ("X", "U", "Lam", "Zl", "Zu")}
    DX, DU = orc.dpd_discrete_bounded(oc._time_grid(T, N), h["X"], h["U"], h["Lam"], h["Zl"], h["Zu"], fx["theta"][0])
    e = _rel(_np(adj["pdata_bar"])[0], contract(DX, DU, Xbar[0], Ubar[0]))
    print("bounded quadrotor on the device: pdata_bar vs dense oracle %.2e" % e)
    assert e <= 1e-8


@pytest.mark.parametrize("name", ["quadrotor", "quadrotor_bounded"])
def test_full_size_batching_and_chunks_pdata(torch_mod, name):
    """4096 quadrotor OCPs, N = 50: pdata_bar rows bit-identical for 1/2/4/8-way splits and for the solution of gradIterBatch(chunks=2);
    theta_bar and x0_bar equal to cpdp_aux_adjoint's; zero rows where the solve did not converge."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc(name, 50)
    B, N, n, m = 4096, 50, oc.n_state, oc.n_control
    qb = synthetic.quad_batch(B)
    rounds = 8 if name == "quadrotor" else int(_np(oc.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])["iters"]).max()) + 1
    args = (qb["x0"], 1.0, qb["theta"], qb["taus"], qb["wp"], qb["sel"])
    _, sol1, _ = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds)
    g = torch.Generator(device=sol1["X"].device).manual_seed(0)
    Xbar = torch.randn(B, N + 1, n, generator=g, device=sol1["X"].device, dtype=torch.float64)
    Ubar = torch.randn(B, N + 1, m, generator=g, device=sol1["X"].device, dtype=torch.float64)
    adj = oc.auxSysAdjointBatch(sol1, Xbar, Ubar, pdata_bar=True)
    ref = oc.auxSysAdjointBatch(sol1, Xbar, Ubar)
    st, ast = _np(sol1["status"]), _np(adj["aux_status"])
    conv = (st == 1) & (ast == 0)
    print("%s, 4096 OCPs: solver status %s, aux status %s" % (name, np.bincount(st, minlength=6).tolist(),
                                                             np.bincount(ast, minlength=5).tolist()))
    assert conv.sum() >= B - 8
    pb = _np(adj["pdata_bar"])
    assert not pb[~conv].any() and np.abs(pb[conv]).max() > 0
    d = {}
    for k in ("theta_bar", "x0_bar"):
        a_, r_ = _np(adj[k]), _np(ref[k])
        d[k] = float((np.abs(a_ - r_).max(axis=1) / np.maximum(np.abs(r_).max(axis=1), 1e-300)).max())
    print("  theta_bar, x0_bar vs cpdp_aux_adjoint: worst row %.2e, %.2e (bit-identical: %s)"
          % (d["theta_bar"], d["x0_bar"], all(torch.equal(adj[k], ref[k]) for k in d)))
    assert max(d.values()) <= 1e-14
    for G in (2, 4, 8):
        parts = []
        for gi in range(G):
            lo, hi = synthetic.shard_bounds(B, G, gi)
            part = dict(sol1, B=hi - lo, pdata=sol1["pdata"][lo:hi],
                        **{k: sol1[k][lo:hi] for k in ("X", "U", "Lam", "status", "Zl", "Zu", "mu") if k in sol1})
            parts.append(_np(oc.auxSysAdjointBatch(part, Xbar[lo:hi], Ubar[lo:hi], pdata_bar=True)["pdata_bar"]))
        assert np.array_equal(np.concatenate(parts), pb), G
    _, sol2, _ = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds, chunks=2)
    sol2.update(theta=sol1["theta"], theta_stride=sol1["theta_stride"], pdata=sol1["pdata"])
    adj2 = oc.auxSysAdjointBatch(sol2, Xbar, Ubar, pdata_bar=True)
    torch.cuda.synchronize()
    for k in ("pdata_bar", "theta_bar", "x0_bar", "aux_status"):
        assert torch.equal(adj[k], adj2[k]), k


def test_goal_recovery_with_adam(torch_mod):
    """Noise-free waypoint demonstrations (positions at nodes 5, 10, .., 25) of 16 synthetic.quad_batch problems solved at their
    true goals; the goals perturbed by N(0, 0.3^2); 40 Adam steps (lr 0.02) on the goals alone through cpdp_layer(pdata_grad=True)
    with the waypoint loss written in torch.  The loss falls below 2 % and the mean goal error below 60 % of their start values
    (first measured run on a B200: 0.85 % and 39 %, DESIGN.md §3.11)."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    from lfsd_b200.autograd import cpdp_layer
    oc = _oc("quadrotor", 25)
    dev = torch.device("cuda", torch.cuda.current_device())
    qb = synthetic.quad_batch(16)
    x0 = torch.tensor(qb["x0"], dtype=torch.float64, device=dev)
    th = torch.tensor(qb["theta"], dtype=torch.float64, device=dev)
    true = torch.tensor(qb["goal"], dtype=torch.float64, device=dev)
    nodes = [5, 10, 15, 20, 25]
    with torch.no_grad():
        X, _, info = cpdp_layer(oc, x0, th, 1.0, pdata=true)
        assert (_np(info["status"]) == 1).all()
        demo = X[:, nodes, :3].clone()
    gen = torch.Generator(device="cpu").manual_seed(1)
    goal = (true + 0.3 * torch.randn(true.shape, generator=gen, dtype=torch.float64).to(dev)).requires_grad_(True)
    opt = torch.optim.Adam([goal], lr=0.02)
    losses, errs = [], []
    for _ in range(40):
        opt.zero_grad()
        X, U, info = cpdp_layer(oc, x0, th, 1.0, pdata=goal, pdata_grad=True)
        loss = ((X[:, nodes, :3] - demo) ** 2).sum() / 16
        loss.backward()
        assert (_np(info["status"]) == 1).all() and (_np(info["aux_status"]) == 0).all()
        losses.append(float(loss.detach()))
        errs.append(float((goal.detach() - true).norm(dim=1).mean()))
        opt.step()
    print("goal recovery: loss %.3e -> %.3e, mean goal error %.3e -> %.3e" % (losses[0], losses[-1], errs[0], errs[-1]))
    print("  losses %s" % ["%.3e" % v for v in losses[::5]])
    assert losses[-1] < 0.02 * losses[0]
    assert errs[-1] < 0.6 * errs[0]
