"""Adjoint of mode 2 and the autograd layer through the CUDA library on the device: the forward-mode and oracle checks of
test_adjoint.py, the full-size batch (unbounded and thrust-bounded) with batching / chunking invariance, and torch.optim steps
through cpdp_layer."""
import os

import numpy as np
import pytest

from tests.adjoint_oracle import AdjointOracle, BoundedAdjointOracle, contract
from tests.bounded_oracle import BoundedOracle
from tests.test_adjoint import X0_TOL, forward_mode, _interp_loss
from tests.test_bounds import CASES as BCASES, _fixture
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
    oc = (standard.STANDARD.get(name) or standard.BOUNDED[name])(n_grid=n_grid)
    oc.build(name=oc.lib_name)
    return oc


def _cot(rng, B, N, n, m):
    return rng.normal(size=(B, N + 1, n)), rng.normal(size=(B, N + 1, m))


@pytest.mark.parametrize("fix", list(CASES))
def test_adjoint_vs_forward_mode_and_oracle_gpu(torch_mod, fix):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = _oc(name, N)
    n, m, r = oc.n_state, oc.n_control, oc.n_auxvar
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    X, U, Lam, th, T = fx["X"][0], fx["U"][0], fx["Lam"][0], fx["theta"][0], float(fx["T"])
    sol = host_sol(oc, T, th, X[None], U[None], Lam[None], pd)
    Xbar, Ubar = _cot(np.random.default_rng(3), 1, N, n, m)
    adj = {k: _np(v) for k, v in oc.auxSysAdjointBatch(sol, Xbar, Ubar).items()}
    aux = {k: _np(v) for k, v in oc.auxSysSolverBatch(sol, fx["taus"][:1], fx["wp"][:1], sel, mode=oc.MODE_DISCRETE).items()}
    assert adj["aux_status"][0] == 0
    e_th = _rel(adj["theta_bar"], forward_mode(aux, Xbar, Ubar, n, m, r))
    orc = AdjointOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    DX, DU = orc.dx0_discrete(oc._time_grid(T, N), X, U, Lam, th)
    e_x0 = _rel(adj["x0_bar"][0], contract(DX, DU, Xbar[0], Ubar[0]))
    print("%s (GPU): theta_bar vs forward mode %.2e, x0_bar vs dense oracle %.2e" % (fix, e_th, e_x0))
    assert e_th <= 1e-12 and e_x0 <= 1e-10


@pytest.mark.parametrize("key", ["pendulum", "robotarm", "quadrotor"])
def test_bounded_adjoint_vs_forward_mode_and_oracle_gpu(torch_mod, key):
    name, fix, mk, sel, bnd, probs = BCASES[key]
    fx = _fixture(fix, probs)
    nb = len(probs)
    N, T = int(fx["n_grid"]), float(fx["T"])
    oc = _oc(name, N)
    n, m, r = oc.n_state, oc.n_control, oc.n_auxvar
    pd = fx["pdata"] if "pdata" in fx else None
    sol = oc.cocSolverBatch(fx["x0"][:nb], T, fx["theta"][:nb], pdata=pd)
    Xbar, Ubar = _cot(np.random.default_rng(11), nb, N, n, m)
    adj = {k: _np(v) for k, v in oc.auxSysAdjointBatch(sol, Xbar, Ubar).items()}
    aux = {k: _np(v) for k, v in oc.auxSysSolverBatch(sol, fx["taus"][:nb], fx["wp"][:nb], sel, mode=oc.MODE_DISCRETE).items()}
    assert (adj["aux_status"] == 0).all() and (_np(sol["status"]) == 1).all()
    e_th = _rel(adj["theta_bar"], forward_mode(aux, Xbar, Ubar, n, m, r))
    solver, ao = BoundedOracle(mk(), *bnd, n_grid=N), BoundedAdjointOracle(mk(), *bnd, n_grid=N)
    e_x0 = 0.0
    for b in range(nb):
        if pd is not None:
            solver.pd = ao.pd = pd[b]
        R = solver.solve_bounded(fx["x0"][b], T, fx["theta"][b])
        DX, DU = ao.dx0_discrete_bounded(R["time_grid"], R["X"], R["U"], R["Lam"], R["Zl"], R["Zu"], fx["theta"][b])
        e_x0 = max(e_x0, _rel(adj["x0_bar"][b], contract(DX, DU, Xbar[b], Ubar[b])))
    print("bounded %s (GPU): theta_bar vs forward mode %.2e, x0_bar vs dense oracle %.2e" % (key, e_th, e_x0))
    assert e_th <= 1e-12 and e_x0 <= X0_TOL[key]


@pytest.mark.parametrize("name", ["quadrotor", "quadrotor_bounded"])
def test_full_size_batching_and_chunks(torch_mod, name):
    """4096 quadrotor OCPs, N = 50 (unbounded and thrust-bounded): theta_bar = the Xa/Ua contraction of mode 2 to 1e-12 on every
    converged problem, zero rows elsewhere; rows bit-identical for 1/2/4/8-way splits of the batch and for the solution of
    gradIterBatch(chunks=2) against chunks=1."""
    torch = torch_mod
    from lfsd_b200 import synthetic
    oc = _oc(name, 50)
    B, N, n, m, r = 4096, 50, oc.n_state, oc.n_control, oc.n_auxvar
    qb = synthetic.quad_batch(B)
    rounds = 8 if name == "quadrotor" else int(_np(oc.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])["iters"]).max()) + 1
    args = (qb["x0"], 1.0, qb["theta"], qb["taus"], qb["wp"], qb["sel"])
    _, sol1, aux1 = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds)
    g = torch.Generator(device=sol1["X"].device).manual_seed(0)
    Xbar = torch.randn(B, N + 1, n, generator=g, device=sol1["X"].device, dtype=torch.float64)
    Ubar = torch.randn(B, N + 1, m, generator=g, device=sol1["X"].device, dtype=torch.float64)
    adj = oc.auxSysAdjointBatch(sol1, Xbar, Ubar)
    st, ast = _np(sol1["status"]), _np(adj["aux_status"])
    conv = (st == 1) & (ast == 0)
    print("%s, 4096 OCPs: solver status %s, adjoint aux status %s" % (name, np.bincount(st, minlength=6).tolist(),
                                                                   np.bincount(ast, minlength=5).tolist()))
    assert conv.sum() >= B - 8
    tb = _np(adj["theta_bar"])
    ref = torch.einsum("bkir,bki->br", aux1["Xa"].view(B, N + 1, n, r), Xbar) + \
        torch.einsum("bkjr,bkj->br", aux1["Ua"].view(B, N + 1, m, r), Ubar)
    ref = _np(ref)
    err = (np.linalg.norm(tb[conv] - ref[conv], axis=1) / np.linalg.norm(ref[conv], axis=1)).max()
    print("  theta_bar vs Xa/Ua contraction: worst row %.2e" % err)
    assert err <= 1e-12
    assert not tb[~conv].any() and not _np(adj["x0_bar"])[~conv].any()
    for G in (2, 4, 8):
        parts = ([], [])
        for gi in range(G):
            lo, hi = synthetic.shard_bounds(B, G, gi)
            part = dict(sol1, B=hi - lo, pdata=sol1["pdata"][lo:hi],
                        **{k: sol1[k][lo:hi] for k in ("X", "U", "Lam", "status", "Zl", "Zu", "mu") if k in sol1})
            a = oc.auxSysAdjointBatch(part, Xbar[lo:hi], Ubar[lo:hi])
            parts[0].append(_np(a["theta_bar"]))
            parts[1].append(_np(a["x0_bar"]))
        assert np.array_equal(np.concatenate(parts[0]), tb) and np.array_equal(np.concatenate(parts[1]), _np(adj["x0_bar"])), G
    _, sol2, _ = oc.gradIterBatch(*args, pdata=qb["goal"], mode=oc.MODE_DISCRETE, rounds=rounds, chunks=2)
    sol2.update(theta=sol1["theta"], theta_stride=sol1["theta_stride"], pdata=sol1["pdata"])
    adj2 = oc.auxSysAdjointBatch(sol2, Xbar, Ubar)
    torch.cuda.synchronize()
    for k in ("theta_bar", "x0_bar", "aux_status"):
        assert torch.equal(adj[k], adj2[k]), k


def test_layer_optim_quad_example(torch_mod):
    """torch.optim (SGD, Nesterov lr 0.01 momentum 0.9 as Examples/quad_example.py) through cpdp_layer with the waypoint loss
    written in torch: ten steps lower the loss, and every solve converges."""
    torch = torch_mod
    from lfsd_b200.autograd import cpdp_layer
    fx = _fx("quadexample")
    oc = _oc("quadrotor", 25)
    dev = torch.device("cuda", torch.cuda.current_device())
    th = torch.tensor(fx["theta"][0], dtype=torch.float64, device=dev, requires_grad=True)
    x0 = torch.tensor(fx["x0"], dtype=torch.float64, device=dev)
    pd = torch.tensor(fx["pdata"], dtype=torch.float64, device=dev)
    opt = torch.optim.SGD([th], lr=0.01, momentum=0.9, nesterov=True)
    losses = []
    for _ in range(10):
        opt.zero_grad()
        X, U, info = cpdp_layer(oc, x0, th, 1.0, pdata=pd)
        loss = _interp_loss(X, fx["taus"], fx["wp"], [0, 1, 2], 1.0)
        loss.backward()
        assert (_np(info["status"]) == 1).all() and (_np(info["aux_status"]) == 0).all()
        losses.append(float(loss.detach()))
        opt.step()
    print("quad_example through cpdp_layer: loss %s" % ["%.4f" % v for v in losses])
    assert losses[-1] < losses[0]
