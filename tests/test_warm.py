"""Warm-started batched solve (cpdp_solve_warm, COCSys.cocSolverBatch(init=, shift=, mu_init=)).  CPU tests: the kernels run in
the thread emulation of tests/emu/ through the same C ABI and host classes as on the GPU, against the warm oracles of
tests/warm_oracle.py (the unchanged Newton iteration of oracle/cpdp_oracle.py and tests/bounded_oracle.py, started from the
guess)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from lfsd_b200.autograd import cpdp_layer
from tests.emu.support import emu_oc
from tests.emu.bounds_support import emu_bounded_oc
from tests.test_adjoint import _torch_oc
from tests.test_bounds import CASES as BCASES, _slacks, _solved
from tests.test_discrete_grad import CASES, _fx, _rel
from tests.warm_oracle import WarmBoundedOracle, WarmOracle, shifted, warm_point

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KEYS = ("X", "U", "Lam", "status", "iters", "kkt", "cost")


def perturbed(theta, seed=0):
    """theta' = theta (1 + 1e-2 xi), xi standard normal with a fixed seed."""
    th = np.asarray(theta, dtype=float)
    return th * (1.0 + 1e-2 * np.random.default_rng(seed).normal(size=th.shape))


def _unbounded(fix):
    name, mk, sel = CASES[fix]
    fx = _fx(fix)
    N = int(fx["n_grid"])
    oc = emu_oc(name, n_grid=N)
    pd = fx["pdata"][:1] if "pdata" in fx.files else None
    return oc, mk, fx, pd, N


# ------------------------------------------------------------------------------------------------ kernels against the oracle
@pytest.mark.parametrize("fix", list(CASES))
def test_warm_solve_matches_oracle(fix):
    """From the solution at theta, re-solve at theta': the kernels take the warm oracle's iterations (same count, same point) and
    end at the cold solve's solution at theta'.  Both stop at a KKT error below tol = 1e-10; the two solutions of the same NLP
    then differ by about the conditioning of its KKT matrix times tol, so they are compared at 1e-6 (relative, 2-norm)."""
    oc, mk, fx, pd, N = _unbounded(fix)
    x0, th, T = fx["x0"][:1], fx["theta"][0], float(fx["T"])
    th2 = perturbed(th)
    s0 = oc.cocSolverBatch(x0, T, th, pdata=pd)
    cold = oc.cocSolverBatch(x0, T, th2, pdata=pd)
    warm = oc.cocSolverBatch(x0, T, th2, pdata=pd, init=s0)
    assert int(s0["status"][0]) == 1 and int(cold["status"][0]) == 1 and int(warm["status"][0]) == 1
    orc = WarmOracle(mk(), n_grid=N)
    if pd is not None:
        orc.pd = pd[0]
    w0, lam0 = warm_point(x0[0], s0["X"][0], s0["U"][0], s0["Lam"][0])
    _, X, U, Lam, info = orc.solve_warm(x0[0], T, th2, w0, lam0)
    assert info["status"] == "converged"
    e = max(_rel(warm["X"][0], X), _rel(warm["U"][0], U), _rel(warm["Lam"][0], Lam))
    ec = max(_rel(warm["X"][0], cold["X"][0]), _rel(warm["U"][0], cold["U"][0]))
    print("%s: iterations cold %d, warm %d (oracle %d); warm vs oracle %.2e, warm vs cold %.2e"
          % (fix, cold["iters"][0], warm["iters"][0], info["iters"], e, ec))
    assert int(warm["iters"][0]) == info["iters"]
    assert e <= 1e-11
    assert ec <= 1e-6


@pytest.mark.parametrize("key", list(BCASES))
def test_bounded_warm_solve_matches_oracle(key):
    """Bounded models: the kernels follow the warm barrier oracle (IPOPT's warm_start_init_point: push 1e-3, z = max(z, 1e-3),
    mu = mu_init) with the same iteration count; every iterate stays strictly inside the box; the result matches the cold
    solve at theta' (1e-6, the tolerance of the bounded tests: the barrier solution moves by O(tol) / slack near an active
    bound)."""
    oc, orc, fx, pd, sel, bnd, nb, sol, ref = _solved(key)
    T = float(fx["T"])
    mk = BCASES[key][2]
    worc = WarmBoundedOracle(mk(), *bnd, n_grid=oc.n_grid)
    th2 = perturbed(fx["theta"][:nb])
    cold = oc.cocSolverBatch(fx["x0"][:nb], T, th2, pdata=pd)
    warm = oc.cocSolverBatch(fx["x0"][:nb], T, th2, pdata=pd, init=sol)
    for b in range(nb):
        if pd is not None:
            worc.pd = pd[b]
        r = worc.solve_warm(fx["x0"][b], T, th2[b], sol["X"][b], sol["U"][b], sol["Lam"][b], sol["Zl"][b], sol["Zu"][b],
                            mu_init=oc.warm_mu_init)
        assert r["status"] == "converged" and int(warm["status"][b]) == 1 and int(cold["status"][b]) == 1
        print("%s/%d: iterations cold %d, warm %d (oracle %d)" % (key, b, cold["iters"][b], warm["iters"][b], r["iters"]))
        assert int(warm["iters"][b]) == r["iters"]
        for k in ("X", "U", "Lam", "Zl", "Zu"):
            assert _rel(warm[k][b], r[k]) < 1e-6, (k, b, _rel(warm[k][b], r[k]))
        for k in ("X", "U"):
            assert _rel(warm[k][b], cold[k][b]) < 1e-6, (k, b, _rel(warm[k][b], cold[k][b]))
    # every iterate of the kernels: a fixed round count stops the solve after each iteration
    for rounds in range(1, int(warm["iters"].max()) + 1):
        s = oc.cocSolverBatch(fx["x0"][:nb], T, th2, pdata=pd, rounds=rounds, init=sol)
        assert _slacks(s["X"], s["U"][:, :-1], bnd).min() > 0.0, rounds


def test_converged_guess_takes_no_iteration():
    for fix in ("pendulum", "quadkat"):
        oc, mk, fx, pd, N = _unbounded(fix)
        x0, th, T = fx["x0"][:1], fx["theta"][:1], float(fx["T"])
        s0 = oc.cocSolverBatch(x0, T, th, pdata=pd)
        w = oc.cocSolverBatch(x0, T, th, pdata=pd, init=s0)
        assert int(w["status"][0]) == 1 and int(w["iters"][0]) == 0
        for k in ("X", "U", "Lam"):
            assert np.array_equal(w[k], s0[k])


# ------------------------------------------------------------------------------------------------ the starting point itself
def _start(oc, x0, T, th, init, shift, mu_init=None):
    """The starting point the warm kernel wrote: max_iter = 0 makes the first round stop before any step."""
    keep = oc.max_iter
    oc.max_iter = 0
    try:
        return oc.cocSolverBatch(x0, T, th, init=init, shift=shift, mu_init=mu_init)
    finally:
        oc.max_iter = keep


def test_shift_writes_the_specified_rows():
    oc, mk, fx, pd, N = _unbounded("pendulum")
    x0, th = fx["x0"], fx["theta"]
    g = dict(X=fx["X"].copy(), U=fx["U"].copy(), Lam=fx["Lam"].copy())
    for shift in (0, 1):
        s = _start(oc, x0, 1.0, th, g, shift)
        for b in range(len(x0)):
            X, U, L = shifted(g["X"][b], shift, N), shifted(g["U"][b], shift, N - 1), shifted(g["Lam"][b], shift, N)
            X[0] = x0[b]
            U[N] = U[N - 1]
            assert np.array_equal(s["X"][b], X) and np.array_equal(s["U"][b], U) and np.array_equal(s["Lam"][b], L)


def test_bounded_start_is_ipopts_warm_start_point():
    """Bounded pendulum (|u| <= 5): the guess (the fixture's unbounded optimum, outside the box) is pushed 1e-3 inside, z = max(z
    guess, 1e-3), or mu_init / slack without a z guess; with and without the shift."""
    oc = emu_bounded_oc("pendulum_bounded")
    fx = _fx("pendulum")
    N, x0 = oc.n_grid, fx["x0"]
    orc = WarmBoundedOracle(BCASES["pendulum"][2](), *BCASES["pendulum"][4], n_grid=N)
    rng = np.random.default_rng(2)
    Z = [rng.uniform(0.0, 2e-3, size=(len(x0), N + 1, 3)) for _ in range(2)]
    for shift in (0, 1):
        for zg in (None, Z):
            init = dict(X=fx["X"], U=fx["U"], Lam=fx["Lam"])
            if zg is not None:
                init.update(Zl=zg[0], Zu=zg[1])
            s = _start(oc, x0, 1.0, fx["theta"], init, shift, mu_init=1e-3)
            for b in range(len(x0)):
                w0, lam0 = warm_point(x0[b], fx["X"][b], fx["U"][b], fx["Lam"][b], shift)
                w = orc.start(w0)
                zs = None if zg is None else [shifted(z[b], shift, N) for z in zg]
                if zs is not None:              # the controls' z repeat row N-1
                    for z, zo in zip(zs, zg):
                        z[:N, 2] = shifted(zo[b][:, 2], shift, N - 1)[:N]
                zl, zu = orc.warm_z(w, *(zs if zs is not None else (None, None)), 1e-3)
                pad = lambda v: np.concatenate([v, np.zeros(1)]).reshape(N + 1, 3)
                assert np.array_equal(pad(w)[:, :2], s["X"][b]) and np.array_equal(pad(w)[:N, 2], s["U"][b][:N, 0])
                assert np.array_equal(s["Lam"][b], lam0.reshape(N + 1, 2))
                assert np.abs(pad(zl) - s["Zl"][b]).max() <= 1e-15 * np.abs(zl).max()
                assert np.abs(pad(zu) - s["Zu"][b]).max() <= 1e-15 * np.abs(zu).max()


# ------------------------------------------------------------------------------------------------ C ABI: aliasing, status, batching
def _abi_solve(oc, x0, th, T, guess, out, shift, init_status=None, mu_init=1e-4):
    """cpdp_solve_warm through the C ABI with explicit buffers (`guess` may be `out` itself)."""
    B, N, S = x0.shape[0], oc.n_grid, oc.steps_per_grid
    ws = oc._workspace(B)
    p = lambda a: 0 if a is None else a.ctypes.data
    return oc._lib.L.cpdp_solve_warm(p(ws), ws.shape[0], B, N, S, T, p(x0), p(th), oc.n_auxvar, 0, oc.tol, oc.max_iter, 0,
                                     p(out["X"]), p(out["U"]), p(out["Lam"]), p(out["status"]), p(out["iters"]), p(out["kkt"]),
                                     p(out["cost"]), 0, p(guess["X"]), p(guess["U"]), p(guess["Lam"]), None, None,
                                     p(init_status), shift, ctypes.c_double(mu_init))


def test_in_place_guess_is_bit_identical_to_separate_buffers():
    oc, mk, fx, pd, N = _unbounded("pendulum")
    x0, th = np.ascontiguousarray(fx["x0"]), perturbed(fx["theta"])
    s0 = oc.cocSolverBatch(x0, 1.0, fx["theta"])
    for shift in (0, 1):
        guess = {k: s0[k].copy() for k in ("X", "U", "Lam")}
        sep = {k: np.zeros_like(s0[k]) for k in KEYS}
        assert _abi_solve(oc, x0, th, 1.0, guess, sep, shift, init_status=s0["status"].copy()) == 0
        inp = {k: s0[k].copy() for k in KEYS}                    # guess, status and outputs in the same buffers
        assert _abi_solve(oc, x0, th, 1.0, inp, inp, shift, init_status=inp["status"]) == 0
        for k in KEYS:
            assert np.array_equal(sep[k], inp[k]), (shift, k)
        assert (sep["status"] == 1).all()


@pytest.mark.parametrize("bounded", [False, True])
def test_unconverged_init_status_gives_the_cold_solve(bounded):
    """A problem whose init_status is not converged starts from k_solve_init's seed: every output equals the cold solve's bits, for
    a full solve and after a fixed number of rounds."""
    oc = emu_bounded_oc("pendulum_bounded") if bounded else emu_oc("pendulum")
    fx = _fx("pendulum")
    x0, th = fx["x0"], perturbed(fx["theta"])
    s0 = oc.cocSolverBatch(x0, 1.0, fx["theta"])
    init = dict(s0, status=np.array([1, 2, 4], dtype=np.int32))
    for rounds in (0, 2):
        cold = oc.cocSolverBatch(x0, 1.0, th, rounds=rounds)
        warm = oc.cocSolverBatch(x0, 1.0, th, rounds=rounds, init=init)
        for k in KEYS + (("Zl", "Zu", "mu") if bounded else ()):
            assert np.array_equal(warm[k][1:], cold[k][1:]), (rounds, k)
        assert int(warm["iters"][0]) < int(cold["iters"][0]) or rounds


def test_rows_do_not_depend_on_batching():
    oc, mk, fx, pd, N = _unbounded("pendulum")
    x0, th = fx["x0"], perturbed(fx["theta"])
    s0 = oc.cocSolverBatch(x0, 1.0, fx["theta"])
    for shift in (0, 1):
        full = oc.cocSolverBatch(x0, 1.0, th, init=s0, shift=shift)
        for b in range(len(x0)):
            one = oc.cocSolverBatch(x0[b:b + 1], 1.0, th[b:b + 1], init={k: s0[k][b:b + 1] for k in ("X", "U", "Lam")},
                                    shift=shift)
            for k in KEYS:
                assert np.array_equal(full[k][b:b + 1], one[k]), (shift, b, k)


def test_init_none_is_the_cold_call():
    oc, mk, fx, pd, N = _unbounded("pendulum")
    a = oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"])
    b = oc.cocSolverBatch(fx["x0"], 1.0, fx["theta"], init=None, shift=1, mu_init=0.5)
    for k in KEYS:
        assert np.array_equal(a[k], b[k])


def test_argument_errors():
    oc, mk, fx, pd, N = _unbounded("pendulum")
    x0 = np.ascontiguousarray(fx["x0"])
    s0 = oc.cocSolverBatch(x0, 1.0, fx["theta"])
    out = {k: np.zeros_like(s0[k]) for k in KEYS}
    g = {k: s0[k].copy() for k in ("X", "U", "Lam")}
    assert _abi_solve(oc, x0, fx["theta"], 1.0, g, out, 2) == -12
    assert _abi_solve(oc, x0, fx["theta"], 1.0, g, out, -1) == -12
    assert _abi_solve(oc, x0, fx["theta"], 1.0, dict(g, U=None), out, 0) == -1
    assert _abi_solve(oc, x0, fx["theta"], 1.0, g, out, 0, mu_init=0.0) == 0          # (an unbounded model has no mu)
    ob = emu_bounded_oc("pendulum_bounded")
    sb = ob.cocSolverBatch(x0, 1.0, fx["theta"])
    gb = {k: sb[k].copy() for k in ("X", "U", "Lam")}
    outb = {k: np.zeros_like(sb[k]) for k in KEYS}
    assert _abi_solve(ob, x0, fx["theta"], 1.0, gb, outb, 0, mu_init=0.0) == -13
    assert _abi_solve(ob, x0, fx["theta"], 1.0, gb, outb, 0, mu_init=-1.0) == -13
    with pytest.raises(ValueError):
        oc.cocSolverBatch(x0, 1.0, fx["theta"], init=dict(g, X=g["X"][:, :-1]))
    with pytest.raises(ValueError):
        ob.cocSolverBatch(x0, 1.0, fx["theta"], init=dict(sb, Zu=None))


# ------------------------------------------------------------------------------------------------ the layer
def test_layer_with_init_gives_the_same_gradients():
    """cpdp_layer(init=...) is not differentiated through the guess: the gradients equal those without it to the accuracy of the
    two solutions (both converged to tol 1e-12)."""
    oc = _torch_oc("pendulum")
    oc.tol = 1e-12
    fx = _fx("pendulum")
    P = torch.from_numpy(np.random.default_rng(4).normal(size=(3, oc.n_grid + 1, 2)))
    x0 = torch.tensor(fx["x0"], requires_grad=True)
    th = torch.tensor(fx["theta"], requires_grad=True)
    X, U, info = cpdp_layer(oc, x0, th, 1.0)
    (X * P).sum().backward()
    g0 = (x0.grad.clone(), th.grad.clone())
    x0.grad = th.grad = None
    th2 = torch.tensor(perturbed(fx["theta"]))
    Xp, Up, infop = cpdp_layer(oc, x0.detach(), th2, 1.0)
    Xw, Uw, infow = cpdp_layer(oc, x0, th, 1.0, init=dict(infop, X=Xp, U=Up))
    assert (infow["status"] == 1).all() and (infow["iters"] > 0).all()
    (Xw * P).sum().backward()
    e = max(_rel(x0.grad.numpy(), g0[0].numpy()), _rel(th.grad.numpy(), g0[1].numpy()))
    print("layer gradients with init vs without: %.2e (solutions %.2e)" % (e, _rel(Xw.detach().numpy(), X.detach().numpy())))
    assert e <= 1e-8


# ------------------------------------------------------------------------------------------------ races
@pytest.mark.parametrize("model", ["pendulum", "pendulum_bounded"])
def test_warm_kernel_is_race_free(model):
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "tsan_warm_run.py"), model], capture_output=True,
                       text=True, env=env, timeout=900)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    assert out.count("warm run") == 2, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
