"""CPU tests (thread emulation) of the eigen-path Newton solve of k_riccati_bdf (csrc/cpdp_bdf.cuh, bdf_eig_basis):
the Lyapunov system X + c (L X + X L') = B solved by a block-diagonal scaling in a real eigenvector basis of L, with a
per-Jacobian fall-back to the Bartels-Stewart sweep when the basis is ill-conditioned.

`tests/golden/bdf_sweep_outputs.npz` holds the outputs of the sweep-only solver (the revision before the eigen path,
computed with `_run_configs` below through its emulation): a build with -DCPDP_BDF_EIG_KAPPA=0 must reproduce them bit for bit."""
import hashlib
import os

import numpy as np
import pytest

from lfsd_b200 import _capi, codegen, standard
from tests.emu.build_emu import build
from tests.emu.support import NumpyMem, _BUILD

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "bdf_sweep_outputs.npz")


def _emu(name, flags=()):
    """COCSys for standard model `name` bound to the emulated kernels compiled with the extra `flags`."""
    oc = standard.STANDARD[name]()
    text, _ = codegen.generate_model_header(name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost,
                                            oc.final_cost, oc.pvar)
    os.makedirs(_BUILD, exist_ok=True)
    src = "".join(open(os.path.join(_capi.CSRC, fn)).read() for fn in sorted(os.listdir(_capi.CSRC))
                  if os.path.isfile(os.path.join(_capi.CSRC, fn)))
    src += open(os.path.join(HERE, "emu", "emu_lib.cpp")).read()
    tag = hashlib.sha1((text + src + " ".join(flags)).encode()).hexdigest()[:12]
    hdr = os.path.join(_BUILD, "model_%s_eig_%s.cuh" % (name, tag))
    so = os.path.join(_BUILD, "libemu_%s_eig_%s.so" % (name, tag))
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        build(hdr, so, ns="cpdp_emu_eig_" + name, extra=["-DCPDP_WITH_BDF"] + list(flags))
    oc._lib = _capi.CpdpLib(so)
    oc._mem = NumpyMem()
    return oc


def _run_configs(pend, quad, phases=3):
    """Mode-1 (BDF) runs of the pendulum (test_emu_kernels' configuration) and of the quadrotor on its stored run (N = 25)."""
    out = {}
    pend.setIntegrator(n_grid=10)
    pend.aux_mode = pend.MODE_BDF
    pend.rtol_back, pend.atol_back, pend.rtol_fwd, pend.atol_fwd = 1e-3, 1e-6, 1e-3, 1e-6
    th = np.array([1.0, 0.5, 1.5])
    sol = pend.cocSolverBatch(np.zeros((1, 2)), 1.0, th)
    out["pend"] = pend.auxSysSolverBatch(sol, phases=phases)
    g = np.load(os.path.join(HERE, "golden", "quad_run.npz"))
    quad.setIntegrator(n_grid=25)
    quad.aux_mode = quad.MODE_BDF
    quad.rtol_back, quad.atol_back, quad.rtol_fwd, quad.atol_fwd = 1e-3, 1e-6, 1e-3, 1e-6
    P = g["parameter_trace"]
    sol = quad.cocSolverBatch(g["ini_state"].reshape(1, 13), 1.0, P[0], pdata=g["goal_position"].reshape(1, 3))
    out["quad"] = quad.auxSysSolverBatch(sol, g["time_grid"], g["waypoints"].reshape(1, -1, 3), [0, 1, 2], phases=phases)
    return out


KEYS = ("Xa", "Ua", "loss", "dtheta", "aux_status", "counters")


@pytest.fixture(scope="module")
def default_run():
    return _run_configs(_emu("pendulum"), _emu("quadrotor"))


def test_eig_off_reproduces_sweep_solver_bitwise():
    got = _run_configs(_emu("pendulum", ["-DCPDP_BDF_EIG_KAPPA=0"]), _emu("quadrotor", ["-DCPDP_BDF_EIG_KAPPA=0"]))
    ref = np.load(GOLDEN)
    for cfg, o in got.items():
        for k in KEYS:
            assert np.array_equal(np.asarray(o[k]), ref["%s_%s" % (cfg, k)]), (cfg, k)


def test_default_matches_sweep_solver(default_run):
    """Same step / LU / Jacobian counters as the sweep solver (and so as scipy, test_emu_kernels); the sensitivities
    agree far inside the oracle tolerances (1e-8 there)."""
    ref = np.load(GOLDEN)
    for cfg, o in default_run.items():
        assert np.array_equal(np.asarray(o["aux_status"]), ref[cfg + "_aux_status"])
        assert np.array_equal(np.asarray(o["counters"]), ref[cfg + "_counters"]), cfg
        for k in ("Xa", "Ua", "loss", "dtheta"):
            a, b = np.asarray(o[k]), ref["%s_%s" % (cfg, k)]
            assert np.linalg.norm(a - b) <= 1e-10 * np.linalg.norm(b), (cfg, k)


def test_path_counts():
    """Most Jacobians take the eigen path; the quadrotor's terminal node (L defective: integrator chains) falls back."""
    got = _run_configs(_emu("pendulum", ["-DCPDP_BDF_PATH_COUNTS"]), _emu("quadrotor", ["-DCPDP_BDF_PATH_COUNTS"]), phases=1)
    for cfg, o in got.items():
        solves_eig, solves_sweep, jac_eig, jac_sweep = np.asarray(o["Ua"]).reshape(-1)[24:28]
        cnt = np.asarray(o["counters"])[0]
        assert jac_eig + jac_sweep == cnt[5]
        assert solves_eig + solves_sweep == cnt[0] - 2 * (10 if cfg == "pend" else 25)     # (two rhs per interval start it)
        assert jac_eig >= 0.8 * cnt[5], (cfg, jac_eig, jac_sweep)
        if cfg == "quad":
            assert jac_sweep >= 1
