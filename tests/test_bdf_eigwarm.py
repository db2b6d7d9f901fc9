"""CPU tests (thread emulation) of the warm start of k_riccati_bdf's eigen path (csrc/cpdp_bdf.cuh, bdf_eig_refine): a Jacobian
that follows one on the eigen path refines the previous eigenbasis by Newton steps on the similarity H L G and runs the Schur
form only when the refinement is rejected.

`tests/golden/bdf_eig_outputs.npz` holds the outputs of the solver before the warm start (eigen path from a Schur form at
every Jacobian, computed with test_bdf_eigsolve's `_run_configs` through its emulation).  A build with
-DCPDP_BDF_EIG_WARM=0, and a build whose acceptance test never passes, must reproduce them bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_bdf_eigsolve import KEYS, _emu, _run_configs

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_EIG = os.path.join(HERE, "golden", "bdf_eig_outputs.npz")
GOLDEN_SWEEP = os.path.join(HERE, "golden", "bdf_sweep_outputs.npz")


def _run(flags=()):
    return _run_configs(_emu("pendulum", list(flags)), _emu("quadrotor", list(flags)))


def _assert_bitwise(got, ref):
    for cfg, o in got.items():
        for k in KEYS:
            assert np.array_equal(np.asarray(o[k]), ref["%s_%s" % (cfg, k)]), (cfg, k)


@pytest.fixture(scope="module")
def default_run():
    return _run()


def test_warm_off_reproduces_previous_solver_bitwise():
    _assert_bitwise(_run(["-DCPDP_BDF_EIG_WARM=0"]), np.load(GOLDEN_EIG))


def test_rejected_refinement_reproduces_previous_solver_bitwise():
    """Tolerance 0: every refinement runs all its steps and is rejected; the Schur form that follows must not see it."""
    _assert_bitwise(_run(["-DCPDP_BDF_REFINE_TOL=0"]), np.load(GOLDEN_EIG))


@pytest.mark.parametrize("golden", [GOLDEN_EIG, GOLDEN_SWEEP], ids=["schur_eigen_path", "sweep_only"])
def test_default_matches_previous_solvers(default_run, golden):
    """Same counters, status and loss as the Schur-form eigen path and the sweep-only solver; Xa, Ua, dL/dtheta within 1e-10."""
    ref = np.load(golden)
    for cfg, o in default_run.items():
        for k in ("aux_status", "counters"):
            assert np.array_equal(np.asarray(o[k]), ref["%s_%s" % (cfg, k)]), (cfg, k)
        for k in ("Xa", "Ua", "loss", "dtheta"):
            a, b = np.asarray(o[k]), ref["%s_%s" % (cfg, k)]
            assert np.linalg.norm(a - b) <= 1e-10 * np.linalg.norm(b), (cfg, k)
    if golden == GOLDEN_EIG:
        for cfg, o in default_run.items():
            assert np.array_equal(np.asarray(o["loss"]), ref[cfg + "_loss"]), cfg


def test_warm_path_counts():
    """The refinement is accepted at most Jacobians after the first; every Jacobian is counted once on the eigen path or the
    sweep, as without it (test_bdf_eigsolve.test_path_counts)."""
    got = _run_configs(_emu("pendulum", ["-DCPDP_BDF_PATH_COUNTS"]), _emu("quadrotor", ["-DCPDP_BDF_PATH_COUNTS"]), phases=1)
    off = _run_configs(_emu("pendulum", ["-DCPDP_BDF_PATH_COUNTS", "-DCPDP_BDF_EIG_WARM=0"]),
                       _emu("quadrotor", ["-DCPDP_BDF_PATH_COUNTS", "-DCPDP_BDF_EIG_WARM=0"]), phases=1)
    for cfg, o in got.items():
        paths = np.asarray(o["Ua"]).reshape(-1)[24:30]
        paths_off = np.asarray(off[cfg]["Ua"]).reshape(-1)[24:30]
        jac_eig, jac_sweep, accepted, rejected = paths[2:6]
        assert np.array_equal(paths[:4], paths_off[:4]), (cfg, paths, paths_off)
        assert paths_off[4] == 0 and paths_off[5] == 0
        assert accepted > 0 and accepted + rejected <= jac_eig + jac_sweep - 1, (cfg, paths)
        assert accepted >= 0.5 * (jac_eig + jac_sweep - 1), (cfg, paths)


def test_emulated_warm_refinement_is_race_free():
    tsan = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not tsan or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="report_bugs=1 exitcode=0 halt_on_error=0")
    r = subprocess.run([sys.executable, os.path.join(HERE, "emu", "tsan_eigwarm_run.py")], capture_output=True, text=True,
                       env=env, timeout=1800)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-2000:]
    line = [ln for ln in out.splitlines() if ln.startswith("warm accepted")]
    assert line and int(line[0].split()[2]) > 0, out[-2000:]
    assert "WARNING: ThreadSanitizer" not in out, out[:4000]
