"""Driver of tests/test_warm.py's race check: the warm start of a small batch through the thread-emulated library built with
-fsanitize=thread (run with libtsan preloaded), shift 0 and 1, the guess and init_status in the output buffers.
TEST INFRASTRUCTURE."""
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tests.emu.support import emu_oc  # noqa: E402
from tests.emu.bounds_support import emu_bounded_oc  # noqa: E402

name = sys.argv[1]
oc = emu_bounded_oc(name, tsan=True) if name.endswith("_bounded") else emu_oc(name, tsan=True)
oc.setIntegrator(n_grid=4)
x0 = np.array([[0.0, 0.0], [0.1, -0.2]])
th = np.array([[1.0, 0.5, 1.5], [1.1, 0.4, 1.4]])
sol = oc.cocSolverBatch(x0, 1.0, th)
sol["status"][1] = 2                                        # one problem starts cold
ws = oc._workspace(2)
p = lambda a: 0 if a is None else a.ctypes.data
th2 = th * 1.01
for shift in (0, 1):
    rc = oc._lib.L.cpdp_solve_warm(p(ws), ws.shape[0], 2, 4, oc.steps_per_grid, 1.0, p(x0), p(th2), 3, 0, oc.tol, oc.max_iter, 0,
                                   p(sol["X"]), p(sol["U"]), p(sol["Lam"]), p(sol["status"]), p(sol["iters"]), p(sol["kkt"]),
                                   p(sol["cost"]), 0, p(sol["X"]), p(sol["U"]), p(sol["Lam"]), None, None, p(sol["status"]),
                                   shift, ctypes.c_double(1e-4))
    print(name, "warm run", shift, "rc", rc, "status", sol["status"], "iters", sol["iters"])
