"""Driver of tests/test_discrete_grad.py::test_discrete_kernels_are_race_free: one small problem through the discrete auxiliary
mode of the thread-emulated library built with -fsanitize=thread (run with libtsan preloaded).  TEST INFRASTRUCTURE."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tests.emu.support import emu_oc  # noqa: E402

name = sys.argv[1]
oc = emu_oc(name, tsan=True)
if name == "pendulum":
    th = np.array([1.0, 0.5, 1.5]); taus = np.array([0.4]); wp = np.array([[[1.0]]]); sel = [0]
    sol = oc.cocSolverBatch(np.zeros((1, 2)), 1.0, th)
else:
    from lfsd_b200 import synthetic
    qb = synthetic.quad_batch(1); oc.setIntegrator(n_grid=4)
    sol = oc.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"]); taus, wp, sel = qb["taus"], qb["wp"], qb["sel"]
aux = oc.auxSysSolverBatch(sol, taus, wp, sel, mode=oc.MODE_DISCRETE)
print(name, "discrete", "status", aux["aux_status"], "dtheta", aux["dtheta"][0])
