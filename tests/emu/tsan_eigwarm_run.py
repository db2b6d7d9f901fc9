"""Driver of tests/test_bdf_eigwarm.py's race check: the quadrotor's stored run (N = 25) through the backward BDF sweep of the
thread-emulated library built with -fsanitize=thread and the path counts (run with libtsan preloaded).  TEST INFRASTRUCTURE."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lfsd_b200 import _capi, codegen, standard  # noqa: E402
from tests.emu.build_emu import build  # noqa: E402
from tests.emu.support import NumpyMem, _BUILD  # noqa: E402

oc = standard.STANDARD["quadrotor"]()
text, _ = codegen.generate_model_header("quadrotor", oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar)
os.makedirs(_BUILD, exist_ok=True)
src = "".join(open(os.path.join(_capi.CSRC, fn)).read() for fn in sorted(os.listdir(_capi.CSRC))
              if os.path.isfile(os.path.join(_capi.CSRC, fn)))
src += open(os.path.join(ROOT, "tests", "emu", "emu_lib.cpp")).read()
tag = hashlib.sha1((text + src + "tsan eigwarm").encode()).hexdigest()[:12]
hdr = os.path.join(_BUILD, "model_quadrotor_eigwarm_tsan_%s.cuh" % tag)
so = os.path.join(_BUILD, "libemu_quadrotor_eigwarm_tsan_%s.so" % tag)
if not os.path.exists(so):
    with open(hdr, "w") as f:
        f.write(text)
    build(hdr, so, tsan=True, ns="cpdp_emu_eigwarm_tsan", extra=["-DCPDP_WITH_BDF", "-DCPDP_BDF_PATH_COUNTS"])
oc._lib = _capi.CpdpLib(so)
oc._mem = NumpyMem()
g = np.load(os.path.join(ROOT, "tests", "golden", "quad_run.npz"))
oc.setIntegrator(n_grid=25)
oc.aux_mode = oc.MODE_BDF
oc.rtol_back, oc.atol_back, oc.rtol_fwd, oc.atol_fwd = 1e-3, 1e-6, 1e-3, 1e-6
sol = oc.cocSolverBatch(g["ini_state"].reshape(1, 13), 1.0, g["parameter_trace"][0], pdata=g["goal_position"].reshape(1, 3))
aux = oc.auxSysSolverBatch(sol, g["time_grid"], g["waypoints"].reshape(1, -1, 3), [0, 1, 2], phases=1)
paths = np.asarray(aux["Ua"]).reshape(-1)[24:30]
print("warm accepted %d rejected %d status %s" % (paths[4], paths[5], aux["aux_status"]))
