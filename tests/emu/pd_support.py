"""CPU-side support of the pdata-gradient tests: the thread-emulated kernel library (tests/emu/emu_lib.cpp) built WITH the companion
header of codegen.generate_pdata_header (-DCPDP_PD_HEADER), and small test models whose goal angle is a per-problem constant.
TEST INFRASTRUCTURE — the product never imports this."""
import hashlib
import os

import sympy as sp

import lfsd_b200  # noqa: F401
from lfsd_b200 import _capi, codegen
from lfsd_b200.CPDP import COCSys, COCSys_TimeVarying
from lfsd_b200.sx import SX, sin, vertcat
from oracle.models import OracleModel
from tests.emu.build_emu import build
from tests.emu.support import NumpyMem, _BUILD

_HERE = os.path.dirname(os.path.abspath(__file__))


def emu_pd_from(oc, name, tsan=False):
    """Binds COCSys `oc` to the host-emulated kernels of its generated header and pdata companion header; returns `oc`."""
    args = (oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost, oc.final_cost, oc.pvar)
    text, _ = codegen.generate_model_header(name, *args, time=getattr(oc, 'time', None), bounds=oc._bounds())
    pd_text, _ = codegen.generate_pdata_header(name, *args, time=getattr(oc, 'time', None))
    src = "".join(open(os.path.join(_capi.CSRC, f)).read() for f in sorted(os.listdir(_capi.CSRC))
                  if os.path.isfile(os.path.join(_capi.CSRC, f)))
    src += open(os.path.join(_HERE, "emu_lib.cpp")).read()
    tag = hashlib.sha1((text + pd_text + src + str(tsan)).encode()).hexdigest()[:12]
    os.makedirs(_BUILD, exist_ok=True)
    hdr = os.path.join(_BUILD, "model_%s_%s.cuh" % (name, tag))
    pd_hdr = os.path.join(_BUILD, "model_%s_%s_pd.cuh" % (name, tag))
    so = os.path.join(_BUILD, "libemupd_%s_%s.so" % (name, tag))
    if not os.path.exists(so):
        with open(hdr, "w") as f:
            f.write(text)
        with open(pd_hdr, "w") as f:
            f.write(pd_text)
        tmp = "%s.tmp%d" % (so, os.getpid())
        build(hdr, tmp, tsan=tsan, ns="cpdp_emupd_" + name, extra=["-DCPDP_WITH_BDF", "-DCPDP_PD_HEADER=\"%s\"" % pd_hdr])
        os.replace(tmp, so)
    oc._lib = _capi.CpdpLib(so)
    oc._mem = NumpyMem()
    return oc


def pendulum_goal_oc(n_grid=10, time_varying=False, through_theta=False):
    """The pendulum of standard.pendulum_oc (theta = [beta, wq, wdq]) with its goal angle g as a per-problem constant:
    h = wq (q - g)^2 + wdq dq^2, c = h + 0.01 u^2, dyn = v f, path = v c.  time_varying: COCSys_TimeVarying with
    v = beta + 2 beta2 t (theta = [beta, beta2, wq, wdq]); otherwise v = beta.  through_theta: the goal is theta_4 + g, so that g
    enters only through theta_4 + g (theta = [beta, wq, wdq, g0])."""
    q, dq, u, g = SX.sym('q'), SX.sym('dq'), SX.sym('u'), SX.sym('g')
    beta, wq, wdq = SX.sym('beta'), SX.sym('wq'), SX.sym('wdq')
    f = vertcat(dq, (u - 10 * sin(q) - 0.1 * dq) / (1.0 / 3))
    goal, th = g, [beta, wq, wdq]
    oc = COCSys_TimeVarying("pendulum_goal_tv") if time_varying else COCSys("pendulum_goal")
    v = beta
    if time_varying:
        t, beta2 = SX.sym('t'), SX.sym('beta2')
        oc.setTimeVariable(t)
        v = beta + 2 * beta2 * t
        th = [beta, beta2, wq, wdq]
    if through_theta:
        g0 = SX.sym('g0')
        goal = g0 + g
        th = th + [g0]
        oc.sys_name = "pendulum_goal_th"
    h = wq * (q - goal) ** 2 + wdq * dq ** 2
    c = h + 0.01 * u ** 2
    oc.setAuxvarVariable(vertcat(*th))
    oc.setStateVariable(vertcat(q, dq))
    oc.setControlVariable(u)
    oc.setProblemVariable(g)
    oc.setDyn(v * f)
    oc.setPathCost(v * c)
    oc.setFinalCost(h)
    oc.setIntegrator(n_grid=n_grid)
    return oc


def pendulum_goal_model(time_varying=False, through_theta=False):
    """OracleModel of pendulum_goal_oc (same symbols, sympy)."""
    q, dq, u, g = sp.symbols('q dq u g', real=True)
    beta, wq, wdq = sp.symbols('beta wq wdq', real=True)
    f = sp.Matrix([dq, (u - 10 * sp.sin(q) - sp.Rational(1, 10) * dq) * 3])
    goal, th, v, t = g, [beta, wq, wdq], beta, None
    if time_varying:
        t, beta2 = sp.symbols('t beta2', real=True)
        v = beta + 2 * beta2 * t
        th = [beta, beta2, wq, wdq]
    if through_theta:
        g0 = sp.Symbol('g0', real=True)
        goal = g0 + g
        th = th + [g0]
    h = wq * (q - goal) ** 2 + wdq * dq ** 2
    c = h + sp.Rational(1, 100) * u ** 2
    mdl = OracleModel('pendulum_goal', [q, dq], [u], th, v * f, v * c, h, sel=[0], pdata=[g])
    if time_varying:
        mdl.time = t
    return mdl

