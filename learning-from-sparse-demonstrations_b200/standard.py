"""The optimal-control systems of the reference's example scripts, built exactly as the scripts build them
(time-warping wrapper: dyn = beta*f, path = beta*c, final cost unscaled, theta = [beta; cost_auxvar]).
Each function returns a COCSys with a stable library name so that ``__graft_entry__.build()`` can prebuild it.
"""
import math

from . import JinEnv
from .CPDP import COCSys, COCSys_TimeVarying
from .sx import SX, vertcat


def _wrap(env, name, n_grid):
    """/root/reference/Examples/pendulum_groundtruth.py:21-30 (identical in every example)."""
    oc = COCSys(name)
    beta = SX.sym('beta')
    oc.setAuxvarVariable(vertcat(beta, env.cost_auxvar))
    oc.setStateVariable(env.X)
    oc.setControlVariable(env.U)
    oc.setDyn(beta * env.f)
    oc.setPathCost(beta * env.path_cost)
    oc.setFinalCost(env.final_cost)
    oc.setIntegrator(n_grid=n_grid)
    oc.env = env
    oc.lib_name = name
    return oc


def pendulum_oc(n_grid=10):
    """Examples/pendulum_groundtruth.py:16-18 ; observed: q (x[0])."""
    env = JinEnv.SinglePendulum()
    env.initDyn(l=1, m=1, damping_ratio=0.1)
    env.initCost(wu=.01)
    oc = _wrap(env, "pendulum", n_grid)
    oc.sel = [0]
    return oc


def robotarm_oc(n_grid=30):
    """Examples/robotarm_random.py:14-29 ; observed: q1, q2."""
    env = JinEnv.RobotArm()
    env.initDyn(l1=1, m1=1, l2=1, m2=1, g=0)
    env.initCost_Polynomial(wu=.5)
    oc = _wrap(env, "robotarm", n_grid)
    oc.sel = [0, 1]
    return oc


def cartpole_oc(n_grid=20):
    """JinEnv.CartPole (JinEnv.py:499-574) behind the same time-warping wrapper; no example script of the reference uses
    it, constants as in the upstream PDP examples (mc = mp = 0.5, l = 1, wu = 0.1); observed: x, q."""
    env = JinEnv.CartPole()
    env.initDyn(mc=0.5, mp=0.5, l=1)
    env.initCost(wu=0.1)
    oc = _wrap(env, "cartpole", n_grid)
    oc.sel = [0, 1]
    return oc


def rocket_oc(n_grid=15):
    """Examples/rocket_groundtruth.py:15-30 ; observed: position and quaternion."""
    env = JinEnv.Rocket()
    env.initDyn(Jx=1, Jy=1, Jz=1, mass=1, l=1)
    env.initCost2(wthrust=0.1)
    oc = _wrap(env, "rocket", n_grid)
    oc.sel = [0, 1, 2, 6, 7, 8, 9]
    return oc


def quadrotor_oc(n_grid=25, goal_position=None):
    """lib/QuadAlgorithm.py:74-104 with QuadPara(1,1,1, mass=1, l=1, c=0.02) (Examples/quad_example.py:26).
    With goal_position=None the goal position is per-problem data (3 constants), which is what the batched
    benchmark needs; a numeric goal is baked into the model like the reference does."""
    env = JinEnv.Quadrotor()
    env.initDyn(Jx=1.0, Jy=1.0, Jz=1.0, mass=1.0, l=1.0, c=0.02)
    goal = JinEnv.QuadStates()
    pvar = None
    if goal_position is None:
        pvar = vertcat(SX.sym('goal_x'), SX.sym('goal_y'), SX.sym('goal_z'))
        goal.position = pvar
        name = "quadrotor"
    else:
        goal.position = list(goal_position)
        name = "quadrotor_fixedgoal"
    env.initCost_Polynomial(goal, w_thrust=0.1)
    oc = _wrap(env, name, n_grid)
    if pvar is not None:
        oc.setProblemVariable(pvar)
    oc.sel = [0, 1, 2]
    return oc


def pendulum_timewarp_oc(n_grid=10, order=2):
    """Examples/pendulum_timewarping.py:15-56: COCSys_TimeVarying with the polynomial time-warping speed
    v(t) = beta1 + 2 beta2 t + ... of the given order (the script ships order 1 active and orders 2-4 commented out; order 2
    is the default here because it is the smallest one in which the time enters the model); observed: q."""
    env = JinEnv.SinglePendulum()
    env.initDyn(l=1, m=1, damping_ratio=0.1)
    env.initCost(wu=.01)
    name = "pendulum_tw%d" % order
    oc = COCSys_TimeVarying(name)
    oc.setStateVariable(env.X)
    oc.setControlVariable(env.U)
    t = SX.sym('t')
    oc.setTimeVariable(t)
    betas = [SX.sym('beta%d' % (i + 1)) for i in range(order)]
    oc.setAuxvarVariable(vertcat(*betas, env.cost_auxvar))
    v = betas[0]
    for i in range(1, order):
        v = v + (i + 1) * betas[i] * t ** i
    oc.setDyn(v * env.f)
    oc.setPathCost(v * env.path_cost)
    oc.setFinalCost(env.final_cost)
    oc.setIntegrator(n_grid=n_grid)
    oc.env = env
    oc.lib_name = name
    oc.sel = [0]
    return oc


# ---- the JinEnv cost definitions no example script uses (SURVEY.md 8f N4), behind the same wrapper ----------------------
def robotarm_wd_oc(n_grid=20):
    """RobotArm.initCost_WeightedDistance (JinEnv.py:239-285): theta = [beta, wq1, wq2, wdq1, wdq2]."""
    env = JinEnv.RobotArm()
    env.initDyn(l1=1, m1=1, l2=1, m2=1, g=0)
    env.initCost_WeightedDistance(wu=.5)
    oc = _wrap(env, "robotarm_wd", n_grid)
    oc.sel = [0, 1]
    return oc


def _quad_env():
    env = JinEnv.Quadrotor()
    env.initDyn(Jx=1.0, Jy=1.0, Jz=1.0, mass=1.0, l=1.0, c=0.02)
    goal = JinEnv.QuadStates()
    pvar = vertcat(SX.sym('goal_x'), SX.sym('goal_y'), SX.sym('goal_z'))
    goal.position = pvar
    return env, goal, pvar


def quadrotor_cost1_oc(n_grid=15):
    """Quadrotor.initCost (JinEnv.py:755-815): theta = [beta, wr, wv, wq, ww]; goal position per problem."""
    env, goal, pvar = _quad_env()
    env.initCost(goal, wthrust=0.1)
    oc = _wrap(env, "quadrotor_cost1", n_grid)
    oc.setProblemVariable(pvar)
    oc.sel = [0, 1, 2]
    return oc


def quadrotor_cost2_oc(n_grid=15):
    """Quadrotor.initCost2 (JinEnv.py:817-884): theta = [beta, wrx..wwz (9), wq]; goal position per problem."""
    env, goal, pvar = _quad_env()
    env.initCost2(goal, wthrust=0.1)
    oc = _wrap(env, "quadrotor_cost2", n_grid)
    oc.setProblemVariable(pvar)
    oc.sel = [0, 1, 2]
    return oc


def rocket_cost1_oc(n_grid=15):
    """Rocket.initCost (JinEnv.py:1328-1399): theta = [beta, wr, wv, wtilt, wsidethrust, ww].
    (Rocket.initCost_Ex, :1475-1551, puts the control-dependent side-thrust term into the FINAL cost: the reference's own
    setFinalCost builds a CasADi Function of (state, auxvar) only and rejects it; here codegen asserts the same.)"""
    env = JinEnv.Rocket()
    env.initDyn(Jx=1, Jy=1, Jz=1, mass=1, l=1)
    env.initCost(wthrust=0.1)
    oc = _wrap(env, "rocket_cost1", n_grid)
    oc.sel = [0, 1, 2, 6, 7, 8, 9]
    return oc


VARIANTS = {"robotarm_wd": robotarm_wd_oc, "quadrotor_cost1": quadrotor_cost1_oc, "quadrotor_cost2": quadrotor_cost2_oc,
            "rocket_cost1": rocket_cost1_oc}

# ---- box-bounded versions (actuator limits, one joint-speed limit) whose bounds are active at the fixtures' optima ----------
def pendulum_bounded_oc(n_grid=10):
    """pendulum_oc with the torque bounded, |u| <= 5 (the unbounded optimum of the fixture reaches 9.95)."""
    oc = pendulum_oc(n_grid)
    oc.setControlVariable(oc.env.U, [-5.0], [5.0])
    oc.lib_name = "pendulum_bounded"
    return oc


def robotarm_bounded_oc(n_grid=30):
    """robotarm_oc with |u_i| <= 3 and the state bound |dq2| <= 4 (unbounded optimum: torque -5.8, dq2 +-6.2)."""
    oc = robotarm_oc(n_grid)
    oc.setStateVariable(oc.env.X, [-1e20, -1e20, -1e20, -4.0], [1e20, 1e20, 1e20, 4.0])
    oc.setControlVariable(oc.env.U, [-3.0, -3.0], [3.0, 3.0])
    oc.lib_name = "robotarm_bounded"
    return oc


def quadrotor_bounded_oc(n_grid=25):
    """quadrotor_oc (goal position per problem) with the rotor thrusts bounded, 1 <= f_i <= 4 (unbounded: 0.54 - 5.88)."""
    oc = quadrotor_oc(n_grid)
    oc.setControlVariable(oc.env.U, [1.0] * 4, [4.0] * 4)
    oc.lib_name = "quadrotor_bounded"
    return oc


BOUNDED = {"pendulum_bounded": pendulum_bounded_oc, "robotarm_bounded": robotarm_bounded_oc,
           "quadrotor_bounded": quadrotor_bounded_oc}

# ---- the same limits as expressions of per-problem constants (DESIGN.md §3.12): one library serves every limit value ------------
def pendulum_pdbounded_oc(n_grid=10):
    """pendulum_bounded_oc with the torque limit per problem, |u| <= umax (pdata = [umax])."""
    oc = pendulum_oc(n_grid)
    umax = SX.sym('umax')
    oc.setProblemVariable(umax)
    oc.setControlVariable(oc.env.U, [-umax], [umax])
    oc.lib_name = "pendulum_pdbounded"
    return oc


def pendulum_pdbounded_ab_oc(n_grid=10):
    """pendulum_bounded_oc with nonlinear limits of two constants (pdata = [a, b]): -a (1 + b^2) <= u <= a + b^2, i.e. |u| <= 5 at
    a = 1, b = 2."""
    oc = pendulum_oc(n_grid)
    a, b = SX.sym('a'), SX.sym('b')
    oc.setProblemVariable(vertcat(a, b))
    oc.setControlVariable(oc.env.U, [-a * (1 + b ** 2)], [a + b ** 2])
    oc.lib_name = "pendulum_pdbounded_ab"
    return oc


def robotarm_pdbounded_oc(n_grid=30):
    """robotarm_bounded_oc with the joint-speed limit per problem, |dq2| <= vmax (pdata = [vmax]); |u_i| <= 3 stays constant."""
    oc = robotarm_oc(n_grid)
    vmax = SX.sym('vmax')
    oc.setProblemVariable(vmax)
    oc.setStateVariable(oc.env.X, [-1e20, -1e20, -1e20, -vmax], [1e20, 1e20, 1e20, vmax])
    oc.setControlVariable(oc.env.U, [-3.0, -3.0], [3.0, 3.0])
    oc.lib_name = "robotarm_pdbounded"
    return oc


def quadrotor_pdbounded_oc(n_grid=25):
    """quadrotor_bounded_oc with the thrust limit per problem, 1 <= f_i <= f_max (pdata = [goal position (3), f_max])."""
    oc = quadrotor_oc(n_grid)
    fmax = SX.sym('f_max')
    oc.setProblemVariable(vertcat(oc.pvar, fmax))
    oc.setControlVariable(oc.env.U, [1.0] * 4, [fmax] * 4)
    oc.lib_name = "quadrotor_pdbounded"
    return oc


# not part of build_all: built on first use
PD_BOUNDED = {"pendulum_pdbounded": pendulum_pdbounded_oc, "pendulum_pdbounded_ab": pendulum_pdbounded_ab_oc,
              "robotarm_pdbounded": robotarm_pdbounded_oc, "quadrotor_pdbounded": quadrotor_pdbounded_oc}

STANDARD = {"pendulum": pendulum_oc, "pendulum_tw2": pendulum_timewarp_oc, "robotarm": robotarm_oc, "rocket": rocket_oc, "quadrotor": quadrotor_oc,
            "cartpole": cartpole_oc}


def build_all(verbose=False):
    libs = {}
    for name, fn in list(STANDARD.items()) + list(VARIANTS.items()) + list(BOUNDED.items()):
        oc = fn()
        libs[name] = oc.build(name=oc.lib_name, verbose=verbose).path
    return libs
