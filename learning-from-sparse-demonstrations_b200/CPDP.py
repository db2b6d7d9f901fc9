"""COCSys — host API of the B200 CPDP path, mirroring the reference class of the same name
(``/root/reference/CPDP/CPDP.py:9-390``): the same setters, ``cocSolver``, ``diffPMP``, ``raccatiODE``,
``auxSysODE``, ``auxSysSolver`` and ``interpolation`` with the same argument meaning and return types, plus
batched variants (``cocSolverBatch``, ``auxSysSolverBatch``, ``gradIterBatch``) that are the reason this package
exists.  Expressions are sympy-backed ``sx.SX`` objects; on first use they are lowered to CUDA device functions
(``codegen.py``), compiled into ``lib/libcpdp_<name>.so`` and driven through the C ABI of ``include/cpdp.h``.

There is no CPU fallback: every numerical method needs a CUDA device and the compiled extension and raises
otherwise.
"""
import numpy
import scipy.interpolate as ip

from . import sx
from .sx import SX, jacobian
from . import codegen
from . import _capi

__all__ = ["COCSys", "COCSys_TimeVarying"]


class _TorchCuda:
    """Device-memory provider: torch is only plumbing (allocation, streams), not the compute path."""

    def __init__(self, device=None):
        import torch
        if not torch.cuda.is_available():
            raise _capi.CpdpError("lfsd_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)

    def empty(self, shape, dtype="f8"):
        t = self.torch
        return t.empty(shape, dtype={"f8": t.float64, "i4": t.int32, "u1": t.uint8}[dtype], device=self.device)

    def zeros(self, shape, dtype="f8"):
        t = self.torch
        return t.zeros(shape, dtype={"f8": t.float64, "i4": t.int32, "u1": t.uint8}[dtype], device=self.device)

    def from_host(self, a, dtype="f8"):
        t = self.torch
        if isinstance(a, t.Tensor):
            return a.to(device=self.device, dtype={"f8": t.float64, "i4": t.int32}[dtype]).contiguous()
        arr = numpy.ascontiguousarray(numpy.asarray(a, dtype={"f8": numpy.float64, "i4": numpy.int32}[dtype]))
        return t.from_numpy(arr).to(self.device, non_blocking=True)

    def to_host(self, x):
        return x.detach().cpu().numpy()

    def ptr(self, x):
        return 0 if x is None else x.data_ptr()

    def stream(self):
        return self.torch.cuda.current_stream(self.device).cuda_stream


class _Interp:
    """scipy interp1d over a node table that also remembers the exact nodes (CPDP.py:384-390)."""

    def __init__(self, x, y, method=1):
        self.time_grid = numpy.asarray(x, dtype=float)
        self.nodes = numpy.asarray(y, dtype=float)
        self.method = method
        self._f = ip.interp1d(self.time_grid, self.nodes, axis=0) if method == 1 else \
            ip.interp1d(self.time_grid, self.nodes, axis=0, kind='cubic')

    def __call__(self, t):
        return self._f(t)


class COCSys:
    """Time-invariant continuous optimal-control system with learnable parameters."""

    # modes of the backward Riccati sweep
    MODE_RK45 = 0     # explicit Dormand-Prince with tolerance knobs (what COCSys_TimeVarying uses, CPDP.py:740)
    MODE_BDF = 1      # scheme of the as-shipped COCSys (CPDP.py:335): scipy-style BDF at default tolerances
    MODE_DISCRETE = 2  # exact derivative of the discretised problem the solver solves (DESIGN.md §3.7); tolerances unused
    # barrier parameter a warm start of a bounded model begins with (mu_init of cocSolverBatch; DESIGN.md §3.10)
    WARM_MU_INIT = 1e-8

    def __init__(self, project_name="myOc"):
        self.sys_name = project_name
        self._lib = None
        self._mem = None
        self._ws = None
        self._ws_key = None
        self.pvar = SX(sx.sp.zeros(0, 1))
        self.n_pvar = 0
        # solver settings of the batched Newton-KKT method
        self.tol = 1e-10
        self.max_iter = 200
        self.aux_mode = COCSys.MODE_BDF
        self.rtol_back, self.atol_back = 1e-3, 1e-6      # scipy defaults (bdf.py:198, rk.py:85)
        self.rtol_fwd, self.atol_fwd = 1e-3, 1e-6
        self.warm_mu_init = COCSys.WARM_MU_INIT

    # ------------------------------------------------------------------ problem definition
    def setAuxvarVariable(self, auxvar=None):
        """CPDP.py:15-17"""
        self.auxvar = SX.sym('auxvar', 1) if auxvar is None else auxvar
        self.n_auxvar = self.auxvar.numel()
        self._lib = None

    def setStateVariable(self, state, state_lb=[], state_ub=[]):
        """CPDP.py:20-31.  Bounds of the wrong length mean "none" (+-1e20), as in the reference; finite bounds are compiled
        into the model and enforced by the solver's barrier method (DESIGN.md §3.8).  A bound entry may also be an SX / sympy
        expression of the problem variables (setProblemVariable): each problem of a batch then has its own bound, evaluated at its
        pdata (DESIGN.md §3.12)."""
        self.state = state
        self.n_state = self.state.numel()
        self.state_lb, self.state_ub = self._check_bounds(state_lb, state_ub, self.n_state)
        self._lib = None

    def setControlVariable(self, control, control_lb=[], control_ub=[]):
        """CPDP.py:34-46"""
        self.control = control
        self.n_control = self.control.numel()
        self.control_lb, self.control_ub = self._check_bounds(control_lb, control_ub, self.n_control)
        self._lib = None

    @staticmethod
    def _check_bounds(lb, ub, n):
        lb, ub = codegen.normalize_bounds(codegen.bound_entries(lb), codegen.bound_entries(ub), n)
        for i, (lo, hi) in enumerate(zip(lb, ub)):
            if codegen.is_symbolic(lo) or codegen.is_symbolic(hi):
                continue                    # checked per problem at run time: lb(pdata) >= ub(pdata) gives CPDP_INFEASIBLE
            if not lo < hi:
                raise ValueError("bound %d: lower bound %r is not below upper bound %r (fixed variables are not supported)"
                                 % (i, lo, hi))
        return lb, ub

    def _bounds(self):
        return (self.state_lb, self.state_ub, self.control_lb, self.control_ub)

    @property
    def bounded(self):
        """True when some state or control bound is finite or an expression of the problem variables."""
        return any(codegen.is_symbolic(v) or abs(v) < 1e19 for v in self.state_lb + self.state_ub + self.control_lb + self.control_ub)

    @property
    def bounds_depend_on_pdata(self):
        """True when some bound is an expression of the problem variables (its value differs per problem)."""
        return codegen.bounds_symbolic(self._bounds())

    def boundsBatch(self, pdata=None):
        """Evaluated bounds of a batch: device arrays (lb, ub) of shape [B, n+m] (states then controls; +-1e20 for none) at
        pdata [B, q] (cpdp_eval_bounds).  For bounds that do not depend on pdata, B is pdata's row count, or 1 without pdata."""
        lib = self.build()
        mem = self._device()
        pd = None
        if pdata is not None:
            pd = mem.from_host(numpy.asarray(pdata, dtype=float).reshape(-1, self.n_pvar) if not hasattr(pdata, 'data_ptr')
                               else pdata)
        elif self.bounds_depend_on_pdata:
            raise ValueError("the bounds depend on the problem variables: pass pdata [B,%d]" % self.n_pvar)
        B = int(pd.shape[0]) if pd is not None else 1
        nz = self.n_state + self.n_control
        lb, ub = mem.empty((B, nz)), mem.empty((B, nz))
        lib.eval_bounds(mem.ptr(pd), B, mem.ptr(lb), mem.ptr(ub), mem.stream())
        return lb, ub

    def setProblemVariable(self, pvar):
        """Extension: symbols that are per-problem constants (e.g. a goal position) — not learnable, not states.
        They let one compiled model serve a batch of different OCPs (BASELINE config 5)."""
        self.pvar = pvar
        self.n_pvar = pvar.numel()
        self._lib = None

    def setDyn(self, ode):
        """CPDP.py:49-57"""
        if not hasattr(self, 'auxvar'):
            self.setAuxvarVariable()
        self.dyn = ode
        self.dfx = jacobian(self.dyn, self.state)
        self.dfu = jacobian(self.dyn, self.control)
        self._lib = None

    def setPathCost(self, path_cost):
        """CPDP.py:60-69"""
        if not hasattr(self, 'auxvar'):
            self.setAuxvarVariable()
        self.path_cost = path_cost
        self.dcx = jacobian(self.path_cost, self.state)
        self.dcu = jacobian(self.path_cost, self.control)
        self._lib = None

    def setFinalCost(self, final_cost):
        """CPDP.py:72-79"""
        if not hasattr(self, 'auxvar'):
            self.setAuxvarVariable()
        self.final_cost = final_cost
        self.dhx = jacobian(self.final_cost, self.state)
        self._lib = None

    def setIntegrator(self, n_grid=10, steps_per_grid=4):
        """CPDP.py:83-87"""
        self.n_grid = int(n_grid)
        self.steps_per_grid = int(steps_per_grid)

    def _assert_defined(self):
        assert hasattr(self, 'state'), "Define the state variable first!"
        assert hasattr(self, 'control'), "Define the control variable first!"
        assert hasattr(self, 'dyn'), "Define the system dynamics first!"
        assert hasattr(self, 'path_cost'), "Define the running cost/reward function first!"
        assert hasattr(self, 'final_cost'), "Define the final cost/reward function first!"

    # ------------------------------------------------------------------ symbolic differentiation (CPDP.py:201-248)
    def diffPMP(self):
        self._assert_defined()
        self.dfx = jacobian(self.dyn, self.state)
        self.dfu = jacobian(self.dyn, self.control)
        self.dfe = jacobian(self.dyn, self.auxvar)
        self.costate = SX.sym('lambda', self.n_state)
        self.path_Hamil = self.path_cost + (self.dyn.T) @ self.costate
        self.final_hamil = self.final_cost
        self.dHx = jacobian(self.path_Hamil, self.state).T
        self.dHu = jacobian(self.path_Hamil, self.control).T
        self.ddHxx = jacobian(self.dHx, self.state)
        self.ddHxu = jacobian(self.dHx, self.control)
        self.ddHxe = jacobian(self.dHx, self.auxvar)
        self.ddHux = jacobian(self.dHu, self.state)
        self.ddHuu = jacobian(self.dHu, self.control)
        self.ddHue = jacobian(self.dHu, self.auxvar)
        self.dhx = jacobian(self.final_hamil, self.state).T
        self.ddhxx = jacobian(self.dhx, self.state)
        self.ddhxe = jacobian(self.dhx, self.auxvar)

    def raccatiODE(self):
        """CPDP.py:253-276.  The Riccati right-hand side lives in the compiled kernels (csrc/cpdp_bdf.cuh,
        ``bdf_rhs_cols``); this only makes sure the model is compiled."""
        self.build()

    def auxSysODE(self):
        """CPDP.py:281-298 (kernel: ``fw_rhs``, csrc/cpdp_fwd.cuh)."""
        self.build()

    # ------------------------------------------------------------------ compilation
    def build(self, name=None, force=False, verbose=False):
        """Generate + compile the CUDA library of this model (cached by content hash) and load it."""
        self._assert_defined()
        if self._lib is not None and not force:
            return self._lib
        text, info = codegen.generate_model_header(name or self.sys_name, self.state, self.control, self.auxvar,
                                                    self.dyn, self.path_cost, self.final_cost, self.pvar,
                                                    time=getattr(self, 'time', None), bounds=self._bounds())
        self.codegen_info = info
        pd_text, _ = codegen.generate_pdata_header(name or self.sys_name, self.state, self.control, self.auxvar, self.dyn,
                                                   self.path_cost, self.final_cost, self.pvar, time=getattr(self, 'time', None),
                                                   bounds=self._bounds())
        libname = name if name is not None else "m" + info["hash"]
        so = _capi.build_model_library(libname, text, force=force, verbose=verbose, pd_header_text=pd_text)
        self._lib = _capi.CpdpLib(so)
        assert (self._lib.n, self._lib.m, self._lib.r, self._lib.q) == \
            (self.n_state, self.n_control, self.n_auxvar, self.n_pvar)
        # (an entry that depends on pdata reads NaN in the library)
        sym = lambda v: float("nan") if codegen.is_symbolic(v) else v
        assert (self._lib.has_bounds, self._lib.bounds_pd) == (self.bounded, self.bounds_depend_on_pdata)
        assert numpy.array_equal(self._lib.lb, [sym(v) for v in self.state_lb + self.control_lb], equal_nan=True) and \
            numpy.array_equal(self._lib.ub, [sym(v) for v in self.state_ub + self.control_ub], equal_nan=True)
        return self._lib

    def _device(self):
        if self._mem is None:
            self._mem = _TorchCuda()
        return self._mem

    def _workspace(self, B, slot=0):
        """Scratch for (B, n_grid, steps_per_grid); `slot` > 0 gives the independent workspaces that chunks running
        concurrently on different streams need (gradIterBatch(chunks=...))."""
        lib = self.build()
        key = (B, self.n_grid, self.steps_per_grid)
        if slot == 0:
            if self._ws_key != key:
                nbytes = lib.workspace_bytes(*key)
                self._ws = self._device().empty((nbytes,), "u1")
                self._ws_key = key
                self._ws_bytes = nbytes
            return self._ws
        pool = self.__dict__.setdefault("_ws_pool", {})
        if pool.get(slot, (None, None))[0] != key:
            nbytes = lib.workspace_bytes(*key)
            pool[slot] = (key, self._device().empty((nbytes,), "u1"))
            self._ws_bytes = nbytes
        return pool[slot][1]

    # ------------------------------------------------------------------ batched path
    def _theta_arg(self, auxvar_value, B):
        """auxvar_value [r] (shared by the batch, stride 0) or [B,r] -> (device array, stride)."""
        mem = self._device()
        th = auxvar_value if hasattr(auxvar_value, 'data_ptr') else \
            numpy.atleast_1d(numpy.asarray(auxvar_value, dtype=float))
        if th.ndim == 1:
            assert th.shape[0] == self.n_auxvar, "auxvar_value has %d entries, expected %d" % (th.shape[0], self.n_auxvar)
            return mem.from_host(th.reshape(1, -1)), 0
        assert tuple(th.shape) == (B, self.n_auxvar)
        return mem.from_host(th), self.n_auxvar

    def cocSolverBatch(self, ini_states, horizon, auxvar_value, pdata=None, rounds=0, init=None, shift=0, mu_init=None, _slot=0):
        """Batched cocSolver: ini_states [B,n]; auxvar_value [r] (shared) or [B,r]; pdata [B,q].
        Returns a dict of device arrays X [B,N+1,n], U [B,N+1,m], Lam [B,N+1,n], status, iters, kkt, cost
        and the host time_grid; a bounded model adds the bound multipliers Zl, Zu [B,N+1,n+m] (row N: the final state's) and
        the final barrier parameter mu [B].

        Warm start (DESIGN.md §3.10): ``init`` is a mapping with X, U, Lam and optionally Zl, Zu, status -- the dict this method
        returns qualifies -- and Newton starts from it instead of the zero seed (tensors are used detached).  Problems whose
        ``init["status"]`` is not `converged` start cold.  shift=1 starts row k from row k+1 of the guess (receding horizon).  A
        bounded model starts a warm problem's barrier parameter at ``mu_init`` (default ``warm_mu_init``; an ``init["mu"]`` is
        not used).  init=None is the cold solve."""
        self._assert_defined()
        if not hasattr(self, 'n_grid'):
            self.setIntegrator()
        lib = self.build()
        mem = self._device()
        x0 = mem.from_host(numpy.asarray(ini_states, dtype=float).reshape(-1, self.n_state)
                           if not hasattr(ini_states, 'data_ptr') else ini_states)
        B = int(x0.shape[0])
        N, S = self.n_grid, self.steps_per_grid
        th, th_stride = self._theta_arg(auxvar_value, B)
        pd = None
        if self.n_pvar > 0:
            assert pdata is not None, "this model has per-problem constants: pass pdata [B,%d]" % self.n_pvar
            pd = mem.from_host(numpy.asarray(pdata, dtype=float).reshape(B, self.n_pvar)
                               if not hasattr(pdata, 'data_ptr') else pdata)
        ws = self._workspace(B, _slot)
        out = dict(X=mem.empty((B, N + 1, self.n_state)), U=mem.empty((B, N + 1, self.n_control)),
                   Lam=mem.empty((B, N + 1, self.n_state)), status=mem.empty((B,), "i4"), iters=mem.empty((B,), "i4"),
                   kkt=mem.empty((B,)), cost=mem.empty((B,)))
        args = (mem.ptr(ws), int(ws.shape[0]), B, N, S, float(horizon), mem.ptr(x0), mem.ptr(th), th_stride, mem.ptr(pd),
                float(self.tol), int(self.max_iter), int(rounds),
                mem.ptr(out["X"]), mem.ptr(out["U"]), mem.ptr(out["Lam"]), mem.ptr(out["status"]), mem.ptr(out["iters"]),
                mem.ptr(out["kkt"]), mem.ptr(out["cost"]), mem.stream())
        if init is None:
            lib.solve(*args)
        else:
            g = self._warm_guess(init, B, N)
            lib.solve_warm(*args, *(mem.ptr(g[k]) for k in ("X", "U", "Lam", "Zl", "Zu", "status")), int(shift),
                           float(self.warm_mu_init if mu_init is None else mu_init))
        if lib.has_bounds:
            nz = self.n_state + self.n_control
            out.update(Zl=mem.empty((B, N + 1, nz)), Zu=mem.empty((B, N + 1, nz)), mu=mem.empty((B,)))
            lib.get_bound_multipliers(mem.ptr(ws), int(ws.shape[0]), B, N, S, mem.ptr(out["Zl"]), mem.ptr(out["Zu"]),
                                      mem.ptr(out["mu"]), mem.stream())
        out.update(time_grid=self._time_grid(horizon, N), horizon=float(horizon),
                   theta=th, theta_stride=th_stride, pdata=pd, B=B, x0=x0, _slot=_slot)
        return out

    def _warm_guess(self, init, B, N):
        """Device arrays of a warm-start mapping (shapes checked; tensors detached)."""
        mem = self._device()
        nz = self.n_state + self.n_control
        shapes = dict(X=(B, N + 1, self.n_state), U=(B, N + 1, self.n_control), Lam=(B, N + 1, self.n_state),
                      Zl=(B, N + 1, nz), Zu=(B, N + 1, nz), status=(B,))
        g = {}
        for k, shp in shapes.items():
            v = init.get(k) if k in ("Zl", "Zu", "status") else init[k]
            if v is None or (k in ("Zl", "Zu") and not self._lib.has_bounds):
                g[k] = None
                continue
            v = v.detach() if hasattr(v, "detach") else numpy.asarray(v)
            v = mem.from_host(v, "i4" if k == "status" else "f8")
            if tuple(v.shape) != shp:
                raise ValueError("init[%r] has shape %s, expected %s" % (k, tuple(v.shape), shp))
            g[k] = v
        if (g["Zl"] is None) != (g["Zu"] is None):
            raise ValueError("init needs both Zl and Zu, or neither")
        return g

    @staticmethod
    def _time_grid(horizon, N):
        """CPDP.py:192"""
        return numpy.array([horizon / N * k for k in range(N + 1)])

    def auxSysSolverBatch(self, sol, taus=None, waypoints=None, sel=None, mode=None, phases=3, out=None):
        """Batched auxSysSolver (+ fused loss closure).  ``sol`` is the dict returned by cocSolverBatch.
        taus [W] or [B,W]; waypoints [B,W,D] (or [W,D] shared by B=1); sel = observed state indices.
        Returns dict with Xa [B,N+1,n*r], Ua [B,N+1,m*r], loss [B], dtheta [B,r], aux_status, counters.
        phases: 1 = backward Riccati sweep only, 2 = forward sweep + loss only (pass the dict of the phase-1 call
        as ``out``), 3 = both (default)."""
        lib = self.build()
        mem = self._device()
        B, N, S = sol["B"], self.n_grid, self.steps_per_grid
        n, m, r = self.n_state, self.n_control, self.n_auxvar
        mode = self.aux_mode if mode is None else mode
        W = D = 0
        tau_d = wp_d = None
        tau_stride = 0
        sel = list(sel) if sel is not None else []
        if taus is not None:
            t_h = numpy.asarray(taus, dtype=float) if not hasattr(taus, 'data_ptr') else taus
            if t_h.ndim == 1:
                t_h = t_h.reshape(1, -1)
            W = int(t_h.shape[1])
            assert t_h.shape[0] in (1, B)
            tau_stride = 0 if (t_h.shape[0] == 1 and B > 1) else W
            tau_d = mem.from_host(t_h)
            D = len(sel)
            wp_h = waypoints if hasattr(waypoints, 'data_ptr') else numpy.asarray(waypoints, dtype=float).reshape(B, W, D)
            wp_d = mem.from_host(wp_h)
        ws = self._workspace(B, sol.get("_slot", 0))
        if lib.has_bounds and int(mode) == COCSys.MODE_DISCRETE and phases & 1:
            self._set_bound_multipliers(sol, ws)
        if out is None:
            out = dict(Xa=mem.empty((B, N + 1, n * r)), Ua=mem.empty((B, N + 1, m * r)), loss=mem.empty((B,)),
                       dtheta=mem.empty((B, r)), aux_status=mem.zeros((B,), "i4"),
                       counters=mem.zeros((B, lib.ncounters), "i4"))
        lib.aux(mem.ptr(ws), int(ws.shape[0]), B, N, S, sol["horizon"], mem.ptr(sol["theta"]), sol["theta_stride"],
                mem.ptr(sol["pdata"]), mem.ptr(sol["X"]), mem.ptr(sol["U"]), mem.ptr(sol["Lam"]), mem.ptr(sol["status"]),
                int(mode), float(self.rtol_back), float(self.atol_back), float(self.rtol_fwd), float(self.atol_fwd),
                W, D, sel, mem.ptr(tau_d), tau_stride, mem.ptr(wp_d),
                mem.ptr(out["Xa"]), mem.ptr(out["Ua"]), mem.ptr(out["loss"]), mem.ptr(out["dtheta"]),
                mem.ptr(out["aux_status"]), mem.ptr(out["counters"]), mem.stream(), phases=phases)
        return out

    def _set_bound_multipliers(self, sol, ws):
        """Mode 2 differentiates the barrier-perturbed KKT system: it reads the bound multipliers from the workspace."""
        if sol.get("Zl") is None:
            raise ValueError("mode 2 on a bounded model needs the bound multipliers Zl, Zu, mu of the solution")
        mem = self._device()
        self._lib.set_bound_multipliers(mem.ptr(ws), int(ws.shape[0]), sol["B"], self.n_grid, self.steps_per_grid,
                                        mem.ptr(sol["Zl"]), mem.ptr(sol["Zu"]), mem.ptr(sol["mu"]), mem.stream())

    def _pdata_workspace(self, B, slot=0):
        """Scratch of the pdata adjoint (cpdp_pdata_workspace_bytes), allocated on first use per slot as _workspace's."""
        lib = self.build()
        key = (B, self.n_grid)
        pool = self.__dict__.setdefault("_pd_ws_pool", {})
        if pool.get(slot, (None, None))[0] != key:
            pool[slot] = (key, self._device().empty((lib.pdata_workspace_bytes(*key),), "u1"))
        return pool[slot][1]

    def auxSysAdjointBatch(self, sol, Xbar=None, Ubar=None, pdata_bar=False):
        """Adjoint of mode 2: the gradient of a loss l(X, U) of the trajectory with respect to theta and x0, from its cotangents
        Xbar = dl/dX [B,N+1,n] and Ubar = dl/dU [B,N+1,m] (either may be None, meaning zero), by one reverse sweep per problem
        (DESIGN.md §3.9).  ``sol`` is the dict returned by cocSolverBatch (or one shaped like it; a bounded model needs its
        Zl, Zu, mu).  Returns device arrays theta_bar [B,r] (per-problem rows, also for a theta shared by the batch), x0_bar
        [B,n] and aux_status [B] (as mode 2: 0 ok, 3 no usable trajectory, 4 Quu not positive definite).  Rows are zero for a
        problem with aux_status != 0 or whose solve did not end `converged`.

        pdata_bar=True also returns pdata_bar [B,q], the gradient with respect to the per-problem constants, from the same sweep
        with q more parameter columns (DESIGN.md §3.11); theta_bar and x0_bar are unchanged.  A model without per-problem
        constants raises ValueError."""
        if Xbar is None and Ubar is None:
            raise ValueError("auxSysAdjointBatch needs a cotangent Xbar or Ubar")
        if pdata_bar and self.n_pvar == 0:
            raise ValueError("pdata_bar=True needs a model with per-problem constants (setProblemVariable)")
        lib = self.build()
        mem = self._device()
        B, N, S = sol["B"], self.n_grid, self.steps_per_grid
        n, m, r = self.n_state, self.n_control, self.n_auxvar
        cot = []
        for v, w in ((Xbar, n), (Ubar, m)):
            if v is not None:
                v = mem.from_host(v if hasattr(v, 'data_ptr') else numpy.asarray(v, dtype=float))
                if tuple(v.shape) != (B, N + 1, w):
                    raise ValueError("cotangent of shape %s, expected %s" % (tuple(v.shape), (B, N + 1, w)))
            cot.append(v)
        ws = self._workspace(B, sol.get("_slot", 0))
        if lib.has_bounds:
            self._set_bound_multipliers(sol, ws)
        out = dict(theta_bar=mem.empty((B, r)), x0_bar=mem.empty((B, n)), aux_status=mem.zeros((B,), "i4"))
        if pdata_bar:
            pws = self._pdata_workspace(B, sol.get("_slot", 0))
            out["pdata_bar"] = mem.empty((B, self.n_pvar))
            lib.aux_adjoint_pd(mem.ptr(ws), int(ws.shape[0]), mem.ptr(pws), int(pws.shape[0]), B, N, S, sol["horizon"],
                               mem.ptr(sol["theta"]), sol["theta_stride"], mem.ptr(sol["pdata"]), mem.ptr(sol["X"]),
                               mem.ptr(sol["U"]), mem.ptr(sol["Lam"]), mem.ptr(sol.get("status")), mem.ptr(cot[0]),
                               mem.ptr(cot[1]), mem.ptr(out["theta_bar"]), mem.ptr(out["x0_bar"]), mem.ptr(out["pdata_bar"]),
                               mem.ptr(out["aux_status"]), mem.stream())
            return out
        lib.aux_adjoint(mem.ptr(ws), int(ws.shape[0]), B, N, S, sol["horizon"], mem.ptr(sol["theta"]), sol["theta_stride"],
                        mem.ptr(sol["pdata"]), mem.ptr(sol["X"]), mem.ptr(sol["U"]), mem.ptr(sol["Lam"]),
                        mem.ptr(sol.get("status")), mem.ptr(cot[0]), mem.ptr(cot[1]), mem.ptr(out["theta_bar"]),
                        mem.ptr(out["x0_bar"]), mem.ptr(out["aux_status"]), mem.stream())
        return out

    def fp64PeakProbe(self, blocks, iters):
        """Launches the library's DFMA throughput probe (bench.py roofline denominator); returns its flop count."""
        lib = self.build()
        mem = self._device()
        if not hasattr(self, '_sink'):
            self._sink = mem.zeros((8,))
        lib.dfma_probe(mem.ptr(self._sink), int(blocks), int(iters), mem.stream())
        return float(blocks) * 256 * 8 * iters * 2

    def reduceBatch(self, loss, dtheta):
        """Fixed-tree sum over problems: returns device array [1+r] = [sum loss | sum dL/dtheta]."""
        lib = self.build()
        mem = self._device()
        B = int(loss.shape[0])
        p2 = 1
        while p2 < B:
            p2 *= 2
        scratch = mem.empty((p2 * (self.n_auxvar + 1),))
        out = mem.empty((self.n_auxvar + 1,))
        lib.reduce(mem.ptr(loss), mem.ptr(dtheta), B, mem.ptr(scratch), mem.ptr(out), mem.stream())
        return out

    def packRows(self, sol, aux):
        """Device rows [B, r+2] = [loss | dL/dtheta | bad] (bad = 1: forward solve not converged or a sweep failed); the
        unit of the cross-GPU all-gather."""
        lib = self.build()
        mem = self._device()
        B = int(aux["loss"].shape[0])
        rows = mem.empty((B, self.n_auxvar + 2))
        lib.pack_rows(mem.ptr(aux["loss"]), mem.ptr(aux["dtheta"]), mem.ptr(sol.get("status")), mem.ptr(aux["aux_status"]), B,
                      mem.ptr(rows), mem.stream())
        return rows

    def reduceRows(self, rows):
        """Fixed-tree sum of packRows rows: device array [r+2] = [sum loss | sum dL/dtheta | number of failed OCPs]."""
        lib = self.build()
        mem = self._device()
        B, C = int(rows.shape[0]), int(rows.shape[1])
        p2 = 1
        while p2 < B:
            p2 *= 2
        scratch = mem.empty((p2 * C,))
        out = mem.empty((C,))
        lib.reduce_rows(mem.ptr(rows), B, C, mem.ptr(scratch), mem.ptr(out), mem.stream())
        return out

    def gradIterBatch(self, ini_states, horizon, auxvar_value, taus, waypoints, sel, pdata=None, mode=None, rounds=0,
                      chunks=1, init=None, shift=0):
        """One CPDP gradient iteration for a batch: forward solve, auxiliary system, loss and dL/dtheta, and their
        fixed-order sums.  Returns (sum_loss_and_grad [1+r] device array, sol dict, aux dict).  ``aux["n_failed"]`` is a
        one-element device array (no host synchronisation): the number of OCPs whose forward solve did not end `converged`
        (incl. still iterating after a fixed number of ``rounds``) or whose sweeps failed -- their rows may be zero, so a
        caller must not step on the sum when it is non-zero (``optim.cpdp_grad_fn`` raises).

        chunks > 1 (needs rounds > 0, i.e. no host synchronisation inside the solve): the batch is cut into that many
        contiguous chunks, each running solve -> backward sweep -> forward sweep on its own CUDA stream with its own
        workspace, so that the under-filled tails of one chunk's kernels (last Newton rounds, last wave of the sweeps)
        overlap the other chunk's work.  Per-problem results do not depend on the chunking and the reduction tree is
        over the whole batch, so the result is bit-identical to chunks=1 (measured: 288 -> 274 ms for 4096 OCPs).

        init, shift: warm start of the forward solve (cocSolverBatch); with chunks > 1 ``init`` is cut along the same bounds."""
        mem = self._device()
        if chunks <= 1 or not hasattr(mem, "torch"):
            sol = self.cocSolverBatch(ini_states, horizon, auxvar_value, pdata=pdata, rounds=rounds, init=init, shift=shift)
            aux = self.auxSysSolverBatch(sol, taus, waypoints, sel, mode=mode)
            full = self.reduceRows(self.packRows(sol, aux))
            aux["n_failed"] = full[1 + self.n_auxvar:]
            return full[:1 + self.n_auxvar], sol, aux
        assert rounds > 0, "chunks > 1 needs a fixed number of Newton rounds (rounds > 0): the adaptive mode blocks the host"
        torch = mem.torch
        x0 = mem.from_host(numpy.asarray(ini_states, dtype=float).reshape(-1, self.n_state)
                           if not hasattr(ini_states, 'data_ptr') else ini_states)
        B = int(x0.shape[0])
        th = auxvar_value if hasattr(auxvar_value, 'data_ptr') else numpy.atleast_1d(numpy.asarray(auxvar_value, dtype=float))
        th = mem.from_host(th) if th.ndim == 2 else th
        pd = None if pdata is None else mem.from_host(numpy.asarray(pdata, dtype=float).reshape(B, self.n_pvar)
                                                      if not hasattr(pdata, 'data_ptr') else pdata)
        t_h = taus if hasattr(taus, 'data_ptr') else numpy.asarray(taus, dtype=float)
        t_h = mem.from_host(t_h) if t_h.ndim == 2 else t_h
        wp = mem.from_host(waypoints if hasattr(waypoints, 'data_ptr') else
                           numpy.asarray(waypoints, dtype=float).reshape(B, -1, len(sel)))
        bounds = [(B * c) // chunks for c in range(chunks + 1)]
        streams = self.__dict__.setdefault("_streams", [])
        while len(streams) < chunks:
            streams.append(torch.cuda.Stream(device=mem.device))
        main = torch.cuda.current_stream(mem.device)
        sols, auxs = [], []
        for c in range(chunks):
            lo, hi = bounds[c], bounds[c + 1]
            st = streams[c]
            st.wait_stream(main)
            with torch.cuda.stream(st):
                ini = None if init is None else {k: v[lo:hi] for k, v in init.items()
                                                 if k in ("X", "U", "Lam", "Zl", "Zu", "status") and v is not None}
                sol = self.cocSolverBatch(x0[lo:hi], horizon, th[lo:hi] if th.ndim == 2 else th,
                                          pdata=None if pd is None else pd[lo:hi], rounds=rounds, init=ini, shift=shift,
                                          _slot=c + 1)
                aux = self.auxSysSolverBatch(sol, t_h[lo:hi] if t_h.ndim == 2 else t_h, wp[lo:hi], sel, mode=mode)
            sols.append(sol)
            auxs.append(aux)
        for st in streams[:chunks]:
            main.wait_stream(st)
        sol = {k: torch.cat([s_[k] for s_ in sols]) for k in ("X", "U", "Lam", "status", "iters", "kkt", "cost")
               + (("Zl", "Zu", "mu") if "Zl" in sols[0] else ())}
        sol.update(time_grid=sols[0]["time_grid"], horizon=float(horizon), B=B, chunks=sols)
        aux = {k: torch.cat([a_[k] for a_ in auxs]) for k in ("Xa", "Ua", "loss", "dtheta", "aux_status", "counters")}
        full = self.reduceRows(self.packRows(sol, aux))
        aux["n_failed"] = full[1 + self.n_auxvar:]
        return full[:1 + self.n_auxvar], sol, aux

    # ------------------------------------------------------------------ reference-shaped single-problem API
    def cocSolver(self, ini_state, horizon, auxvar_value=1, interplation_level=1, print_level=0):
        """CPDP.py:92-198: returns (time_grid, opt_sol) with opt_sol(t) -> [x | u | costate]."""
        self._assert_defined()
        if not hasattr(self, 'n_grid'):
            self.setIntegrator()
        if type(ini_state) is list:
            ini_state = numpy.array(ini_state).flatten()
        pd = getattr(self, 'pdata_value', None)
        sol = self.cocSolverBatch(numpy.asarray(ini_state, dtype=float).reshape(1, -1), horizon,
                                  numpy.atleast_1d(numpy.asarray(auxvar_value, dtype=float)), pdata=pd)
        mem = self._device()
        X, U, Lam = (mem.to_host(sol[k])[0] for k in ("X", "U", "Lam"))
        self.last_status = int(mem.to_host(sol["status"])[0])
        self.last_iters = int(mem.to_host(sol["iters"])[0])
        if print_level:
            print("cocSolver: status=%s iterations=%d kkt=%.3e cost=%.10g" % (
                _capi.STATUS_NAMES[self.last_status], self.last_iters,
                float(mem.to_host(sol["kkt"])[0]), float(mem.to_host(sol["cost"])[0])))
        time_grid = sol["time_grid"]
        opt_sol = self.interpolation(time_grid, numpy.concatenate((X, U, Lam), axis=1), interplation_level)
        opt_sol._batch = sol
        return time_grid, opt_sol

    def auxSysSolver(self, time_grid, opt_sol, auxvar_value=1):
        """CPDP.py:301-381: returns auxsys_sol(t) -> [vec(dx/dtheta) | vec(du/dtheta)]."""
        self._assert_defined()
        mem = self._device()
        n, m = self.n_state, self.n_control
        nodes = opt_sol.nodes if hasattr(opt_sol, 'nodes') else numpy.asarray(opt_sol(time_grid))
        time_grid = numpy.asarray(time_grid, dtype=float)
        N = time_grid.size - 1
        assert N == self.n_grid, "time_grid does not match setIntegrator(n_grid)"
        # the sweeps integrate the LINEAR interpolant of the node table on the uniform grid cocSolver returns (CPDP.py:192,386)
        if getattr(opt_sol, 'method', 1) != 1:
            raise NotImplementedError("auxSysSolver integrates the linear interpolant (interplation_level=1, the level every "
                                      "reference script uses); a cubic opt_sol is not supported")
        if not numpy.allclose(time_grid, numpy.linspace(0.0, time_grid[-1], N + 1), rtol=0, atol=1e-12 * max(1.0, abs(time_grid[-1]))):
            raise NotImplementedError("auxSysSolver needs the uniform time grid returned by cocSolver")
        th, th_stride = self._theta_arg(numpy.atleast_1d(numpy.asarray(auxvar_value, dtype=float)), 1)
        pd = getattr(self, 'pdata_value', None)
        sol = dict(B=1, horizon=float(time_grid[-1]), theta=th, theta_stride=th_stride,
                   pdata=None if pd is None else mem.from_host(numpy.asarray(pd, dtype=float).reshape(1, -1)),
                   X=mem.from_host(nodes[:, :n].reshape(1, N + 1, n)),
                   U=mem.from_host(nodes[:, n:n + m].reshape(1, N + 1, m)),
                   Lam=mem.from_host(nodes[:, n + m:].reshape(1, N + 1, n)), status=None)
        batch = getattr(opt_sol, '_batch', None)       # bound multipliers of the cocSolver call behind opt_sol (bounded models)
        if batch is not None and batch.get("Zl") is not None:
            sol.update(Zl=batch["Zl"], Zu=batch["Zu"], mu=batch["mu"])
        aux = self.auxSysSolverBatch(sol)
        self.last_aux_status = int(mem.to_host(aux["aux_status"])[0])
        self.last_aux_counters = mem.to_host(aux["counters"])[0]
        Xa, Ua = mem.to_host(aux["Xa"])[0], mem.to_host(aux["Ua"])[0]
        return self.interpolation(time_grid, numpy.concatenate((Xa, Ua), axis=1))

    def interpolation(self, x, y, method=1):
        """CPDP.py:384-390"""
        return _Interp(x, y, method)


class COCSys_TimeVarying(COCSys):
    """Time-varying continuous optimal-control system: dynamics, path cost and final cost may depend on the time ``t``
    explicitly (polynomial time-warping v(t) = beta1 + 2 beta2 t + ...), mirroring the reference class of the same name
    (``/root/reference/CPDP/CPDP.py:394-787``; driver ``Examples/pendulum_timewarping.py``).  Differences from COCSys, all the
    reference's own:
      * ``setTimeVariable`` (:434); every model function takes the time;
      * the RK4 interval map freezes ``t = t_k`` over the whole grid interval (:512-519, 554-555) and the grid is
        ``numpy.linspace(0, horizon, n_grid + 1)`` (:544);
      * the backward Riccati sweep is integrated by ``solve_ivp``'s default RK45, not BDF (:740) -> ``aux_mode = MODE_RK45``.
    The kernels are the same ones (``cpdp_solve`` / ``cpdp_aux``): the code generator emits the time as one more model
    constant that the kernels fill in per node / per stage time."""

    def __init__(self, project_name="myOc"):
        super().__init__(project_name)
        self.aux_mode = COCSys.MODE_RK45

    def setTimeVariable(self, t=None):
        """CPDP.py:434-435"""
        self.time = SX.sym('time', 1) if t is None else t
        self._lib = None

    def _ensure_time(self):
        if not hasattr(self, 'time'):
            self.setTimeVariable()

    def setDyn(self, ode):
        """CPDP.py:438-450"""
        self._ensure_time()
        super().setDyn(ode)

    def setPathCost(self, path_cost):
        """CPDP.py:453-466"""
        self._ensure_time()
        super().setPathCost(path_cost)

    def setFinalCost(self, final_cost):
        """CPDP.py:469-478"""
        self._ensure_time()
        super().setFinalCost(final_cost)

    @staticmethod
    def _time_grid(horizon, N):
        """CPDP.py:544"""
        return numpy.linspace(0, horizon, N + 1)
