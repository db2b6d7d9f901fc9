"""Parameter-update rules and the learning loop of the reference's quadrotor learner, the immediate caller of the
CPDP gradient iteration (SURVEY.md 8f, row N1).

Mirrors ``/root/reference/lib/QuadAlgorithm.py``:
  * ``load_optimization_function``  (:132-191)  same dictionary keys, same ``Exception("Wrong optimization method type!")``
  * state initialisation            (:106-130)
  * ``Vanilla_gradient_descent`` (:454-466), ``Nesterov`` (:469-494, incl. the optional second evaluation at the new
    point when ``true_loss_print_flag`` is set), ``Adam`` (:497-520), ``Nadam`` (:523-548), ``AMSGrad`` (:551-578)
  * the loop, its stop rule ``loss > 0.9 and |dL| > 0.05`` and the projection ``theta[0] = max(theta[0], 1e-8)`` (:239-257)

The r = len(theta) doubles of optimiser state are updated with exactly the reference's numpy expressions (so a run is
reproducible against the stored ``parameter_trace``); every loss / gradient evaluation goes through the CUDA path
(``COCSys.gradIterBatch``), one device-to-host read of 1 + r doubles per evaluation.
"""
import numpy as np


class Learner:
    """``grad_fn(theta) -> (loss, dL/dtheta)`` is the CPDP gradient iteration (summed over the batch of OCPs)."""

    def __init__(self, grad_fn, n_auxvar):
        self.grad_fn = grad_fn
        self.n_auxvar = int(n_auxvar)
        self.loss_trace = []
        self.parameter_trace = []

    # ------------------------------------------------------------------ QuadAlgorithm.py:132-191
    def load_optimization_function(self, para_input: dict):
        self.learning_rate = para_input["learning_rate"]
        self.iter_num = para_input["iter_num"]
        self.optimization_method_str = para_input["method"]
        m = para_input["method"]
        if m == "Vanilla":
            self.optimization_function = lambda theta, idx: self.Vanilla_gradient_descent(theta)
        elif m == "Nesterov":
            self.mu_momentum = para_input["mu"]
            self.actual_loss_print_nesterov_flag = para_input["true_loss_print_flag"]
            self.optimization_function = lambda theta, idx: self.Nesterov(theta)
        elif m in ("Adam", "Nadam", "AMSGrad"):
            self.beta_1 = para_input["beta_1"]
            self.beta_2 = para_input["beta_2"]
            self.epsilon = para_input["epsilon"]
            fn = {"Adam": self.Adam, "Nadam": self.Nadam, "AMSGrad": self.AMSGrad}[m]
            self.optimization_function = lambda theta, idx: fn(theta, idx)
        else:
            raise Exception("Wrong optimization method type!")
        # state (QuadAlgorithm.py:106-130): integer-zero arrays there, promoted to float by the first update
        z = np.array([0] * self.n_auxvar)
        self.velocity_Nesterov = z.copy()
        self.momentum_vector = z.copy()
        self.velocity_vector = z.copy()
        self.velocity_vector_hat = z.copy()

    # ------------------------------------------------------------------ update rules
    def Vanilla_gradient_descent(self, current_parameter):
        loss, diff_loss = self.grad_fn(current_parameter)
        current_parameter = current_parameter - self.learning_rate * np.array(diff_loss)
        return loss, diff_loss, current_parameter

    def Nesterov(self, current_parameter):
        parameter_momentum = current_parameter + self.mu_momentum * self.velocity_Nesterov
        loss, diff_loss = self.grad_fn(parameter_momentum)
        self.velocity_Nesterov = self.mu_momentum * self.velocity_Nesterov - self.learning_rate * np.array(diff_loss)
        current_parameter = current_parameter + self.velocity_Nesterov
        if self.actual_loss_print_nesterov_flag:
            loss, diff_loss = self.grad_fn(current_parameter)
        return loss, diff_loss, current_parameter

    def _moments(self, diff_loss):
        self.momentum_vector = self.beta_1 * self.momentum_vector + (1 - self.beta_1) * np.array(diff_loss)
        self.velocity_vector = self.beta_2 * self.velocity_vector + (1 - self.beta_2) * np.power(diff_loss, 2)

    def Adam(self, current_parameter, iter_idx_now: int):
        idx = iter_idx_now + 1
        loss, diff_loss = self.grad_fn(current_parameter)
        self._moments(diff_loss)
        m_hat = self.momentum_vector / (1 - np.power(self.beta_1, idx))
        v_hat = self.velocity_vector / (1 - np.power(self.beta_2, idx))
        current_parameter = current_parameter - self.learning_rate * m_hat / (np.sqrt(v_hat) + self.epsilon)
        return loss, diff_loss, current_parameter

    def Nadam(self, current_parameter, iter_idx_now: int):
        idx = iter_idx_now + 1
        loss, diff_loss = self.grad_fn(current_parameter)
        self._moments(diff_loss)
        m_hat = self.momentum_vector / (1 - np.power(self.beta_1, idx))
        v_hat = self.velocity_vector / (1 - np.power(self.beta_2, idx))
        current_parameter = current_parameter - self.learning_rate * \
            (self.beta_1 * m_hat + ((1 - self.beta_1) / (1 - np.power(self.beta_1, idx))) * np.array(diff_loss)) \
            / (np.sqrt(v_hat) + self.epsilon)
        return loss, diff_loss, current_parameter

    def AMSGrad(self, current_parameter, iter_idx_now: int):
        loss, diff_loss = self.grad_fn(current_parameter)
        self._moments(diff_loss)
        self.velocity_vector_hat = np.maximum(self.velocity_vector_hat, self.velocity_vector)
        current_parameter = current_parameter - self.learning_rate * self.momentum_vector \
            / (np.sqrt(self.velocity_vector_hat) + self.epsilon)
        return loss, diff_loss, current_parameter

    # ------------------------------------------------------------------ QuadAlgorithm.py:231-257
    def run(self, initial_parameter, print_flag=False, max_iter=None):
        self.loss_trace = []
        self.parameter_trace = []
        current_parameter = np.array(initial_parameter, dtype=float)
        self.parameter_trace.append(current_parameter.tolist())
        loss = 100
        diff_loss_norm = 100
        n = self.iter_num if max_iter is None else min(self.iter_num, max_iter)
        for j in range(n):
            if (loss > 0.9) and (diff_loss_norm > 0.05):
                loss, diff_loss, current_parameter = self.optimization_function(current_parameter, j)
                self.loss_trace.append(loss)
                diff_loss_norm = np.linalg.norm(diff_loss)
                current_parameter[0] = max(current_parameter[0], 1e-8)          # projection step
                self.parameter_trace.append(current_parameter.tolist())
                if print_flag:
                    print('iter:', j, ', loss:', self.loss_trace[-1], ', loss gradient norm:', diff_loss_norm)
            else:
                if print_flag:
                    print("The loss is less than threshold, stop the iteration.")
                break
        return current_parameter


def cpdp_grad_fn(oc, ini_states, horizon, taus, waypoints, sel, pdata=None, mode=None):
    """grad_fn for ``Learner`` backed by the CUDA path: theta -> (sum of losses, sum of dL/dtheta) over the batch of OCPs
    (one forward solve + auxiliary system + loss per OCP, fixed-tree reduction; COCSys.gradIterBatch)."""
    mem = oc._device()

    def fn(theta):
        red, sol, aux = oc.gradIterBatch(ini_states, horizon, np.asarray(theta, dtype=float), taus, waypoints, sel,
                                         pdata=pdata, mode=mode)
        v = np.asarray(mem.to_host(red), dtype=float)
        n_failed = int(round(float(np.asarray(mem.to_host(aux["n_failed"]))[0])))
        if n_failed:
            st = np.asarray(mem.to_host(sol["status"]))
            ast = np.asarray(mem.to_host(aux["aux_status"]))
            raise FloatingPointError("CPDP gradient iteration failed for %d OCP(s): forward solve not converged for %d, "
                                     "auxiliary sweep failed for %d (the reference would step on garbage or crash in "
                                     "solve_ivp here)" % (n_failed, int((st != 1).sum()), int((ast != 0).sum())))
        return float(v[0]), v[1:].copy()
    return fn


METHOD_IDS = {"Vanilla": 0, "Nesterov": 1, "Adam": 2, "Nadam": 3, "AMSGrad": 4}


class DeviceLearner:
    """The same learner with the whole loop on the GPU: evaluation point, CPDP gradient iteration, update, projection, stop
    rule and traces are kernel launches on one stream (``cpdp_optim_step`` around ``COCSys.gradIterBatch``), nothing returns
    to the host until ``run`` reads the traces at the end.  Same dictionary keys as ``Learner`` /
    ``QuadAlgorithm.load_optimization_function`` (lib/QuadAlgorithm.py:132-191).  The per-iteration failure count of the
    gradient iteration is accumulated on the device and checked once after the run.

    Difference from the reference, stated: once the stop rule fires the remaining launches of the run are no-ops on the
    parameter (the stream cannot `break`); ``check_every`` > 0 makes the host poll the stop flag every that many iterations
    and leave early.

    warm_start=True: every evaluation after the first starts its forward solve from the previous evaluation's solution (kept on
    the device; with Nesterov's second evaluation, the last solve of either kind), and a problem whose previous solve did not
    converge starts cold (``COCSys.cocSolverBatch(init=...)``, DESIGN.md §3.10)."""

    def __init__(self, oc, ini_states, horizon, taus, waypoints, sel, pdata=None, mode=None, rounds=0, chunks=1, warm_start=False):
        self.oc = oc
        self.args = (ini_states, horizon, taus, waypoints, sel)
        self.kw = dict(pdata=pdata, mode=mode, rounds=rounds, chunks=chunks)
        self.warm_start = bool(warm_start)
        self.n_auxvar = oc.n_auxvar
        self.loss_trace = []
        self.parameter_trace = []

    def load_optimization_function(self, para_input: dict):
        m = para_input["method"]
        if m not in METHOD_IDS:
            raise Exception("Wrong optimization method type!")
        self.method = METHOD_IDS[m]
        self.learning_rate = float(para_input["learning_rate"])
        self.iter_num = int(para_input["iter_num"])
        self.mu = float(para_input.get("mu", 0.0))
        self.true_loss = bool(para_input.get("true_loss_print_flag", False)) and m == "Nesterov"
        self.beta_1 = float(para_input.get("beta_1", 0.0))
        self.beta_2 = float(para_input.get("beta_2", 0.0))
        self.epsilon = float(para_input.get("epsilon", 0.0))

    def run(self, initial_parameter, check_every=0, loss_stop=0.9, grad_stop=0.05):
        oc = self.oc
        lib = oc.build()
        mem = oc._device()
        r, cap = self.n_auxvar, self.iter_num
        th0 = np.array(initial_parameter, dtype=float).reshape(r)
        theta = mem.from_host(th0)
        theta_eval = mem.from_host(th0.reshape(1, r))
        state = mem.zeros((3, r))
        it = mem.zeros((2,), "i4")
        loss_trace = mem.zeros((cap,))
        ptrace = mem.zeros((cap + 1, r))
        ptrace[0] = theta
        failed = mem.zeros((1,))
        x0, horizon, taus, wp, sel = self.args
        # inputs go to the device once; every iteration then reads them (and theta_eval) in place
        x0 = mem.from_host(np.asarray(x0, dtype=float).reshape(-1, oc.n_state)) if not hasattr(x0, "data_ptr") else x0
        B = int(x0.shape[0])
        taus = mem.from_host(np.asarray(taus, dtype=float).reshape(-1, np.asarray(taus).shape[-1])) if not hasattr(taus, "data_ptr") else taus
        wp = mem.from_host(np.asarray(wp, dtype=float).reshape(B, -1, len(sel))) if not hasattr(wp, "data_ptr") else wp
        if self.kw["pdata"] is not None and not hasattr(self.kw["pdata"], "data_ptr"):
            self.kw["pdata"] = mem.from_host(np.asarray(self.kw["pdata"], dtype=float).reshape(B, oc.n_pvar))
        hyper = (self.method, self.learning_rate, self.mu, self.beta_1, self.beta_2, self.epsilon, float(loss_stop), float(grad_stop))

        def step(phase, red, defer):
            lib.optim_step(phase, *hyper, mem.ptr(theta), mem.ptr(theta_eval), mem.ptr(state), mem.ptr(red), mem.ptr(it),
                           mem.ptr(loss_trace), mem.ptr(ptrace), cap, defer, mem.stream())

        prev = {}

        def evaluate():
            full, sol, aux = oc.gradIterBatch(x0, horizon, theta_eval.reshape(r), taus, wp, sel, init=prev.get("sol"), **self.kw)
            failed.__iadd__(aux["n_failed"])
            if self.warm_start:
                prev["sol"] = sol
            return full

        for j in range(cap):
            step(0, None, 0)
            red = evaluate()
            step(1, red, 1 if self.true_loss else 0)
            if self.true_loss:
                step(0, None, 1)
                step(2, evaluate(), 0)
            if check_every and (j + 1) % check_every == 0 and int(mem.to_host(it)[1]):
                break
        done = int(mem.to_host(it)[0])
        nf = float(np.asarray(mem.to_host(failed))[0])
        if nf:
            raise FloatingPointError("%d CPDP evaluation(s) of the run had failed OCPs" % int(round(nf)))
        self.loss_trace = np.asarray(mem.to_host(loss_trace))[:done].tolist()
        self.parameter_trace = np.asarray(mem.to_host(ptrace))[:done + 1].tolist()
        self.stopped_early = bool(int(mem.to_host(it)[1]))
        return np.asarray(mem.to_host(theta), dtype=float).copy()
