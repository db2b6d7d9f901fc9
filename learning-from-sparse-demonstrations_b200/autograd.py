"""torch.autograd layer over the batched solve: ``X, U, info = cpdp_layer(oc, x0, theta, horizon)`` returns the optimal trajectories
as tensors that any loss written in torch can consume, and ``loss.backward()`` carries its gradient to ``x0`` and ``theta`` (and, with ``pdata_grad=True``, to the per-problem constants ``pdata``).

Forward is ``COCSys.cocSolverBatch``; backward is ``COCSys.auxSysAdjointBatch`` (the adjoint of mode 2, DESIGN.md §3.9) on the
saved solution, so the gradient is the exact derivative of the discretised problem the solver solves.  Problems whose solve did
not converge, or whose auxiliary system failed (``info["aux_status"]`` != 0 after backward), contribute zero gradient: check
``info["status"]`` before stepping on it.  Only first derivatives exist (``once_differentiable``)."""
import torch
from torch.autograd.function import once_differentiable

__all__ = ["cpdp_layer"]

_SAVED = ("X", "U", "Lam", "status", "theta", "pdata", "Zl", "Zu", "mu")


class CpdpSolve(torch.autograd.Function):
    """(x0 [B,n], theta [r] or [B,r]) -> (X [B,N+1,n], U [B,N+1,m]); the non-differentiable outputs go to ``info``."""

    @staticmethod
    def forward(ctx, x0, theta, oc, horizon, pdata, rounds, info, init, shift, pdata_grad):
        if pdata is not None and hasattr(pdata, "detach"):
            pdata = pdata.detach()
        sol = oc.cocSolverBatch(x0.detach(), horizon, theta.detach(), pdata=pdata, rounds=rounds, init=init, shift=shift)
        mem = oc._device()
        info.update({k: sol[k] for k in ("Lam", "status", "iters", "kkt", "cost", "Zl", "Zu", "mu") if k in sol})
        info["aux_status"] = mem.zeros((sol["B"],), "i4")
        ctx.oc, ctx.info = oc, info
        ctx.keep = {k: sol[k] for k in ("B", "horizon", "theta_stride", "_slot")}
        ctx.saved_keys = [k for k in _SAVED if k in sol]
        ctx.save_for_backward(*(sol[k] for k in ctx.saved_keys))
        ctx.shared = theta.dim() == 1
        ctx.like = ((x0.device, x0.dtype), (theta.device, theta.dtype))
        ctx.pd_like = (pdata.device, pdata.dtype) if pdata_grad else None
        ctx.set_materialize_grads(False)
        X, U = sol["X"], sol["U"]
        return X, U

    @staticmethod
    @once_differentiable
    def backward(ctx, Xbar, Ubar):
        oc, info = ctx.oc, ctx.info
        (x0_dev, x0_dt), (th_dev, th_dt) = ctx.like
        if Xbar is None and Ubar is None:
            return None, None, None, None, None, None, None, None, None, None
        sol = dict(ctx.keep, **dict(zip(ctx.saved_keys, ctx.saved_tensors)))
        want_pd = ctx.pd_like is not None and ctx.needs_input_grad[4]
        adj = oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=want_pd)
        info["aux_status"].copy_(adj["aux_status"])
        gx0 = gth = None
        if ctx.needs_input_grad[0]:
            gx0 = adj["x0_bar"].to(device=x0_dev, dtype=x0_dt)
        if ctx.needs_input_grad[1]:
            tb = adj["theta_bar"]
            if ctx.shared:
                # a theta shared by the batch: fixed-tree sum of the per-problem rows (depends on B only, not on timing)
                tb = oc.reduceRows(tb)
            gth = tb.to(device=th_dev, dtype=th_dt)
        gpd = adj["pdata_bar"].to(device=ctx.pd_like[0], dtype=ctx.pd_like[1]) if want_pd else None
        return gx0, gth, None, None, gpd, None, None, None, None, None


def cpdp_layer(oc, x0, theta, horizon, pdata=None, rounds=0, init=None, shift=0, pdata_grad=False):
    """Differentiable batched solve.  x0 [B,n]; theta [r] (shared by the batch) or [B,r]; pdata [B,q] (per-problem constants,
    differentiable with ``pdata_grad=True``: then backward returns its gradient, DESIGN.md §3.11); rounds as in ``cocSolverBatch``.  Returns (X [B,N+1,n], U [B,N+1,m], info) where info holds Lam, status,
    iters, kkt, cost (and Zl, Zu, mu for a bounded model), and an aux_status tensor that backward fills in place.

    init, shift: warm start of the solve as in ``cocSolverBatch``, e.g. ``init=dict(info, X=X, U=U)`` of the previous call.  It is
    not differentiated: the converged point does not depend on where the solve started, beyond the solver tolerance."""
    if pdata_grad:
        if pdata is None or oc.n_pvar == 0:
            raise ValueError("pdata_grad=True needs a model with per-problem constants and a pdata [B,q] tensor")
    elif pdata is not None and getattr(pdata, "requires_grad", False):
        raise NotImplementedError("cpdp_layer differentiates with respect to x0 and theta unless pdata_grad=True: pass "
                                  "pdata_grad=True for the gradient with respect to the per-problem constants pdata")
    info = {}
    X, U = CpdpSolve.apply(x0, theta, oc, float(horizon), pdata, int(rounds), info, init, int(shift), bool(pdata_grad))
    return X, U, info
