"""What the warm start (cocSolverBatch(init=...), DESIGN.md §3.10) saves on the headline batch: 4096 quadrotor OCPs, n_grid 50,
synthetic.quad_batch, one device.  Cold and warm are alternated in one process; CUDA events, warm-up, median of --reps.

  (a) learner_step:     the solve at theta_1 = theta_0 - 0.01 * dL/dtheta (the first step of a mode-2 Nesterov learner at lr 0.01),
                        cold against warm from the solution at theta_0.  L is the mean loss over the batch (the step the
                        single-problem quad_example.py learner takes), and, as a second line, the batch's summed loss (the step
                        DeviceLearner takes at lr 0.01 on 4096 problems: 4096 times longer);
  (b) device_learner:   ms per iteration of DeviceLearner(mode=2, Nesterov lr 0.01 / B mu 0.9: the mean loss), warm_start False
                        against True;
  (c) receding_horizon: ms per step of a 20-step loop (x <- X[:, 1]), cold against shift = 1;
  (d) bounded_mu_sweep: the thrust-bounded quadrotor (1 <= f_i <= 4), (a)'s solve warm-started at each mu_init.
Each line carries the Newton iterations per OCP (mean, p50 / p90 / p99 / max) and the solve ms.

    python tools/bench_warm.py [--batch 4096] [--n-grid 50] [--reps 5] > profiles/r07_bench_warm.jsonl
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_discrete import gpu_info  # noqa: E402


def iters_stats(it):
    it = np.asarray(it)
    return {"mean": round(float(it.mean()), 3),
            "p50_p90_p99_max": [int(np.percentile(it, q, method="higher")) for q in (50, 90, 99)] + [int(it.max())]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--n-grid", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--learner-iters", type=int, default=6)
    ap.add_argument("--mpc-steps", type=int, default=20)
    a = ap.parse_args()

    import torch
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic
    from lfsd_b200.optim import DeviceLearner
    assert torch.cuda.is_available(), "tools/bench_warm.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    oc = standard.quadrotor_oc(n_grid=a.n_grid)
    ob = standard.quadrotor_bounded_oc(n_grid=a.n_grid)
    for o in (oc, ob):
        o.build(name=o.lib_name)
    qb = synthetic.quad_batch(a.batch)
    inp = {k: torch.from_numpy(np.ascontiguousarray(qb[k])).to(dev) for k in ("x0", "goal", "wp", "taus")}
    gpu, power = gpu_info()
    common = dict(tool="tools/bench_warm.py", batch=a.batch, n_grid=a.n_grid, gpu=gpu, power_limit=power)
    timing = "CUDA events, %d warm-up repetition(s), median of %d repetitions, cold and warm alternated in one process" % (
        a.warmup, a.reps)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    def solve(o, th, **kw):
        return o.cocSolverBatch(inp["x0"], 1.0, th, pdata=inp["goal"], **kw)

    # theta_1: the first step of the mode-2 Nesterov learner (zero velocity: theta_1 = theta_0 - lr * dL/dtheta)
    th0 = np.asarray(qb["theta"], dtype=float)
    red, _, _ = oc.gradIterBatch(inp["x0"], 1.0, th0, inp["taus"], inp["wp"], qb["sel"], pdata=inp["goal"], mode=oc.MODE_DISCRETE)
    grad = red.cpu().numpy()[1:]
    steps = {"mean": th0 - 0.01 * grad / a.batch, "sum": th0 - 0.01 * grad}
    for t in steps.values():
        t[0] = max(t[0], 1e-8)

    # (a) and (d)
    def step_case(o, mus, th1):
        base = solve(o, th0)
        torch.cuda.synchronize()
        t = {k: [] for k in ["cold"] + ["warm_%g" % m for m in mus]}
        last = {}
        for rep in range(a.warmup + a.reps):
            for k in t:
                kw = {} if k == "cold" else dict(init=base, mu_init=float(k[5:]))
                ms, s = timed(lambda: solve(o, th1, **kw))
                if rep >= a.warmup:
                    t[k].append(ms)
                last[k] = s
        out = {}
        for k in t:
            st = last[k]["status"].cpu().numpy()
            out[k] = dict(solve_ms=round(float(np.median(t[k])), 3), solve_ms_all=[round(v, 3) for v in t[k]],
                          newton_iters=iters_stats(last[k]["iters"].cpu().numpy()),
                          status_counts=np.bincount(st, minlength=6).tolist())
        return out

    for k, th1 in steps.items():
        r = step_case(oc, [oc.warm_mu_init], th1)
        print(json.dumps(dict(common, case="a_learner_step", model="quadrotor", loss=k,
                              step="theta_1 = theta_0 - 0.01 dL/dtheta, L the %s of the batch's losses (mode 2)" % k,
                              step_rel_norm=float(np.linalg.norm(th1 - th0) / np.linalg.norm(th0)),
                              cold=r["cold"], warm=r["warm_%g" % oc.warm_mu_init], timing=timing)), flush=True)

    # (b) DeviceLearner ms per iteration
    para = {"learning_rate": 0.01 / a.batch, "iter_num": a.learner_iters, "method": "Nesterov", "mu": 0.9, "true_loss_print_flag": True}
    tl = {False: [], True: []}
    traces = {}
    failures = []
    for rep in range(a.warmup + a.reps):
        for warm in (False, True):
            D = DeviceLearner(oc, inp["x0"], 1.0, inp["taus"], inp["wp"], qb["sel"], pdata=inp["goal"], mode=oc.MODE_DISCRETE,
                              warm_start=warm)
            D.load_optimization_function(para)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            try:
                D.run(th0, loss_stop=-1.0, grad_stop=-1.0)      # (run ends in a device-to-host read: synchronised)
            except FloatingPointError as e:                      # (reported, not hidden: the line says which run failed)
                failures.append("%s: %s" % ("warm" if warm else "cold", e))
            dt = (time.perf_counter() - t0) * 1e3 / a.learner_iters
            if rep >= a.warmup:
                tl[warm].append(dt)
            traces[warm] = D.loss_trace
    lc, lw = np.array(traces[False]), np.array(traces[True])
    print(json.dumps(dict(common, case="b_device_learner", model="quadrotor",
                          config="mode 2, Nesterov lr 0.01 / batch mu 0.9, true_loss_print_flag (2 evaluations per iteration), %d iterations"
                                 % a.learner_iters,
                          cold_ms_per_iter=round(float(np.median(tl[False])), 3), warm_ms_per_iter=round(float(np.median(tl[True])), 3),
                          cold_all=[round(v, 3) for v in tl[False]], warm_all=[round(v, 3) for v in tl[True]],
                          loss_trace_max_rel_diff=float(np.abs(lw - lc).max() / np.abs(lc).max()) if len(lw) == len(lc) else None,
                          runs_with_failed_ocps=failures,
                          timing="host clock around DeviceLearner.run (ends synchronised), %d warm-up, median of %d, alternated"
                                 % (a.warmup, a.reps))), flush=True)

    # (c) receding horizon
    tm = {"cold": [], "shift1": []}
    it = {"cold": [], "shift1": []}
    for rep in range(a.warmup + a.reps):
        x = {"cold": inp["x0"].clone(), "shift1": inp["x0"].clone()}
        prev = None
        for s in range(a.mpc_steps):
            for k in ("cold", "shift1"):
                kw = dict(init=prev, shift=1) if k == "shift1" else {}
                ms, sol = timed(lambda: oc.cocSolverBatch(x[k], 1.0, th0, pdata=inp["goal"], **kw))
                if rep >= a.warmup and s > 0:
                    tm[k].append(ms)
                    it[k].append(sol["iters"].cpu().numpy())
                if k == "shift1":
                    prev = sol
                x[k] = sol["X"][:, 1].contiguous()
    print(json.dumps(dict(common, case="c_receding_horizon", model="quadrotor", steps=a.mpc_steps,
                          cold=dict(ms_per_step=round(float(np.median(tm["cold"])), 3), newton_iters=iters_stats(np.concatenate(it["cold"]))),
                          shift1=dict(ms_per_step=round(float(np.median(tm["shift1"])), 3),
                                      newton_iters=iters_stats(np.concatenate(it["shift1"]))),
                          timing="CUDA events per solve, steps 2..%d of %d repetitions (after %d warm-up), median over steps and "
                                 "repetitions; cold and shift=1 alternated step by step" % (a.mpc_steps, a.reps, a.warmup))),
          flush=True)

    # (d) bounded mu_init sweep
    mus = [1e-1, 1e-2, 1e-3, 1e-4, 1e-5, 1e-6, 1e-7, 1e-8]
    r = step_case(ob, mus, steps["mean"])
    print(json.dumps(dict(common, case="d_bounded_mu_sweep", model="quadrotor thrust-bounded (1 <= f_i <= 4)",
                          step="(a)'s mean-loss step (the unbounded model's gradient)", results=r,
                          timing=timing)), flush=True)


if __name__ == "__main__":
    main()
