"""Cost of the box bounds on the headline batch (4096 quadrotor OCPs, n_grid 50, synthetic.quad_batch): the unbounded model
against the thrust-bounded one (standard.quadrotor_bounded_oc, 1 <= f_i <= 4), alternated in one process.

Per model: the forward solve with the adaptive round count (ms, Newton iterations per OCP: distribution and quantiles, solver
status counts, rounds launched), the mode-2 auxiliary system at that solution (ms), and a full mode-1 gradient step as bench.py
times it (gradIterBatch with chunks and a fixed round count; the bounded model's fixed count is taken from its measured
iterations).  CUDA events, warm-up, median over --reps alternated repetitions.  Prints one JSON line per model.

    python tools/bench_bounds.py [--batch 4096] [--n-grid 50] [--reps 5] > profiles/r05_bench_bounds.jsonl
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_discrete import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--n-grid", type=int, default=50)
    ap.add_argument("--chunks", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=8, help="fixed Newton rounds of the unbounded model's mode-1 step (bench.py's)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()

    import torch
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic
    assert torch.cuda.is_available(), "tools/bench_bounds.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ocs = {"unbounded": standard.quadrotor_oc(n_grid=a.n_grid), "thrust_bounded": standard.quadrotor_bounded_oc(n_grid=a.n_grid)}
    for oc in ocs.values():
        oc.build(name=oc.lib_name)
    qb = synthetic.quad_batch(a.batch)
    inp = {k: torch.from_numpy(np.ascontiguousarray(qb[k])).to(dev) for k in ("x0", "goal", "wp", "taus", "theta")}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    def solve(oc):
        return oc.cocSolverBatch(inp["x0"], 1.0, inp["theta"], pdata=inp["goal"])

    # the adaptive solve tells how many rounds the fixed-round step needs
    rounds = {}
    for k, oc in ocs.items():
        solve(oc)
        torch.cuda.synchronize()
        it = solve(oc)["iters"].cpu().numpy()
        rounds[k] = a.rounds if k == "unbounded" else int(it.max()) + 1

    def step(k):
        oc = ocs[k]
        return oc.gradIterBatch(inp["x0"], 1.0, inp["theta"], inp["taus"], inp["wp"], qb["sel"], pdata=inp["goal"],
                                mode=oc.MODE_BDF, rounds=rounds[k], chunks=a.chunks)

    t_solve = {k: [] for k in ocs}
    t_aux2 = {k: [] for k in ocs}
    t_step = {k: [] for k in ocs}
    last = {}
    for rep in range(a.warmup + a.reps):
        for k, oc in ocs.items():
            ts, sol = timed(lambda: solve(oc))
            nr = oc._lib.last_rounds()
            ta, aux2 = timed(lambda: oc.auxSysSolverBatch(sol, inp["taus"], inp["wp"], qb["sel"], mode=oc.MODE_DISCRETE))
            tt, st = timed(lambda: step(k))
            if rep >= a.warmup:
                t_solve[k].append(ts)
                t_aux2[k].append(ta)
                t_step[k].append(tt)
            last[k] = (sol, aux2, st, nr)

    gpu, power = gpu_info()
    for k, oc in ocs.items():
        sol, aux2, (red, ss, sa), nr = last[k]
        it = sol["iters"].cpu().numpy()
        status = sol["status"].cpu().numpy()
        line = {
            "tool": "tools/bench_bounds.py", "model": k, "bounds": "1 <= f_i <= 4" if k != "unbounded" else "none",
            "batch": a.batch, "n_grid": a.n_grid,
            "solve_ms": round(float(np.median(t_solve[k])), 3), "solve_ms_all": [round(v, 3) for v in t_solve[k]],
            "solve_rounds_launched": nr,
            "newton_iters_hist": {str(v): int(c) for v, c in zip(*np.unique(it, return_counts=True))},
            "newton_iters_mean": round(float(it.mean()), 3),
            "newton_iters_p50_p90_p99_max": [int(np.percentile(it, q, method="higher")) for q in (50, 90, 99)] + [int(it.max())],
            "solve_status_counts": np.bincount(status, minlength=6).tolist(),
            "mode2_aux_ms": round(float(np.median(t_aux2[k])), 3),
            "mode2_aux_status_counts": np.bincount(aux2["aux_status"].cpu().numpy(), minlength=6).tolist(),
            "mode1_step_ms": round(float(np.median(t_step[k])), 3), "mode1_step_ms_all": [round(v, 3) for v in t_step[k]],
            "mode1_step_rounds": rounds[k], "mode1_step_chunks": a.chunks,
            "mode1_step_n_failed": float(sa["n_failed"].cpu().numpy()[0]),
            "timing": "CUDA events, %d warm-up repetition(s), median of %d repetitions, models alternated in one process"
                      % (a.warmup, a.reps),
            "gpu": gpu, "power_limit": power,
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
