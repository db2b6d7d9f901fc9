"""Step time of the three auxiliary modes on the headline batch (4096 quadrotor OCPs, n_grid 50, synthetic.quad_batch), one
process, modes alternated: 1 (as-shipped BDF backward sweep), 0 (RK45 backward sweep), 2 (exact discrete derivative).

A step is what bench.py times: COCSys.gradIterBatch with the batch in two chunks on two streams and a fixed number of Newton
rounds, inputs resident in HBM.  The aux phases are timed separately on one stream at the converged solution of one solve
(phase 1 = backward sweep / stage derivatives + backward recursion, phase 2 = forward sweep / rollout, both with the loss).
CUDA events, warm-up, median over --reps alternated repetitions.  Prints one JSON line per mode.

    python tools/bench_discrete.py [--batch 4096] [--n-grid 50] [--reps 7] > out.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:          # (the number is still reported, with the reason the card could not be named)
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--n-grid", type=int, default=50)
    ap.add_argument("--chunks", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()

    import torch
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic
    assert torch.cuda.is_available(), "tools/bench_discrete.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    oc = standard.quadrotor_oc(n_grid=a.n_grid)
    oc.build(name=oc.lib_name)
    qb = synthetic.quad_batch(a.batch)
    inp = {k: torch.from_numpy(np.ascontiguousarray(qb[k])).to(dev) for k in ("x0", "goal", "wp", "taus", "theta")}
    modes = (oc.MODE_BDF, oc.MODE_RK45, oc.MODE_DISCRETE)
    names = {oc.MODE_BDF: "bdf", oc.MODE_RK45: "rk45", oc.MODE_DISCRETE: "discrete"}

    def step(mode):
        return oc.gradIterBatch(inp["x0"], 1.0, inp["theta"], inp["taus"], inp["wp"], qb["sel"], pdata=inp["goal"], mode=mode,
                                rounds=a.rounds, chunks=a.chunks)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    step_ms = {m: [] for m in modes}
    last = {}
    for m in modes:
        for _ in range(a.warmup):
            step(m)
    torch.cuda.synchronize()
    for _ in range(a.reps):
        for m in modes:
            ms, res = timed(lambda: step(m))
            step_ms[m].append(ms)
            last[m] = res

    # aux phases alone, one stream, at the solution of one solve
    sol = oc.cocSolverBatch(inp["x0"], 1.0, inp["theta"], pdata=inp["goal"])
    ph1 = {m: [] for m in modes}
    ph2 = {m: [] for m in modes}
    for rep in range(a.reps + a.warmup):
        for m in modes:
            t1, aux = timed(lambda: oc.auxSysSolverBatch(sol, inp["taus"], inp["wp"], qb["sel"], mode=m, phases=1))
            t2, aux = timed(lambda: oc.auxSysSolverBatch(sol, inp["taus"], inp["wp"], qb["sel"], mode=m, phases=2, out=aux))
            if rep >= a.warmup:
                ph1[m].append(t1)
                ph2[m].append(t2)

    gpu, power = gpu_info()
    ref = last[oc.MODE_DISCRETE][0].cpu().numpy()
    for m in modes:
        red, s, aux = last[m]
        red = red.cpu().numpy()
        med = float(np.median(step_ms[m]))
        line = {
            "tool": "tools/bench_discrete.py", "aux_mode": m, "aux_mode_name": names[m], "batch": a.batch, "n_grid": a.n_grid,
            "chunks": a.chunks, "newton_rounds": a.rounds,
            "ms_per_step": round(med, 3), "ms_per_step_all": [round(v, 3) for v in step_ms[m]],
            "ocp_grad_iters_per_s": round(a.batch / (med / 1e3), 1),
            "aux_phase1_ms": round(float(np.median(ph1[m])), 3), "aux_phase2_ms": round(float(np.median(ph2[m])), 3),
            "n_failed": float(aux["n_failed"].cpu().numpy()[0]),
            "aux_status_counts": np.bincount(aux["aux_status"].cpu().numpy(), minlength=6).tolist(),
            "sum_loss": float(red[0]),
            "grad_rel_diff_vs_discrete": float(np.linalg.norm(red[1:] - ref[1:]) / np.linalg.norm(ref[1:])),
            "timing": "CUDA events, %d warm-up steps per mode, median of %d repetitions, modes alternated in one process" % (a.warmup, a.reps),
            "gpu": gpu, "power_limit": power,
        }
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
