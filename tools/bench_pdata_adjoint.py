"""Cost of the pdata adjoint (cpdp_aux_adjoint_pd) against the theta/x0 adjoint (cpdp_aux_adjoint) on the headline batch
(4096 quadrotor OCPs, n_grid 50, synthetic.quad_batch, goal positions as pdata).

Timed, alternated in one process (CUDA events, warm-up, median over --reps repetitions):
  * cpdp_aux_adjoint (auxSysAdjointBatch) and cpdp_aux_adjoint_pd (auxSysAdjointBatch(pdata_bar=True));
  * cpdp_layer forward + backward with a dense tracking loss, without and with pdata_grad=True.
Then, in a separate torch.profiler run, the device time of every kernel the two entry points launch.
Prints one JSON line per measurement group.

    python tools/bench_pdata_adjoint.py [--batch 4096] [--n-grid 50] [--reps 7] > profiles/r09_bench_pdata.jsonl
"""
import argparse
import json
import os
import re
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
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--profile-reps", type=int, default=3)
    a = ap.parse_args()

    import torch
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic
    from lfsd_b200.autograd import cpdp_layer
    assert torch.cuda.is_available(), "tools/bench_pdata_adjoint.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu, power = gpu_info()
    oc = standard.quadrotor_oc(n_grid=a.n_grid)
    oc.build(name=oc.lib_name)
    B, N, n, m = a.batch, a.n_grid, oc.n_state, oc.n_control
    qb = synthetic.quad_batch(B)
    inp = {k: torch.from_numpy(np.ascontiguousarray(qb[k])).to(dev) for k in ("x0", "goal", "theta")}
    g = torch.Generator(device=dev).manual_seed(0)
    Xbar = torch.randn(B, N + 1, n, generator=g, device=dev, dtype=torch.float64)
    Ubar = torch.randn(B, N + 1, m, generator=g, device=dev, dtype=torch.float64)
    Xref = torch.randn(B, N + 1, n, generator=g, device=dev, dtype=torch.float64)
    theta = inp["theta"].clone().requires_grad_(True)
    goal = inp["goal"].clone().requires_grad_(True)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    def layer_step(pd_grad):
        theta.grad = goal.grad = None
        X, U, info = cpdp_layer(oc, inp["x0"], theta, 1.0, pdata=goal if pd_grad else inp["goal"], pdata_grad=pd_grad)
        loss = ((X - Xref) ** 2).sum() + 1e-2 * (U ** 2).sum()
        loss.backward()
        return info

    sol = oc.cocSolverBatch(inp["x0"], 1.0, inp["theta"], pdata=inp["goal"])
    t = {k: [] for k in ("aux_adjoint", "aux_adjoint_pd", "layer_fwd_bwd", "layer_fwd_bwd_pdata_grad")}
    for rep in range(a.warmup + a.reps):
        tj, adj = timed(lambda: oc.auxSysAdjointBatch(sol, Xbar, Ubar))
        tp, adjp = timed(lambda: oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True))
        tl, _ = timed(lambda: layer_step(False))
        tq, info = timed(lambda: layer_step(True))
        if rep >= a.warmup:
            for k, v in zip(t, (tj, tp, tl, tq)):
                t[k].append(v)
    line = {"tool": "tools/bench_pdata_adjoint.py", "model": "quadrotor", "batch": B, "n_grid": N,
            "solve_status_counts": np.bincount(sol["status"].cpu().numpy(), minlength=6).tolist(),
            "adjoint_pd_aux_status_counts": np.bincount(adjp["aux_status"].cpu().numpy(), minlength=5).tolist(),
            "theta_bar_equal": bool(torch.equal(adj["theta_bar"], adjp["theta_bar"])),
            "x0_bar_equal": bool(torch.equal(adj["x0_bar"], adjp["x0_bar"])),
            "timing": "CUDA events, %d warm-up repetition(s), median of %d repetitions, the four measurements alternated in one "
                      "process" % (a.warmup, a.reps),
            "gpu": gpu, "power_limit": power}
    for k, v in t.items():
        line[k + "_ms"] = round(float(np.median(v)), 3)
        line[k + "_ms_all"] = [round(x, 3) for x in v]
    print(json.dumps(line), flush=True)

    from torch.profiler import profile, ProfilerActivity
    for what, pd in (("cpdp_aux_adjoint", False), ("cpdp_aux_adjoint_pd", True)):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.profile_reps):
                oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=pd)
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.key_averages():
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            if dt > 0 and "cpdp_quadrotor" in ev.key:
                mt = re.search(r"cpdp_quadrotor::(k_\w+)", ev.key)
                short = mt.group(1) if mt else ev.key
                kernels[short] = {"calls": ev.count, "ms_per_call": round(dt / 1000.0 / ev.count, 4)}
        print(json.dumps({"tool": "tools/bench_pdata_adjoint.py", "what": "torch.profiler device time per kernel of " + what,
                          "batch": B, "n_grid": N, "profiled_calls": a.profile_reps, "kernels": kernels,
                          "gpu": gpu, "power_limit": power}), flush=True)


if __name__ == "__main__":
    main()
