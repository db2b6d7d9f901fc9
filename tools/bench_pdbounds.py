"""Cost of bounds that depend on pdata (DESIGN.md §3.12) on the headline batch (4096 quadrotor OCPs, n_grid 50,
synthetic.quad_batch): the thrust-bounded quadrotor with its limit compiled in against the same model with the limit f_max in pdata.

Three cases, alternated in one process (CUDA events, warm-up, median over --reps repetitions):
  * const     quadrotor_bounded (1 <= f_i <= 4 compiled in);
  * pd_same   quadrotor_pdbounded at f_max = 4 for every problem (the same problems);
  * pd_var    quadrotor_pdbounded with a per-problem f_max uniform in [3.5, 5].
For each: the solve (with mean / p50 / p90 / max iterations), mode-2 aux and cpdp_aux_adjoint_pd.  One JSON line per case.

    python tools/bench_pdbounds.py [--batch 4096] [--n-grid 50] [--reps 5] > profiles/r10_bench_pdbounds.jsonl
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()

    import torch
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic
    assert torch.cuda.is_available(), "tools/bench_pdbounds.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu, power = gpu_info()
    B, N = a.batch, a.n_grid
    qb = synthetic.quad_batch(B)
    rng = np.random.default_rng(7)
    fvar = rng.uniform(3.5, 5.0, size=(B, 1))
    goal = qb["goal"]
    cases = {
        "const": (standard.quadrotor_bounded_oc(n_grid=N), goal),
        "pd_same": (standard.quadrotor_pdbounded_oc(n_grid=N), np.hstack([goal, np.full((B, 1), 4.0)])),
        "pd_var": (standard.quadrotor_pdbounded_oc(n_grid=N), np.hstack([goal, fvar])),
    }
    x0 = torch.from_numpy(qb["x0"]).to(dev)
    taus = torch.from_numpy(np.tile(qb["taus"], (B, 1))).to(dev)
    wp = torch.from_numpy(qb["wp"]).to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    Xbar = torch.randn(B, N + 1, 13, generator=g, device=dev, dtype=torch.float64)
    Ubar = torch.randn(B, N + 1, 4, generator=g, device=dev, dtype=torch.float64)
    for oc, _ in cases.values():
        oc.build(name=oc.lib_name)
    pds = {k: torch.from_numpy(np.ascontiguousarray(v[1])).to(dev) for k, v in cases.items()}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    times = {k: dict(solve=[], aux=[], adjoint_pd=[]) for k in cases}
    last = {}
    for rep in range(a.warmup + a.reps):
        for k, (oc, _) in cases.items():
            ts, sol = timed(lambda: oc.cocSolverBatch(x0, 1.0, qb["theta"], pdata=pds[k]))
            ta, aux = timed(lambda: oc.auxSysSolverBatch(sol, taus, wp, qb["sel"], mode=oc.MODE_DISCRETE))
            tp, adj = timed(lambda: oc.auxSysAdjointBatch(sol, Xbar, Ubar, pdata_bar=True))
            if rep >= a.warmup:
                times[k]["solve"].append(ts)
                times[k]["aux"].append(ta)
                times[k]["adjoint_pd"].append(tp)
            last[k] = (sol, aux, adj)
    for k in cases:
        sol, aux, adj = last[k]
        st = sol["status"].cpu().numpy()
        it = sol["iters"].cpu().numpy()
        conv = st == 1
        rec = dict(case=k, model=cases[k][0].lib_name, batch=B, n_grid=N, gpu=gpu, power_limit=power,
                   status_counts={str(s): int((st == s).sum()) for s in np.unique(st)},
                   iters_mean=float(it[conv].mean()), iters_p50=float(np.percentile(it[conv], 50)),
                   iters_p90=float(np.percentile(it[conv], 90)), iters_max=int(it[conv].max()),
                   aux_status_nonzero=int((aux["aux_status"] != 0).sum().item()),
                   adjoint_status_nonzero=int((adj["aux_status"] != 0).sum().item()), reps=a.reps)
        for part, v in times[k].items():
            rec[part + "_ms_median"] = float(np.median(v))
            rec[part + "_ms_all"] = [round(x, 3) for x in v]
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
