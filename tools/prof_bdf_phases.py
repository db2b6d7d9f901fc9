#!/usr/bin/env python3
"""Developer tool (not part of the product path): builds tuning variants of the quadrotor library (residency of
k_riccati_bdf, optional clock64 phase instrumentation) and times the backward sweep alone at several batch sizes.

  python tools/prof_bdf_phases.py --build-only            (here: cross-compiles the variants into lib/)
  python tools/prof_bdf_phases.py --batches 148,512,4096  (GPU box: loads the prebuilt variants, prints one JSON line each)
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {
    "base": [],
    "time": ["-DCPDP_BDF_TIMING"],
    "eig_off": ["-DCPDP_BDF_EIG_KAPPA=0"],                    # every Newton solve on the Bartels-Stewart sweep
    "time_eig_off": ["-DCPDP_BDF_TIMING", "-DCPDP_BDF_EIG_KAPPA=0"],
    "l2s1": ["-DCPDP_BDF_LMUL_UNROLL=2", "-DCPDP_BDF_STENCIL_UNROLL=1"],
    "l1s1": ["-DCPDP_BDF_LMUL_UNROLL=1", "-DCPDP_BDF_STENCIL_UNROLL=1"],
    "l4s2": ["-DCPDP_BDF_LMUL_UNROLL=4", "-DCPDP_BDF_STENCIL_UNROLL=2"],
    "unclamped": ["-DCPDP_BDF_SWEEP_UNCLAMPED"],
    "prev": [],                                  # (a library built by hand from another revision of the sources, for A/B runs)
    "l2": ["-DCPDP_BDF_LMUL_UNROLL=2"],
    "l4": ["-DCPDP_BDF_LMUL_UNROLL=4"],
    "r168": ["-DCPDP_BDF_MINB=12"],
    "r128": ["-DCPDP_BDF_MINB=16"],
    "l13s1": ["-DCPDP_BDF_LMUL_UNROLL=13", "-DCPDP_BDF_STENCIL_UNROLL=1"],
}
PHASES = ["prepare", "rhs", "jacobian", "schur", "factor", "solve", "norm", "change_D", "total"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="148,512,4096")
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--n-grid", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--build-only", action="store_true")
    a = ap.parse_args()
    import lfsd_b200  # noqa: F401
    from lfsd_b200 import standard, synthetic, _capi, codegen
    oc = standard.quadrotor_oc(n_grid=a.n_grid)
    text, info = codegen.generate_model_header(oc.lib_name, oc.state, oc.control, oc.auxvar, oc.dyn, oc.path_cost,
                                               oc.final_cost, oc.pvar)
    libs = {}
    for v in a.variants.split(","):
        so = os.path.join(_capi.LIB_DIR, "libcpdp_quadrotor_%s.so" % v)
        if a.build_only or not os.path.exists(so):
            _capi.EXTRA_NVCC_FLAGS = VARIANTS[v]
            so = _capi.build_model_library("quadrotor_" + v, text, force=True)
            _capi.EXTRA_NVCC_FLAGS = []
            print("built", so, file=sys.stderr)
        libs[v] = so
    if a.build_only:
        return
    import torch
    for B in [int(x) for x in a.batches.split(",")]:
        qb = synthetic.quad_batch(B)
        base = standard.quadrotor_oc(n_grid=a.n_grid)
        base.build(name=base.lib_name)
        sol = base.cocSolverBatch(qb["x0"], 1.0, qb["theta"], pdata=qb["goal"])
        torch.cuda.synchronize()
        for v, so in libs.items():
            oc2 = standard.quadrotor_oc(n_grid=a.n_grid)
            oc2._lib = _capi.CpdpLib(so)
            oc2.aux_mode = oc2.MODE_BDF
            times = []
            for _ in range(a.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                aux = oc2.auxSysSolverBatch(sol, qb["taus"], qb["wp"], qb["sel"], phases=1)
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            out = {"variant": v, "batch": B, "ms": [round(t, 3) for t in times],
                   "failed": int((aux["aux_status"] != 0).sum().item())}
            if "time" in v:
                tp = aux["Ua"].reshape(B, -1)[:, :28].cpu().numpy()
                tot = tp[:, 8].mean()
                out["cycles_total_mean"] = float(tot)
                out["phase_share"] = {PHASES[i]: round(float(tp[:, i].mean() / tot), 4) for i in range(8)}
                out["phase_share"]["glue"] = round(float(1.0 - tp[:, :8].sum(1).mean() / tot), 4)
                cnt = aux["counters"].cpu().numpy().astype(float)
                out["cycles_per_call"] = {
                    "prepare": float(tp[:, 0].mean() / (cnt[:, 1].mean() + 2 * a.n_grid)),
                    "rhs": float(tp[:, 1].mean() / cnt[:, 0].mean()),
                    "jacobian": float(tp[:, 2].mean() / cnt[:, 5].mean()),
                    "schur": float(tp[:, 3].mean() / cnt[:, 5].mean()),
                    "factor": float(tp[:, 4].mean() / cnt[:, 4].mean()),
                    "solve": float(tp[:, 5].mean() / (cnt[:, 0].mean() - 2 * a.n_grid)),
                }
                nsol = cnt[:, 0].mean() - 2 * a.n_grid
                # Newton solves / Jacobians on the eigen path and on the sweep (path counts of the timing build)
                n_eig, n_sweep, j_eig, j_sweep = (float(tp[:, 24 + i].mean()) for i in range(4))
                out["paths"] = {"solves_eig": n_eig, "solves_sweep": n_sweep, "jac_eig": j_eig, "jac_sweep": j_sweep,
                                "solves_sweep_share": round(n_sweep / max(n_eig + n_sweep, 1e-300), 4)}
                per = lambda col, n_: float(tp[:, col].mean() / n_) if n_ > 0 else None
                out["solve_cycles_per_call"] = {"QtBQ": per(10, nsol), "QYQt": per(14, nsol), "sym_W": per(15, nsol),
                                                "block_scaling": per(9, n_eig), "stencil_in": per(11, n_sweep),
                                                "sweep": per(12, n_sweep), "stencil_out": per(13, n_sweep)}
                nj = cnt[:, 5].mean()
                out["schur_cycles_per_call"] = {nm: float(tp[:, 16 + i].mean() / nj) for i, nm in enumerate(
                    ["hessenberg", "qr_scans", "qr_scans_plus_chase", "rotations", "rotations_plus_packing", "eig_basis"])}
                out["counters_mean"] = {"rhs": cnt[:, 0].mean(), "steps": cnt[:, 1].mean(), "lu": cnt[:, 4].mean(), "jac": nj}
            print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
