#!/usr/bin/env python3
"""Benchmark of the CPDP gradient iteration (BASELINE.json metric: OCP gradient-iterations per second on batched
quadrotor OCPs, n_grid 50).

  python bench.py --gpus N --steps K --warmup W              our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W      the CPU oracle (stand-in for the reference's
                                                             CasADi/IPOPT/scipy path, which cannot run in this image)

One "step" = one CPDP gradient iteration for every OCP of the batch: forward solve from the zero seed, auxiliary
system (backward Riccati + forward sweep), loss and dL/dtheta, and the fixed-order cross-problem reduction.
Prints ONE JSON line on rank 0.  The inputs are seeded, so with the same arguments every run solves the same problems;
--dump-outputs DIR saves what the last timed step returned (see dump_outputs) to compare two builds output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "CPDP OCP gradient-iterations per second (batched quadrotor OCPs, n_grid 50)"
PORT_S_PER_OCP = 2.4      # core-seconds per OCP of the CPU port on the GPU boxes' host cores (measured; sizes the reference arm)
UNIT = "ocp_grad_iters/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="OCPs in total (--scaling strong, BASELINE's configuration) or per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--n-grid", type=int, default=50)
    ap.add_argument("--mode", default=None, choices=["bdf", "rk45"], help="backward Riccati integrator")
    ap.add_argument("--rtol", type=float, default=1e-3)
    ap.add_argument("--atol", type=float, default=1e-6)
    ap.add_argument("--chunks", type=int, default=2, help="batch chunks on separate CUDA streams (1 = single stream)")
    ap.add_argument("--rounds", type=int, default=8, help="Newton rounds launched per solve when chunks > 1 (no host sync)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the CPU baseline sample (0 = one per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-deadline", type=float, default=200.0, help="stop starting new CPU-baseline steps after this many seconds")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64), to compare two builds output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


# ----------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle) — the ONLY place besides tests/ and smoke() that touches oracle/
# ----------------------------------------------------------------------------------------------------------------
_ORC = None


def _cpu_init(n_grid):
    """Worker initialiser: one BLAS thread per worker (the oracle's linear algebra is 260x260 at most; the default
    all-core BLAS pool in every worker oversubscribes a many-core host catastrophically)."""
    global _ORC
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1)
    except Exception:
        pass
    from oracle import models
    from oracle.cpdp_oracle import Oracle
    _ORC = Oracle(models.quadrotor(), n_grid=n_grid)


def _cpu_ready(_):
    return os.getpid()


def _cpu_one(job):
    x0, goal, theta, taus, wp = job
    _ORC.pd = goal
    t0 = time.time()
    # as shipped: BDF backward, RK45 forward (scipy's own solve_ivp); Newton steps through the stage-structured (Riccati)
    # factorisation of the KKT matrix, so the port is not charged for a dense factorisation no sparse NLP solver performs
    loss, dl, ex = _ORC.grad_iter(x0, 1.0, theta, taus, wp, linear_solver="riccati")
    return loss, dl, ex["info"]["iters"], time.time() - t0


def cpu_baseline(n_grid, sample, steps=1, warmup=0, max_workers=0, deadline_s=240.0):
    """Oracle (the CPU restatement of the reference algorithm) on a bounded sample of the same synthetic batch, one
    process per host core.  Each step maps `sample` OCPs (default: four per worker) over the pool; the run stops
    taking new steps after `deadline_s`.  Returns (cpu_baseline dict, seconds, steps done)."""
    import multiprocessing
    from lfsd_b200 import synthetic
    # one BLAS / OpenMP thread per worker, decided before the workers import numpy: fresh interpreters (spawn) that inherit
    # these variables.  (Forked workers inherit an already initialised all-core BLAS pool; threadpoolctl alone did not
    # tame it when torch had not been imported first, and 16 x 16 spinning threads never finish.)
    for var in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[var] = "1"
    Pool = multiprocessing.get_context("spawn").Pool
    cores = os.cpu_count() or 1
    workers = min(cores, max_workers) if max_workers else cores
    sample = sample or 4 * workers          # ~10-15 s of CPU work on the box's cores
    workers = min(workers, sample)
    qb = synthetic.quad_batch(max(sample, 1))
    jobs = [(qb["x0"][b], qb["goal"][b], qb["theta"], qb["taus"], qb["wp"][b]) for b in range(sample)]
    t_pool = time.time()
    with Pool(workers, initializer=_cpu_init, initargs=(n_grid,)) as pool:
        pool.map(_cpu_ready, range(workers), chunksize=1)          # model build (sympy) is outside the timed region
        print("[cpu_baseline] %d workers ready after %.1f s" % (workers, time.time() - t_pool), file=sys.stderr, flush=True)
        for _ in range(warmup):
            pool.map(_cpu_one, jobs[:workers], chunksize=1)
        t0 = time.time()
        done = 0
        per = []
        for _ in range(steps):
            res = pool.map(_cpu_one, jobs, chunksize=1)
            per += [r[3] for r in res]
            done += 1
            print("[cpu_baseline] step %d: %.1f s elapsed, %.1f s per OCP per core" % (done, time.time() - t0, float(np.mean(per))),
                  file=sys.stderr, flush=True)
            if time.time() - t0 > deadline_s:
                break
        dt = time.time() - t0
    value = sample * done / dt
    return dict(value=value, unit=UNIT, cores=workers, kind="port", sample_ocps=sample,
                sample="%d OCPs per step (first indices of the seeded 4096-OCP batch), n_grid %d, %d step(s), %.1f s wall, "
                       "%.1f s per OCP per core; numpy/scipy port of the reference algorithm (Newton-KKT with a stage-structured "
                       "factorisation in place of IPOPT/MUMPS, scipy's BDF/RK45 called as shipped, model functions through "
                       "sympy.lambdify), one single-threaded process per host core (%d cores); its speed relative to the real "
                       "CasADi VM + IPOPT is unknown"
                       % (sample, n_grid, done, dt, float(np.mean(per)), cores)), dt, done


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def flop_model(info, n, m, r, N, S, iters_sum, B, cnt, mode):
    """Executed useful fp64 flops of one step (DESIGN.md section 5): op counts of the generated model code after CSE
    plus the sparse / packed-symmetric linear algebra around it, times the counters the kernels record (Newton
    iterations, rhs evaluations, LU factorisations).  cnt = summed counters [back rhs, back steps, fwd rhs, fwd steps,
    back LU, back Jacobians].  These are the flops of OUR formulation (sparsity and symmetry exploited), i.e. a lower
    bound on the dense algorithmic counts of SURVEY.md 8d."""
    nz = n + m
    stages = 4 * S
    per_int = stages * (2 * info["ops_fc"] + info["ops_hgrad"] + 8 * n)                     # k_stage_adjoint
    per_int += stages * nz * (info["ops_dir"] + 2 * (nz // 2 + 1) * n + 6 * n)              # k_stage_hessian (symmetric accumulation)
    per_int += 2 * n * n * nz + 2 * nz * nz * n + 2 * m * m * (n + 1) + 2 * n * n * m + 4 * n * nz + stages * info["ops_fc"]
    solve = iters_sum * N * per_int
    nnzx, nnzu = info["nnz_fx"], info["nnz_fu"]
    nt = n * (n + 1) // 2
    ric = 2 * nnzu * (n + r) + 2 * m * m * n + nt * (4 * nnzx / n * 1.0 + 4 * m) + n * r * (2 * nnzx / n + 2 + 2 * m)
    pmp = info["ops_pmp"] + 2 * (2 * n + m) * 3 + 2 * m ** 3
    fwd = pmp + 2 * nnzu * (n + r) + 2 * m * m * (n + r) + 2 * m * n * r + n * r * (2 * nnzx / n + 2 * nnzu / n + 1) \
        + 4 * (nt + n * r)
    ny_r, ny_f = nt + n * r, n * r
    if mode == "bdf":
        # k_riccati_bdf as built in round 2 (DESIGN.md 3.2): full n x (n+r) state columns, dense products in the Newton solve.
        # per rhs evaluation (= Newton iteration): right-hand side on the 20 columns of [P|W] (sparse fx, fu through COO lists,
        #   Huu^-1, the Y'Yp term), four 13^3 real products of the two-sided Schur transforms, the two block-rotation stencils,
        #   the complex triangular Lyapunov sweep (8 flops per complex multiply-add), the W block (X C and (I+cL)^-1), norms;
        # per accepted step: PMP matrices at t_new, predictor / psi / difference update, change_D;
        # per "LU" event (new c): Gauss-Jordan inverse of I + cL on [A | I] (26 columns, 13 pivots), Lyapunov pivots;
        # per Jacobian: closed-form L, C; Householder-Hessenberg + Francis QR with vectors (~25 n^3 + 10/3 n^3, LAPACK count)
        ncol = n + r
        rhs_cols = ncol * (2 * nnzu + 2 * m * m + 2 * nnzx + 2 * m * n + 6 * n)
        sweep_macs = sum((n - 1 - i) + (n - 1 - j) for i in range(n) for j in range(i, n))
        solve_bs = 4 * 2 * n ** 3 + 24 * nt + 20 * n * n + 8 * sweep_macs + 12 * nt + 2 * (2 * n * n * r) + 4 * n * n
        back = cnt[0] * (rhs_cols + solve_bs + 8 * n * ncol) \
            + cnt[1] * (pmp + 30 * n * ncol) + cnt[4] * (2 * n * n * 2 * n + 12 * nt) \
            + cnt[5] * (2 * n * n * m * 2 + 2 * n ** 3 + 2 * n * n * r + 25 * n ** 3 + 10.0 / 3 * n ** 3)
    else:
        back = cnt[0] * (ric + pmp * 6.0 / 7 + 16 * ny_r)
    fwdf = cnt[2] * (fwd + 16 * ny_f)
    return dict(solve=float(solve), aux_backward=float(back), aux_forward=float(fwdf), total=float(solve + back + fwdf))


DUMP_BYTES = 32 << 20          # what --dump-outputs writes at most


def dump_outputs(path, red, sol, aux, first):
    """Writes what one step returned to its caller as path/<name>.npy, all float64: the reduced row `reduced` [sum loss |
    sum dL/dtheta | failed OCPs], every OCP's status / iters / kkt / cost / loss / dtheta / aux_status / counters, and the
    trajectories X, U, Lam, Xa, Ua of a fixed seeded sample of the OCPs, as many as DUMP_BYTES leaves room for; `sample_index`
    holds the sample's global problem indices (`first` = index of this shard's first OCP)."""
    import torch
    B = int(aux["loss"].shape[0])
    whole = {"reduced": red, **{k: sol[k] for k in ("status", "iters", "kkt", "cost")},
             **{k: aux[k] for k in ("loss", "dtheta", "aux_status", "counters")}}
    traj = {**{k: sol[k] for k in ("X", "U", "Lam")}, **{k: aux[k] for k in ("Xa", "Ua")}}
    per_ocp = 8 * (1 + sum(v[0].numel() for v in traj.values()))
    k = min(B, (DUMP_BYTES - 8 * sum(v.numel() for v in whole.values())) // per_ocp)
    assert k > 0, "--dump-outputs: the per-OCP results of %d OCPs alone exceed %d bytes" % (B, DUMP_BYTES)
    idx = np.sort(np.random.default_rng(0).choice(B, k, replace=False))
    sel = torch.from_numpy(idx).to(red.device)
    out = {name: v.cpu().numpy() for name, v in whole.items()}
    out.update({name: v.index_select(0, sel).cpu().numpy() for name, v in traj.items()})
    out["sample_index"] = first + idx
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(v, dtype=np.float64))


def run_ours(a):
    import torch
    import torch.distributed as dist
    import lfsd_b200
    from lfsd_b200 import standard, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its "NCCL version ..." banner to stdout while the communicator
        # is created, so file descriptor 1 points at stderr until that has happened
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    B_total = a.batch * world if a.scaling == "weak" else a.batch
    lo, hi = synthetic.shard_bounds(B_total, world, rank)
    Bl = hi - lo

    oc = standard.quadrotor_oc(n_grid=a.n_grid)
    lib = oc.build(name=oc.lib_name)
    mode = a.mode or ("bdf" if hasattr(lib.L, "cpdp_has_bdf") else "rk45")
    oc.aux_mode = oc.MODE_BDF if mode == "bdf" else oc.MODE_RK45
    oc.rtol_back, oc.atol_back = a.rtol, a.atol
    qb = synthetic.quad_batch(B_total)
    # pinned host buffers (the e2e leg copies them every step)
    host = {k: torch.from_numpy(np.ascontiguousarray(qb[k][lo:hi])).pin_memory() for k in ("x0", "goal", "wp")}
    host["taus"] = torch.from_numpy(qb["taus"]).pin_memory()
    host["theta"] = torch.from_numpy(qb["theta"]).pin_memory()
    h2d_bytes = sum(v.numel() * 8 for v in host.values())
    resident = {k: v.to(dev) for k, v in host.items()}
    r = oc.n_auxvar
    gathered = torch.empty((B_total, r + 2), dtype=torch.float64, device=dev)
    result_host = torch.empty((r + 2,), dtype=torch.float64).pin_memory()
    stats = {}

    def step(inp):
        if a.chunks > 1:
            # two halves of the shard on two streams, fixed number of Newton rounds (no host synchronisation): the tails
            # of one half's kernels overlap the other half's work; results are bit-identical to the single-stream path
            _, sol, aux = oc.gradIterBatch(inp["x0"], 1.0, inp["theta"], inp["taus"], inp["wp"], qb["sel"], pdata=inp["goal"],
                                           rounds=a.rounds, chunks=a.chunks)
        else:
            sol = oc.cocSolverBatch(inp["x0"], 1.0, inp["theta"], pdata=inp["goal"])
            aux = oc.auxSysSolverBatch(sol, inp["taus"], inp["wp"], qb["sel"])
        stats["rounds"] = lib.last_rounds()
        rows = oc.packRows(sol, aux)                        # [loss | dL/dtheta | failed] per OCP, packed on the device
        if world > 1:
            dist.all_gather_into_tensor(gathered, rows)     # the single exchange of the iteration (72 B / OCP)
            allrows = gathered
        else:
            allrows = rows
        red = oc.reduceRows(allrows)                        # [sum loss | sum dL/dtheta | number of failed OCPs]
        return red, sol, aux

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        red, sol, aux = step(resident)
    sync_all()

    # ---- timed region 1: inputs resident in HBM ------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ph = []
    sync_all()
    ev[0].record()
    for _ in range(a.steps):
        red, sol, aux = step(resident)
    ev[1].record()
    sync_all()
    ms = ev[0].elapsed_time(ev[1])
    clocks = sampler.stop() if rank == 0 else None
    red_t, sol_t, aux_t = red, sol, aux
    # ---- phase times (single stream, each phase alone; explains `value`, is not part of it) -------------------------
    for _ in range(3):                                    # untimed: allocates the single-stream workspace, warms the caches
        s0 = oc.cocSolverBatch(resident["x0"], 1.0, resident["theta"], pdata=resident["goal"])
        oc.auxSysSolverBatch(s0, resident["taus"], resident["wp"], qb["sel"])
    sync_all()
    for _ in range(a.steps):
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        sol = oc.cocSolverBatch(resident["x0"], 1.0, resident["theta"], pdata=resident["goal"])
        e1.record()
        aux = oc.auxSysSolverBatch(sol, resident["taus"], resident["wp"], qb["sel"], phases=1)     # backward kernel alone
        e2.record()
        aux = oc.auxSysSolverBatch(sol, resident["taus"], resident["wp"], qb["sel"], phases=2, out=aux)
        rows = oc.packRows(sol, aux)
        if world > 1:
            dist.all_gather_into_tensor(gathered, rows)
            allrows = gathered
        else:
            allrows = rows
        red = oc.reduceRows(allrows)
        e3.record()
        ph.append((e0, e1, e2, e3))
    sync_all()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    solve_ms = float(np.median([p[0].elapsed_time(p[1]) for p in ph]))
    back_ms = float(np.median([p[1].elapsed_time(p[2]) for p in ph]))
    fwd_ms = float(np.median([p[2].elapsed_time(p[3]) for p in ph]))
    rounds = lib.last_rounds()

    # ---- timed region 2: end to end through the public API with HOST buffers ---------------------------------
    sync_all()
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev2[0].record()
    for _ in range(a.steps):
        inp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        red, sol, aux = step(inp)
        result_host.copy_(red, non_blocking=True)
        torch.cuda.current_stream().synchronize()          # the caller consumes loss / gradient on the host
    ev2[1].record()
    sync_all()
    t2 = torch.tensor([ev2[0].elapsed_time(ev2[1])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    ms_e2e = float(t2.item())

    # ---- FP64 pipe peak, measured on this GPU (MEASURED_PEAKS.json has no fp64 entry) --------------------------
    peak_tf = None
    if rank == 0:
        best = 1e30
        for _ in range(4):
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            fl = oc.fp64PeakProbe(148 * 8, 100000)
            p1.record()
            torch.cuda.synchronize()
            best = min(best, p0.elapsed_time(p1))
        peak_tf = fl / (best / 1e3) / 1e12

    # ---- statistics -----------------------------------------------------------------------------------------
    status = sol["status"].cpu().numpy()
    iters = sol["iters"].cpu().numpy()
    cnt = aux["counters"].cpu().numpy().astype(np.int64)
    loc = torch.tensor([float(iters.sum()), float((status != 1).sum()), float((aux["aux_status"] != 0).sum().item())]
                       + [float(x) for x in cnt.sum(0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(loc)
    loc = loc.cpu().numpy()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    info = oc.codegen_info
    fm = flop_model(info, oc.n_state, oc.n_control, r, a.n_grid, oc.steps_per_grid, loc[0], B_total, loc[3:9], mode)
    step_s = ms / a.steps / 1e3
    value = B_total * a.steps / (ms / 1e3)
    nominal_tf = 148 * 64 * 2 * 1.965e9 / 1e12
    # roofline of the dominant kernel: the backward Riccati sweep (one launch per step, timed alone with CUDA events)
    kname = "k_riccati_bdf" if mode == "bdf" else "k_riccati_rk45"
    dom_flops = fm["aux_backward"] / world
    achieved_tf = dom_flops / (back_ms / 1e3) / 1e12
    mp = {}
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # DRAM traffic of the dominant kernel: taken from the committed `ncu --set full` capture of the same launch shape
    # (profiles/r01_ncu_<kernel>.json, written by tools/ncu_summary.py); null when no capture of this shape exists.
    traffic, traffic_src = None, None
    try:
        pname = "r02_ncu_%s.json" % kname if os.path.exists(os.path.join(ROOT, "profiles", "r02_ncu_%s.json" % kname)) else "r01_ncu_%s.json" % kname
        prof = json.load(open(os.path.join(ROOT, "profiles", pname)))
        if prof.get("batch") == Bl and prof.get("n_grid") == a.n_grid:
            traffic = prof["dram_bytes_read"] + prof["dram_bytes_write"]
            traffic_src = "profiles/" + pname
    except Exception:
        pass
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%d quadrotor OCPs%s (n=13,m=4,r=7), n_grid 50, S=4, T=1, shared theta0, "
                               "rng default_rng(20210308); SURVEY.md 8d / BASELINE.json configs[4]" % (
                                   a.batch, " per GPU (weak scaling)" if a.scaling == "weak" else " in total, sharded contiguously over the GPUs (strong scaling)"),
                   "n_grid": a.n_grid, "global_batch": B_total, "aux_mode": mode, "rtol_back": a.rtol, "atol_back": a.atol,
                   "parallelism": "dp%d contiguous shards, all-gather of per-OCP (loss,dtheta) rows + fixed-tree sum" % world,
                   "streams": "%d chunk(s) of each shard on separate CUDA streams, %s" % (
                       a.chunks, ("%d Newton rounds per solve, no host sync" % a.rounds) if a.chunks > 1 else "adaptive Newton rounds"),
                   "l2": "inputs larger than L2: per-step working set (~%.1f GB workspace + outputs) exceeds the 126 MB L2, "
                         "every step starts from the zero seed" % (lib.workspace_bytes(Bl, a.n_grid, 4) / 1e9)},
        "e2e": {"value": B_total * a.steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": (r + 2) * 8},
        # timed region: per chunk k_solve_init + k_compact + 4 kernels per Newton round + backward + forward sweep, then
        # k_pack_rows + k_reduce_rows (single-stream mode launches only the rounds the adaptive solve needed)
        "gpu_launches": a.steps * ((a.chunks * (2 + 4 * a.rounds + 2) + 2) if a.chunks > 1 else (2 + 4 * rounds + 2 + 2)),
        "clocks": clocks,
        "roofline": {"bound": "fp64", "kernel": kname, "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved_tf / peak_tf if peak_tf else None, "traffic": traffic, "traffic_source": traffic_src,
                     "kernel_ms": back_ms,
                     "note": "dominant kernel = backward Riccati sweep, one launch per step, timed alone with CUDA events; "
                             "achieved = executed useful fp64 flops of that launch (DESIGN.md flop model x the rhs / step / LU "
                             "counters the kernel records) / its duration; peak = DFMA throughput measured in this run with "
                             "cpdp_dfma_probe (nominal 148 SM x 64 lanes x 2 x 1.965 GHz = %.1f TFLOP/s); the path is "
                             "fp64-compute/latency bound, not HBM bound: see hbm_gbs" % nominal_tf,
                     "whole_step": {"achieved": fm["total"] / world / step_s / 1e12,
                                    "frac": (fm["total"] / world / step_s / 1e12 / peak_tf) if peak_tf else None},
                     "hbm_gbs": {"achieved": (traffic / (back_ms / 1e3) / 1e9) if traffic else None, "peak": mp.get("hbm_gbs")},
                     "flops_per_step": fm,
                     "phase_ms": {"solve": solve_ms, "aux_backward": back_ms, "aux_forward_loss_reduce": fwd_ms}},
        "stats": {"newton_iters_mean": loc[0] / B_total, "newton_rounds": rounds, "not_converged": int(loc[1]),
                  "aux_failed": int(loc[2]), "back_rhs_mean": loc[3] / B_total, "back_steps_mean": loc[4] / B_total,
                  "fwd_rhs_mean": loc[5] / B_total, "fwd_steps_mean": loc[6] / B_total,
                  "back_lu_mean": loc[7] / B_total, "back_jac_mean": loc[8] / B_total,
                  "loss_sum": float(red[0].item()), "failed_ocps_in_reduced_row": int(round(float(red[-1].item())))},
    }
    # a step that averaged failed problems into its gradient is not a valid measurement (fixed Newton rounds that are too few
    # would leave problems `running`; the count travels with the reduced row, see cpdp_pack_rows)
    out["valid"] = (int(loc[1]) == 0 and int(loc[2]) == 0 and out["stats"]["failed_ocps_in_reduced_row"] == 0)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, red_t, sol_t, aux_t, lo)
    if world == 1 and not a.no_cpu_baseline:
        cb, _, _ = cpu_baseline(a.n_grid, a.cpu_sample, deadline_s=a.cpu_deadline)
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import lfsd_b200  # noqa: F401
    # every step = a bounded sample of the workload, sized so that --steps of them end within the deadline: the port needs
    # about PORT_S_PER_OCP core-seconds per OCP, so a step may hold  cores * deadline / (steps * PORT_S_PER_OCP)  OCPs
    cores = os.cpu_count() or 1
    sample = a.cpu_sample or max(cores, min(4 * cores, int(cores * 0.8 * a.cpu_deadline / (max(a.steps + a.warmup, 1) * PORT_S_PER_OCP))))
    cb, dt, steps = cpu_baseline(a.n_grid, sample, steps=a.steps, warmup=0, deadline_s=a.cpu_deadline)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
           "warmup": a.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": a.scaling,
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%d quadrotor OCPs per step (bounded sample: the first indices of the seeded 4096-OCP batch), n_grid %d"
                                  % (cb["sample_ocps"], a.n_grid),
                      "note": "the reference's CasADi/IPOPT path cannot run in this image (no casadi); this is the numpy/scipy port of "
                              "the same algorithm (kind 'port'): its speed relative to CasADi's C++ VM + IPOPT/MUMPS is unknown"},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
