"""Generates parity fixtures with the CPU oracle (oracle/cpdp_oracle.py), which is itself pinned against the
reference's stored run (tests/test_oracle_kat.py).  Run from the repo root:  python tests/golden/make_oracle_fixtures.py
Output: tests/golden/oracle_<case>.npz with the converged trajectory and the loss / gradient under
  asshipped : BDF backward (scipy defaults) + RK45 forward (defaults)   = what the reference's COCSys computes
  rk45      : RK45 backward (defaults) + RK45 forward (defaults)
  tight     : rtol 1e-10 / atol 1e-12 both sweeps
  asshipped_cj : as shipped, but scipy's BDF is handed the closed-form Jacobian instead of its finite-difference one
  asshipped_ra : as shipped (finite-difference Jacobian), Riccati RHS evaluated with a different association of the
                 same products -> |dl_asshipped_ra - dl_asshipped| is the reference's own roundoff reproducibility band
"""
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import lfsd_b200  # noqa: E402,F401
from lfsd_b200 import synthetic  # noqa: E402
from oracle import models  # noqa: E402
from oracle.cpdp_oracle import Oracle, TIGHT, OracleIntegrationError  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def run_problem(args):
    kind, n_grid, x0, T, theta, pd, taus, wp = args
    mdl = getattr(models, kind)()
    orc = Oracle(mdl, n_grid=n_grid)
    variants = (('asshipped', {'method': 'BDF'}, {}), ('rk45', {}, {}), ('tight', TIGHT, TIGHT),
                ('asshipped_cj', {'method': 'BDF', 'jac': 'closed'}, {}),
                ('asshipped_ra', {'method': 'BDF', 'reassoc': True}, {}))
    if orc.tv:      # COCSys_TimeVarying integrates both sweeps with solve_ivp's default RK45 (CPDP.py:740,773)
        variants = (('asshipped', {}, {}), ('rk45', {}, {}), ('tight', TIGHT, TIGHT))
    if pd is not None:
        orc.pd = np.asarray(pd, dtype=float)
    tg, X, U, Lam, info = orc.solve(x0, T, theta, return_info=True)
    out = dict(X=X, U=U, Lam=Lam, iters=info['iters'], J=info['J'], kkt=info['kkt'])
    for tag, back, fwd in variants:
        try:
            Xa, Ua, PW, cnt = orc.aux(tg, X, U, Lam, theta, back=back, fwd=fwd, return_counts=True)
        except OracleIntegrationError as e:      # solve_ivp gave up (the reference would crash here): record it
            print('FAILED VARIANT', kind, n_grid, np.asarray(theta), tag, e, flush=True)
            n, m, r = orc.n, orc.m, orc.r
            Xa = np.full((n_grid + 1, n * r), np.nan); Ua = np.full((n_grid + 1, m * r), np.nan)
            PW = np.full((n_grid + 1, n * n + n * r), np.nan); cnt = dict(back_rhs=-1, fwd_rhs=-1)
        loss, dl = orc.loss_grad(taus, wp, tg, X, Xa)
        out['ok_' + tag] = bool(np.isfinite(Xa).all())
        out['loss_' + tag] = loss; out['dl_' + tag] = dl
        if tag == 'asshipped_ra':
            continue
        out['Xa_' + tag] = Xa; out['Ua_' + tag] = Ua
        out['cnt_' + tag] = np.array([cnt['back_rhs'], cnt['fwd_rhs']])
        if tag == 'asshipped':
            out['PW_asshipped'] = PW
    return out


def stack(results):
    return {k: np.stack([np.asarray(r[k]) for r in results]) for k in results[0]}


def shrink_quad50(d):
    """Keeps oracle_quad50.npz under 1 MB: no test reads the Riccati nodes PW, and the sensitivity trajectories Xa / Ua are
    stored in float32 (rounding <= 6e-8 relative; the tests hold them to 1e-5)."""
    d.pop('PW_asshipped')
    for k in [k for k in d if k.startswith(('Xa_', 'Ua_'))]:
        d[k] = d[k].astype(np.float32)


def main():
    t0 = time.time()
    jobs = {}
    # pendulum, as in Examples/pendulum_groundtruth.py: waypoints from theta*=[2,1,1] at grid idx [1,3,6,7,9]
    mdl = models.pendulum(); orc = Oracle(mdl, n_grid=10)
    tg, Xs, _, _ = orc.solve([0.0, 0.0], 1.0, [2.0, 1.0, 1.0])
    idx = [1, 3, 6, 7, 9]
    p_taus, p_wp = tg[idx], Xs[idx, 0:1]
    jobs['pendulum'] = [('pendulum', 10, np.zeros(2), 1.0, np.array(th), None, p_taus, p_wp)
                        for th in ([1.0, 0.5, 1.5], [2.0, 1.0, 1.0], [1.3, 0.8, 1.2])]
    ab = synthetic.robotarm_batch(4)
    jobs['robotarm'] = [('robotarm', 30, ab['x0'][b], 1.0, ab['theta'][b], None, ab['taus'], ab['wp'][b]) for b in range(4)]
    jobs['robotarm'][0] = ('robotarm', 30, ab['x0'][0], 1.0, np.array([5.0, 1, 1, 1, 1]), None, ab['taus'], ab['wp'][0])
    rb = synthetic.rocket_batch(2)
    mdl = models.rocket(); orc = Oracle(mdl, n_grid=15)
    rjobs = []
    for b in range(2):
        tg, Xs, _, _ = orc.solve(rb['x0'][b], 3.0, rb['theta_true'])
        rjobs.append(('rocket', 15, rb['x0'][b], 3.0, rb['theta0'], None, tg[rb['tau_idx']], Xs[rb['tau_idx']][:, rb['sel']]))
    jobs['rocket'] = rjobs
    # Examples/pendulum_timewarping.py:60-68 (T = 0.2, five waypoints) with the second-order time-warping polynomial
    tw_T = 0.2
    tw_taus = np.array([0.1, 0.3, 0.6, 0.7, 0.9]) / 1 * tw_T
    tw_wp = np.array([[0.5], [1.8], [2.0], [2.9], [3.1]])
    jobs['pendulum_tw2'] = [('pendulum_timewarp', 10, np.zeros(2), tw_T, np.array(th), None, tw_taus, tw_wp)
                            for th in ([1.0, 1.0, 1.0, 1.0], [2.5, 0.7, 0.8, 1.3], [4.0, -1.5, 1.2, 0.6])]
    qb = synthetic.quad_batch(4096)
    jobs['quad50'] = [('quadrotor', 50, qb['x0'][b], 1.0, qb['theta'], qb['goal'][b], qb['taus'], qb['wp'][b]) for b in range(6)]
    g = np.load(os.path.join(HERE, 'quad_run.npz'))
    jobs['quadkat'] = [('quadrotor', 25, g['ini_state'], 1.0, g['parameter_trace'][0], g['goal_position'], g['time_grid'], g['waypoints'])]
    # BASELINE configs[3]: Examples/quad_example.py:31-57 as scripted (start [0,0,.6], goal [3,3,1.5], five waypoints at
    # tau = [1..5]/6 after the learner's normalisation, lib/QuadAlgorithm.py:221-223; n_grid 25; theta0 of :235)
    jobs['quadexample'] = [('quadrotor', 25, np.array([0, 0, 0.6, 0, 0, 0, 1.0, 0, 0, 0, 0, 0, 0]), 1.0,
                            np.array([1, 0.1, 0.1, 0.1, 0.1, 0.1, -1.0]), np.array([3.0, 3.0, 1.5]),
                            np.array([1.0, 2.0, 3.0, 4.0, 5.0]) / 6,
                            np.array([[0.5, 0.5, 0.6], [1.0, 1.0, 0.8], [1.5, 1.5, 1.0], [2.0, 2.0, 1.2], [2.5, 2.5, 1.5]]))]
    only = [a for a in sys.argv[1:] if not a.startswith('-')]
    if only:
        jobs = {k: v for k, v in jobs.items() if k in only}
    flat = [(name, j) for name, lst in jobs.items() for j in lst]
    with Pool(min(8, os.cpu_count())) as pool:
        res = pool.map(run_problem, [j for _, j in flat], chunksize=1)
    for name in jobs:
        rs = [r for (nm, _), r in zip(flat, res) if nm == name]
        js = jobs[name]
        d = stack(rs)
        d.update(x0=np.stack([j[2] for j in js]), theta=np.stack([j[4] for j in js]), T=js[0][3], n_grid=js[0][1],
                 taus=np.stack([j[6] for j in js]), wp=np.stack([j[7] for j in js]))
        if js[0][5] is not None:
            d['pdata'] = np.stack([j[5] for j in js])
        if name == 'quad50':
            shrink_quad50(d)
        np.savez_compressed(os.path.join(HERE, 'oracle_%s.npz' % name), **d)
        print(name, 'iters', d['iters'], 'loss', d['loss_asshipped'], 'time %.0fs' % (time.time() - t0))


if __name__ == '__main__':
    main()
