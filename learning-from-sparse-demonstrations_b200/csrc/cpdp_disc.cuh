// Discrete auxiliary mode (cpdp_aux mode 2): dx/dtheta, du/dtheta, the loss and dL/dtheta as the EXACT derivative of the solver's
// own output.  Differentiating the KKT conditions of the RK4 multiple-shooting NLP at the converged point (X, U, Lam) with respect
// to theta gives an equality-constrained LQR in the r columns of (dX/dtheta, dU/dtheta) (DESIGN.md §3.7):
//     min  sum_k 1/2 Z_k' H_k Z_k + Z_k' Hth_k + 1/2 X_N' hxx X_N + X_N' hxe
//     s.t. X_{k+1} = A_k X_k + B_k U_k + E_k,  X_0 = 0,          Z_k = [X_k; U_k]
// with [A B], H of the interval Lagrangian q_k + lam_{k+1}'F_k (k_stage_adjoint + k_stage_hessian, unchanged), E_k = dF_k/dtheta and
// Hth_k = d(grad_z of the interval Lagrangian)/dtheta (k_stage_theta), solved by a Riccati recursion with no regularisation
// (k_aux_discrete).  Kernels:
//   k_disc_select       active list of the problems with a usable trajectory (the others get aux_status 3), counters zeroed
//   k_stage_theta<PM>   NZ + NP + PM::NQ threads per interval: the NZ (x,u) sensitivity columns, the NP theta columns and the
//                       PM::NQ pdata columns through the 4S stages
//   k_aux_discrete<PM>  one warp per problem: phase 1 backward recursion (gains to the workspace), phase 2 rollout + loss (NoPd
//                       only: with pdata columns the kernel runs phase 1 whatever `phase` says)
// PM is NoPd (no pdata columns) for mode 2 and cpdp_aux_adjoint, ModelPd for cpdp_aux_adjoint_pd.
#pragma once
#include "cpdp_aux.cuh"

namespace CPDP_NS {

struct DiscWs {
    double* Hth;           // [B*N][NZ][NP]  d(grad_z (q_k + lam_{k+1}'F_k))/dtheta
    double* E;             // [B*N][NX][NP]  dF_k/dtheta
    double* Kth;           // [B*N][NU][NP]  feed-forward gains of the recursion (the feedback gains go to SolveArgs::Kf)
};

// The NQ per-problem constants as extra parameter columns (cpdp_aux_adjoint_pd, DESIGN.md §3.11): mode 2's three arrays for them,
// in a separate caller-provided workspace.  The kernels of mode 2 are templates on the model's pdata derivatives PM (struct ModelPd
// of the companion header, PM::NQ extra columns); NoPd (0 columns) is mode 2 and its adjoint with respect to theta and x0 alone.
struct PdWs {
    double* Hpd;           // [B*N][NZ][NQ]  d(grad_z (q_k + lam_{k+1}'F_k))/dpd
    double* Epd;           // [B*N][NX][NQ]  dF_k/dpd
    double* Kpd;           // [B*N][NU][NQ]  feed-forward gains
};
struct NoPd { static constexpr int NQ = 0; };

CPDP_HD bool disc_usable(const int* solve_status, int b) {
    return !solve_status || (solve_status[b] != ST_NUMERIC && solve_status[b] != ST_RUNNING &&
                             !(HAS_BOUNDS && solve_status[b] == ST_INFEASIBLE));
}

// k_disc_select: ordered list of the problems with a usable trajectory (single CTA, as k_compact); aux_status 0 / 3, counters 0.
CPDP_GLOBAL void __launch_bounds__(COMPACT_THREADS) k_disc_select(AuxArgs x, SolveArgs a) {
    CPDP_SHARED int s_cnt[COMPACT_THREADS + 1];
    const int tid = threadIdx.x;
    const int chunk = (a.B + COMPACT_THREADS - 1) / COMPACT_THREADS;
    const int lo = tid * chunk, hi = (lo + chunk < a.B) ? lo + chunk : a.B;
    int c = 0;
    for (int i = lo; i < hi; ++i) {
        const bool ok = disc_usable(x.solve_status, i);
        c += ok;
        x.aux_status[i] = ok ? 0 : 3;
        for (int e = 0; e < NCOUNTERS; ++e) x.counters[(size_t)i * NCOUNTERS + e] = 0;
    }
    s_cnt[tid] = c;
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int i = 0; i < COMPACT_THREADS; ++i) { const int v = s_cnt[i]; s_cnt[i] = run; run += v; }
        s_cnt[COMPACT_THREADS] = run;
        *a.nact = run;
    }
    __syncthreads();
    int o = s_cnt[tid];
    for (int i = lo; i < hi; ++i) if (disc_usable(x.solve_status, i)) a.act[o++] = i;
}

// ------------------------------------------------------------------------------------------------
// k_stage_theta<PM>: NZ + NP + PM::NQ threads per (problem, interval), TPC intervals per CTA.
// Thread j < NZ propagates column j of d(stage state)/d(x_k, u_k) through the 4S stages as k_stage_hessian does and parks its stage
// rows in shared memory; thread NZ + p propagates column p of d(stage state)/dtheta (zero at the interval start) with Model::dir_th
// and accumulates column p of  Hth = sum_s Sz_s' [Hess_zz(Ham_s) [Sth_s; 0] + Hess_ztheta(Ham_s)],  Ham_s = w_s c + mu_s'f, reading
// the Sz rows of the stage.  Writes E = Sth at the interval end and Hth.  PM::NQ > 0 (the pdata columns of cpdp_aux_adjoint_pd):
// thread NZ + NP + q propagates column q of d(stage state)/dpd with PM::dir_pd the same way and writes E^pd, H^pd.
// ------------------------------------------------------------------------------------------------
#ifndef CPDP_THETA_THREADS
#define CPDP_THETA_THREADS 64
#endif
constexpr int THETA_THREADS = CPDP_THETA_THREADS;
static_assert(THETA_THREADS % 32 == 0, "k_stage_theta: whole warps");

template <class PM>
CPDP_GLOBAL void __launch_bounds__(THETA_THREADS) k_stage_theta(SolveArgs a, DiscWs d, PdWs pw) {
    constexpr int XQ = PM::NQ;
    constexpr int NZP = NZ + NP + XQ;              // threads per interval
    constexpr int TPC = THETA_THREADS / NZP;       // intervals per CTA
    static_assert(TPC >= 1, "k_stage_theta: a CTA must hold the NZ + NP + NQ columns of one interval");
    CPDP_SHARED double s_x[TPC][NX];
    CPDP_SHARED double s_mu[TPC][NX];
    CPDP_SHARED double s_u[TPC][NU];
    CPDP_SHARED double s_th[TPC][NP];
    CPDP_SHARED double s_pd[TPC][NQT > 0 ? NQT : 1];
    CPDP_SHARED double s_S[TPC][NZ][NX];          // state rows of the NZ (x,u) sensitivity columns at the current stage
    CPDP_SHARED int s_gi[TPC];                     // global interval index b*N+k of each slot, -1 if none
    const int tid = threadIdx.x;
    const int kk = tid / NZP, j = tid % NZP;
    const int kc = kk < TPC ? kk : 0;
    const bool zcol = j < NZ;                      // (x,u) column j, else theta column j - NZ
    const bool qcol = XQ > 0 && j >= NZ + NP;      // pdata column j - NZ - NP
    const int total = *a.nact * a.N;
    const int ngroups = (total + TPC - 1) / TPC;
    const double DT = a.T / a.N / a.S;
    const double bco[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
    const double aco[4] = {0.0, 0.5, 0.5, 1.0};
    const int nstage = 4 * a.S;

    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
        __syncthreads();
        for (int t = tid; t < TPC; t += THETA_THREADS) {
            const int li = grp * TPC + t;
            s_gi[t] = (li < total) ? a.act[li / a.N] * a.N + li % a.N : -1;
        }
        __syncthreads();
        for (int t = tid; t < TPC * (NU + NP + NQ); t += THETA_THREADS) {
            const int q = t / (NU + NP + NQ), e = t % (NU + NP + NQ);
            const int gi = s_gi[q];
            if (gi >= 0) {
                const int b = gi / a.N, k = gi % a.N;
                if (e < NU) s_u[q][e] = a.U[((size_t)b * (a.N + 1) + k) * NU + e];
                else if (e < NU + NP) s_th[q][e - NU] = theta_of(a, b)[e - NU];
                else s_pd[q][e - NU - NP] = pdata_of(a, b)[e - NU - NP];
            }
        }
        if (HAS_TIME) {
            for (int t = tid; t < TPC; t += THETA_THREADS) if (s_gi[t] >= 0) s_pd[t][NQ] = grid_time(a.T, a.N, s_gi[t] % a.N);
        }
        const bool mine = (kk < TPC) && (s_gi[kc] >= 0);
        const int gi = mine ? s_gi[kk] : -1;

        double Sx[NX], Sn[NX], dX[NX], df[NX], du[NU], dth[NP], hz[NZ], Hc[NZ];
        for (int i = 0; i < NX; ++i) { Sx[i] = (zcol && i == j) ? 1.0 : 0.0; df[i] = 0.0; }
        for (int i = 0; i < NU; ++i) du[i] = (zcol && NX + i == j) ? 1.0 : 0.0;
        for (int i = 0; i < NP; ++i) dth[i] = (!zcol && NZ + i == j) ? 1.0 : 0.0;
        double dpd[XQ > 0 ? XQ : 1];
        for (int i = 0; i < XQ; ++i) dpd[i] = (NZ + NP + i == j) ? 1.0 : 0.0;
        for (int i = 0; i < NZ; ++i) Hc[i] = 0.0;

        for (int s = 0; s < a.S; ++s) {
            for (int i = 0; i < NX; ++i) Sn[i] = Sx[i];
            for (int st = 0; st < 4; ++st) {
                const int sidx = s * 4 + st;
                __syncthreads();                   // the previous stage's readers of s_x, s_mu and s_S are done
                for (int t = tid; t < TPC * 2 * NX; t += THETA_THREADS) {
                    const int q = t % TPC, e = t / TPC;
                    const int g2 = s_gi[q];
                    if (g2 >= 0) {
                        if (e < NX) s_x[q][e] = a.xs[stage_off(g2, sidx, nstage, e)];
                        else s_mu[q][e - NX] = a.mu[stage_off(g2, sidx, nstage, e - NX)];
                    }
                }
                __syncthreads();
                if (mine) {
                    const double ca = aco[st] * DT;
                    for (int i = 0; i < NX; ++i) dX[i] = Sx[i] + ca * df[i];
                    if (zcol) {
                        Model::dir(s_x[kc], s_u[kc], s_th[kc], s_pd[kc], s_mu[kc], bco[st] * DT, dX, du, df, hz);
                        for (int i = 0; i < NX; ++i) s_S[kc][j][i] = dX[i];
                    } else if (qcol) {
                        if constexpr (XQ > 0)
                            PM::dir_pd(s_x[kc], s_u[kc], s_th[kc], s_pd[kc], s_mu[kc], bco[st] * DT, dX, du, dpd, df, hz);
                    } else {
                        Model::dir_th(s_x[kc], s_u[kc], s_th[kc], s_pd[kc], s_mu[kc], bco[st] * DT, dX, du, dth, df, hz);
                    }
                }
                __syncthreads();
                if (mine) {
                    if (!zcol) {
                        // Hc[i] += hz[i] (control rows) + sum_e S_i[e] hz[e]
                        for (int i = 0; i < NZ; ++i) {
                            double acc = (i >= NX) ? hz[i] : 0.0;
                            for (int e = 0; e < NX; ++e) acc += s_S[kc][i][e] * hz[e];
                            Hc[i] += acc;
                        }
                    }
                    const double cb = bco[st] * DT;
                    for (int i = 0; i < NX; ++i) Sn[i] += cb * df[i];
                }
            }
            for (int i = 0; i < NX; ++i) Sx[i] = Sn[i];
        }
        if (mine && qcol) {
            if constexpr (XQ > 0) {
                const int q = j - NZ - NP;
                double* E = pw.Epd + (size_t)gi * NX * XQ;
                for (int i = 0; i < NX; ++i) E[i * XQ + q] = Sx[i];
                double* Ht = pw.Hpd + (size_t)gi * NZ * XQ;
                for (int i = 0; i < NZ; ++i) Ht[i * XQ + q] = Hc[i];
            }
        } else if (mine && !zcol) {
            const int p = j - NZ;
            double* E = d.E + (size_t)gi * NX * NP;
            for (int i = 0; i < NX; ++i) E[i * NP + p] = Sx[i];
            double* Ht = d.Hth + (size_t)gi * NZ * NP;
            for (int i = 0; i < NZ; ++i) Ht[i * NP + p] = Hc[i];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_aux_discrete<PM>: one warp per problem (grid = B; problems with aux_status != 0 only write their zero loss row in phase 2).
// Phase 1, backward (k = N-1 .. 0), in the column style of k_newton_step: lane c owns column c of  G = [A B | E]  (NX x (NZ+NP)):
//     Y[:, c] = V G[:, c] (+ W[:, c-NZ] for the theta columns),   Q[:, c] = [H | Hth][:, c] + [A B]' Y[:, c]
//     Quu = L L' (lane 0; not positive definite -> aux_status 4),  gains  K = -Quu^{-1} Qux,  Kth = -Quu^{-1} Qu,theta
//     V <- Qxx + Qxu K (symmetrised as in k_newton_step),  W <- Qx,theta + Qxu Kth
// PM::NQ > 0: NQ more columns of G = [A B | E | E^pd] and Q ride along; W^pd starts at hxp = d(grad_x h)/dpd and the gains K^pd go
// to pw.Kpd.  Every other column's arithmetic is that of NoPd.
// Phase 2, forward: lane p < NP owns column p of dX/dtheta:  Ua_k = K Xa_k + Kth,  Xa_{k+1} = A Xa_k + B Ua_k + E_k,  Ua_N = Ua_{N-1};
// then the loss and dL/dtheta of k_aux_forward's tail (same formula, same summation order).
// ------------------------------------------------------------------------------------------------
constexpr int DISC_THREADS = 32;
static_assert(NP <= DISC_THREADS, "k_aux_discrete maps one lane per column of dX/dtheta in the rollout");

template <class PM>
CPDP_GLOBAL void __launch_bounds__(DISC_THREADS) k_aux_discrete(AuxArgs x, SolveArgs a, DiscWs d, int phase, PdWs pw) {
    constexpr int XQ = PM::NQ;
    constexpr int DCOL = NZ + NP + XQ;             // columns of [A B | E | E^pd] and [Q | Qtheta | Qpd]
    constexpr int DCS = DCOL | 1;                  // odd row strides (conflict-free row reads by lane)
    constexpr int NPS = (NP + XQ) | 1;
    const int b = blockIdx.x, lane = threadIdx.x;
    const int N = a.N;
    if (x.aux_status[b] != 0) {
        if (XQ == 0 && phase == 2) {
            if (lane == 0) x.loss[b] = 0.0;
            for (int i = lane; i < NP; i += DISC_THREADS) x.dtheta[(size_t)b * NP + i] = 0.0;
        }
        return;
    }
    const size_t ib = (size_t)b * N;
    if (XQ > 0 || phase == 1) {
        CPDP_SHARED double s_V[NX * NXS], s_W[NX * NPS], s_G[NX * DCS], s_Y[NX * DCS], s_Q[NZ * DCS], s_K[NU * DCS];
        CPDP_SHARED double s_hxx[NX * NX], s_hxe[NX * NP], s_L[NU * NU];
        CPDP_SHARED int s_flag;
        if (lane == 0) {
            PdBuf pdb;
            const double* pd = pd_at(pdata_of(a, b), grid_time(a.T, N, N), pdb);
            Model::term2(a.X + ((size_t)b * (N + 1) + N) * NX, theta_of(a, b), pd, s_hxx, s_hxe);
            if constexpr (XQ > 0) PM::term2_pd(a.X + ((size_t)b * (N + 1) + N) * NX, theta_of(a, b), pd, s_G);     // hxp, parked in G
            s_flag = 0;
        }
        NWT_SYNC();
        for (int q = lane; q < NX * NX; q += DISC_THREADS) {
            const int i = q / NX, c = q % NX;
            s_V[i * NXS + c] = 0.5 * (s_hxx[i * NX + c] + s_hxx[c * NX + i]);
            if constexpr (HAS_BOUNDS) {
                // bounded model: the barrier-perturbed KKT system adds Sigma = Z_L S_L^-1 + Z_U S_U^-1 of the final state
                if (i == c) {
                    const size_t o = ((size_t)b * (N + 1) + N) * NZ + i;
                    double sg, bg;
                    bnd_terms(i, a.X[((size_t)b * (N + 1) + N) * NX + i], a.zL[o], a.zU[o], 0.0, sg, bg);
                    s_V[i * NXS + c] += sg;
                }
            }
        }
        for (int q = lane; q < NX * NP; q += DISC_THREADS) s_W[(q / NP) * NPS + q % NP] = s_hxe[q];
        if constexpr (XQ > 0) {
            for (int q = lane; q < NX * XQ; q += DISC_THREADS) s_W[(q / XQ) * NPS + NP + q % XQ] = s_G[q];     // W^pd starts at hxp
        }
        NWT_SYNC();
        for (int k = N - 1; k >= 0; --k) {
            const double* ABg = a.AB + (ib + k) * NX * NZ;
            const double* Hg = a.H + (ib + k) * NZ * NZ;
            const double* Eg = d.E + (ib + k) * NX * NP;
            const double* Htg = d.Hth + (ib + k) * NZ * NP;
            const double* Epg = pw.Epd + (ib + k) * NX * XQ;
            const double* Hpg = pw.Hpd + (ib + k) * NZ * XQ;
            for (int c = lane; c < DCOL; c += DISC_THREADS) {
                NWT_UNROLL for (int e = 0; e < NX; ++e)
                    s_G[e * DCS + c] = (c < NZ) ? ABg[e * NZ + c] : (c < NZ + NP) ? Eg[e * NP + c - NZ] : Epg[e * XQ + c - NZ - NP];
            }
            NWT_SYNC();
            for (int c = lane; c < DCOL; c += DISC_THREADS) {
                double y[NX];
                NWT_UNROLL for (int i = 0; i < NX; ++i) y[i] = (c < NZ) ? 0.0 : s_W[i * NPS + c - NZ];
                nwt_mac<NX>(s_V, NXS, s_G + c, DCS, NX, y);                    // (V symmetric: row e of V is column e)
                NWT_UNROLL for (int i = 0; i < NX; ++i) s_Y[i * DCS + c] = y[i];
                double q[NZ];
                NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_)
                    q[r_] = (c < NZ) ? Hg[r_ * NZ + c] : (c < NZ + NP) ? Htg[r_ * NP + c - NZ] : Hpg[r_ * XQ + c - NZ - NP];
                if constexpr (HAS_BOUNDS) {
                    if (c < NZ) {                          // + Sigma_k (diagonal) of the barrier-perturbed KKT system
                        const size_t o = ((size_t)b * (N + 1) + k) * NZ + c;
                        const double w = (c < NX) ? a.X[((size_t)b * (N + 1) + k) * NX + c] : a.U[((size_t)b * (N + 1) + k) * NU + c - NX];
                        double sg, bg;
                        bnd_terms(c, w, a.zL[o], a.zU[o], 0.0, sg, bg);
                        NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) if (r_ == c) q[r_] += sg;
                    }
                }
                nwt_mac<NZ>(s_G, DCS, s_Y + c, DCS, NX, q);                    // (my own column of Y: no barrier needed)
                NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) s_Q[r_ * DCS + c] = q[r_];
            }
            NWT_SYNC();
            if (lane == 0) {
                for (int r_ = 0; r_ < NU; ++r_)
                    for (int c = 0; c < NU; ++c)
                        s_L[r_ * NU + c] = 0.5 * (s_Q[(NX + r_) * DCS + NX + c] + s_Q[(NX + c) * DCS + NX + r_]);
                if (!chol_inplace<NU>(s_L)) s_flag = 1;
            }
            NWT_SYNC();
            if (s_flag) break;
            // gain columns: c < NX feedback (Qux symmetrised), c >= NZ feed-forward
            for (int c = lane; c < DCOL; c += DISC_THREADS) {
                if (c >= NX && c < NZ) continue;
                double rhs[NU];
                NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_)
                    rhs[r_] = (c < NX) ? 0.5 * (s_Q[(NX + r_) * DCS + c] + s_Q[c * DCS + NX + r_]) : s_Q[(NX + r_) * DCS + c];
                chol_solve<NU>(s_L, rhs);
                NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) {
                    s_K[r_ * DCS + c] = -rhs[r_];
                    if (c < NX) a.Kf[(ib + k) * NU * NX + r_ * NX + c] = -rhs[r_];
                    else if (c < NZ + NP) d.Kth[(ib + k) * NU * NP + r_ * NP + c - NZ] = -rhs[r_];
                    else pw.Kpd[(ib + k) * NU * XQ + r_ * XQ + c - NZ - NP] = -rhs[r_];
                }
            }
            NWT_SYNC();
            // V = Qxx + Qxu K (exactly symmetric, as in k_newton_step), W = Qx,theta + Qxu Kth
            for (int c = lane; c < DCOL; c += DISC_THREADS) {
                if (c >= NX && c < NZ) continue;
                double vnew[NX];
                NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) {
                    if (c < NX) {
                        const double acc = 0.5 * (s_Q[r_ * DCS + c] + s_Q[c * DCS + r_]);
                        double a1 = 0.0, a2 = 0.0;
                        NWT_UNROLL for (int e = 0; e < NU; ++e) {
                            a1 += 0.5 * (s_Q[r_ * DCS + NX + e] + s_Q[(NX + e) * DCS + r_]) * s_K[e * DCS + c];
                            a2 += 0.5 * (s_Q[c * DCS + NX + e] + s_Q[(NX + e) * DCS + c]) * s_K[e * DCS + r_];
                        }
                        vnew[r_] = acc + 0.5 * (a1 + a2);
                    } else {
                        double acc = s_Q[r_ * DCS + c];
                        NWT_UNROLL for (int e = 0; e < NU; ++e)
                            acc += 0.5 * (s_Q[r_ * DCS + NX + e] + s_Q[(NX + e) * DCS + r_]) * s_K[e * DCS + c];
                        vnew[r_] = acc;
                    }
                }
                // (every read of the old V and W of this stage lies before the barriers above)
                if (c < NX) { NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) s_V[r_ * NXS + c] = vnew[r_]; }
                else { NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) s_W[r_ * NPS + c - NZ] = vnew[r_]; }
            }
            NWT_SYNC();
        }
        if (s_flag && lane == 0) x.aux_status[b] = 4;
        return;
    }

    // ---- phase 2: rollout
    const bool act = lane < NP;
    const int p = act ? lane : 0;
    double* Xa = x.Xa + (size_t)b * (N + 1) * NX * NP;
    double* Ua = x.Ua + (size_t)b * (N + 1) * NU * NP;
    double xa[NX], ua[NU];
    NWT_UNROLL for (int i = 0; i < NX; ++i) xa[i] = 0.0;
    NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) ua[r_] = 0.0;
    if (act) { NWT_UNROLL for (int i = 0; i < NX; ++i) Xa[i * NP + p] = 0.0; }
    CPDP_LOOP for (int k = 0; k < N; ++k) {
        const double* Kk = a.Kf + (ib + k) * NU * NX;
        const double* Ktk = d.Kth + (ib + k) * NU * NP;
        const double* ABg = a.AB + (ib + k) * NX * NZ;
        const double* Eg = d.E + (ib + k) * NX * NP;
        NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) {
            double acc = Ktk[r_ * NP + p];
            NWT_UNROLL for (int c = 0; c < NX; ++c) acc += Kk[r_ * NX + c] * xa[c];
            ua[r_] = acc;
        }
        double xn[NX];
        NWT_UNROLL for (int i = 0; i < NX; ++i) {
            double acc = Eg[i * NP + p];
            NWT_UNROLL for (int c = 0; c < NX; ++c) acc += ABg[i * NZ + c] * xa[c];
            NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) acc += ABg[i * NZ + NX + r_] * ua[r_];
            xn[i] = acc;
        }
        NWT_UNROLL for (int i = 0; i < NX; ++i) xa[i] = xn[i];
        if (act) {
            NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) Ua[(size_t)k * NU * NP + r_ * NP + p] = ua[r_];
            NWT_UNROLL for (int i = 0; i < NX; ++i) Xa[(size_t)(k + 1) * NX * NP + i * NP + p] = xa[i];
        }
    }
    if (act) { NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) Ua[(size_t)N * NU * NP + r_ * NP + p] = ua[r_]; }     // CPDP.py:191
#ifdef __CUDACC__
    __threadfence_block();
#endif
    NWT_SYNC();

    // ---- loss and gradient: the tail of k_aux_forward, term for term (lane 0 the loss, parameter i by lane i % 32; a waypoint
    //      time outside [0, T] gives status 5)
    const double dt = a.T / N;
    const double* Xn = a.X + (size_t)b * (N + 1) * NX;
    const double* taus = x.taus + (size_t)b * x.taus_stride;
    const double* wp = x.wp + (size_t)b * x.W * x.D;
    int st = 0;
    for (int w = 0; w < x.W; ++w) if (!(taus[w] >= 0.0 && taus[w] <= dt * N)) st = 5;
    if (st != 0 && lane == 0) x.aux_status[b] = st;
    if (lane == 0) {
        double lo_ = 0.0;
        for (int w = 0; w < x.W && st == 0; ++w) {
            const double t = taus[w];
            const int lo = interp_lo(t, dt, N);
            const double xlo = dt * lo, xhi = dt * (lo + 1);
            for (int dd = 0; dd < x.D; ++dd) {
                const int si = x.sel[dd];
                const double yv = interp_val(Xn[(size_t)lo * NX + si], Xn[(size_t)(lo + 1) * NX + si], xlo, xhi, t);
                const double diff = yv - wp[(size_t)w * x.D + dd];
                lo_ += diff * diff;
            }
        }
        x.loss[b] = lo_;
    }
    for (int i = lane; i < NP; i += DISC_THREADS) {
        double acc = 0.0;
        for (int w = 0; w < x.W && st == 0; ++w) {
            const double t = taus[w];
            const int lo = interp_lo(t, dt, N);
            const double xlo = dt * lo, xhi = dt * (lo + 1);
            for (int dd = 0; dd < x.D; ++dd) {
                const int si = x.sel[dd];
                const double yv = interp_val(Xn[(size_t)lo * NX + si], Xn[(size_t)(lo + 1) * NX + si], xlo, xhi, t);
                const double diff = yv - wp[(size_t)w * x.D + dd];
                const double xv = interp_val(Xa[(size_t)lo * NX * NP + si * NP + i], Xa[(size_t)(lo + 1) * NX * NP + si * NP + i], xlo, xhi, t);
                acc += diff * xv;
            }
        }
        x.dtheta[(size_t)b * NP + i] = acc;
    }
}

}  // namespace CPDP_NS
