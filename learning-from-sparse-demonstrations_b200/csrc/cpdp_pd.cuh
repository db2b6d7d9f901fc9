// Adjoint of mode 2 with respect to the per-problem constants pdata (cpdp_aux_adjoint_pd, DESIGN.md §3.11).  In the KKT system of the
// RK4 multiple-shooting NLP the NQ constants enter exactly as theta does, so they ride along as NQ extra parameter columns of the
// mode-2 adjoint launch sequence instead of a second pass:
//     k_disc_select, k_stage_adjoint, k_stage_hessian      unchanged
//     k_stage_theta_pd      k_stage_theta + NQ threads per interval (ModelPd::dir_pd): E^pd = dF_k/dpd, H^pd
//     k_aux_discrete_pd     phase 1 of k_aux_discrete with NQ more columns: K, Kth and K^pd; W^pd starts at hxp
//     k_aux_adjoint_pd      k_aux_adjoint, lane l owning column l of [theta | pdata]:  pdata_bar += K^pd' g + E^pd' p
// The derivatives with respect to pdata come from the companion header model_<name>_pd.cuh (struct ModelPd, codegen.py
// generate_pdata_header), passed as -DCPDP_PD_HEADER.  The kernels are templates on ModelPd, so a library instantiates them only
// when the model has constants and NZ + NP + NQ <= 32 (the columns fit the idle lanes and threads of the existing kernels).
#pragma once
#include "cpdp_adj.cuh"
#ifdef CPDP_PD_HEADER
#include CPDP_PD_HEADER
#endif

namespace CPDP_NS {

// ------------------------------------------------------------------------------------------------
// k_stage_theta_pd: k_stage_theta (cpdp_disc.cuh) with NZ + NP + NQ threads per interval.  Threads j < NZ + NP do exactly what they
// do there; thread NZ + NP + q propagates column q of d(stage state)/dpd with PM::dir_pd the same way and writes E^pd, H^pd.
// ------------------------------------------------------------------------------------------------
template <class PM>
CPDP_GLOBAL void __launch_bounds__(THETA_THREADS) k_stage_theta_pd(SolveArgs a, DiscWs d, PdWs pw) {
    constexpr int XQ = PM::NQ;
    constexpr int NZPQ = NZ + NP + XQ;
    constexpr int TPCQ = THETA_THREADS / NZPQ;
    static_assert(TPCQ >= 1, "k_stage_theta_pd: a CTA must hold the NZ + NP + NQ columns of one interval");
    CPDP_SHARED double s_x[TPCQ][NX];
    CPDP_SHARED double s_mu[TPCQ][NX];
    CPDP_SHARED double s_u[TPCQ][NU];
    CPDP_SHARED double s_th[TPCQ][NP];
    CPDP_SHARED double s_pd[TPCQ][NQT > 0 ? NQT : 1];
    CPDP_SHARED double s_S[TPCQ][NZ][NX];          // state rows of the NZ (x,u) sensitivity columns at the current stage
    CPDP_SHARED int s_gi[TPCQ];                     // global interval index b*N+k of each slot, -1 if none
    const int tid = threadIdx.x;
    const int kk = tid / NZPQ, j = tid % NZPQ;
    const int kc = kk < TPCQ ? kk : 0;
    const bool zcol = j < NZ;                      // (x,u) column j, else theta column j - NZ
    const bool qcol = j >= NZ + NP;                // pdata column j - NZ - NP
    const int total = *a.nact * a.N;
    const int ngroups = (total + TPCQ - 1) / TPCQ;
    const double DT = a.T / a.N / a.S;
    const double bco[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
    const double aco[4] = {0.0, 0.5, 0.5, 1.0};
    const int nstage = 4 * a.S;

    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
        __syncthreads();
        for (int t = tid; t < TPCQ; t += THETA_THREADS) {
            const int li = grp * TPCQ + t;
            s_gi[t] = (li < total) ? a.act[li / a.N] * a.N + li % a.N : -1;
        }
        __syncthreads();
        for (int t = tid; t < TPCQ * (NU + NP + NQ); t += THETA_THREADS) {
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
            for (int t = tid; t < TPCQ; t += THETA_THREADS) if (s_gi[t] >= 0) s_pd[t][NQ] = grid_time(a.T, a.N, s_gi[t] % a.N);
        }
        const bool mine = (kk < TPCQ) && (s_gi[kc] >= 0);
        const int gi = mine ? s_gi[kk] : -1;

        double Sx[NX], Sn[NX], dX[NX], df[NX], du[NU], dth[NP], hz[NZ], Hc[NZ];
        for (int i = 0; i < NX; ++i) { Sx[i] = (zcol && i == j) ? 1.0 : 0.0; df[i] = 0.0; }
        for (int i = 0; i < NU; ++i) du[i] = (zcol && NX + i == j) ? 1.0 : 0.0;
        for (int i = 0; i < NP; ++i) dth[i] = (!zcol && NZ + i == j) ? 1.0 : 0.0;
        double dpd[XQ];
        for (int i = 0; i < XQ; ++i) dpd[i] = (NZ + NP + i == j) ? 1.0 : 0.0;
        for (int i = 0; i < NZ; ++i) Hc[i] = 0.0;

        for (int s = 0; s < a.S; ++s) {
            for (int i = 0; i < NX; ++i) Sn[i] = Sx[i];
            for (int st = 0; st < 4; ++st) {
                const int sidx = s * 4 + st;
                __syncthreads();                   // the previous stage's readers of s_x, s_mu and s_S are done
                for (int t = tid; t < TPCQ * 2 * NX; t += THETA_THREADS) {
                    const int q = t % TPCQ, e = t / TPCQ;
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
                    } else {
                        if (qcol) PM::dir_pd(s_x[kc], s_u[kc], s_th[kc], s_pd[kc], s_mu[kc], bco[st] * DT, dX, du, dpd, df, hz);
                        else Model::dir_th(s_x[kc], s_u[kc], s_th[kc], s_pd[kc], s_mu[kc], bco[st] * DT, dX, du, dth, df, hz);
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
            const int q = j - NZ - NP;
            double* E = pw.Epd + (size_t)gi * NX * XQ;
            for (int i = 0; i < NX; ++i) E[i * XQ + q] = Sx[i];
            double* Ht = pw.Hpd + (size_t)gi * NZ * XQ;
            for (int i = 0; i < NZ; ++i) Ht[i * XQ + q] = Hc[i];
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
// k_aux_discrete_pd: phase 1 of k_aux_discrete (cpdp_disc.cuh) with NQ more columns of G = [A B | E | E^pd] and Q riding along:
// W^pd starts at hxp = d(grad_x h)/dpd and the gains K^pd go to pw.Kpd.  Every other column's arithmetic is that of k_aux_discrete.
// ------------------------------------------------------------------------------------------------
template <class PM>
CPDP_GLOBAL void __launch_bounds__(DISC_THREADS) k_aux_discrete_pd(AuxArgs x, SolveArgs a, DiscWs d, PdWs pw) {
    constexpr int XQ = PM::NQ;
    const int b = blockIdx.x, lane = threadIdx.x;
    if (x.aux_status[b] != 0) return;
    constexpr int DCOLQ = NZ + NP + XQ;             // columns of [A B | E | E^pd] and [Q | Qtheta | Qpd]
    constexpr int DCSQ = DCOLQ | 1;                  // odd row strides (conflict-free row reads by lane)
    constexpr int NPSQ = (NP + XQ) | 1;
    const int N = a.N;
    const size_t ib = (size_t)b * N;
    CPDP_SHARED double s_V[NX * NXS], s_W[NX * NPSQ], s_G[NX * DCSQ], s_Y[NX * DCSQ], s_Q[NZ * DCSQ], s_K[NU * DCSQ];
    CPDP_SHARED double s_hxx[NX * NX], s_hxe[NX * NP], s_L[NU * NU];
    CPDP_SHARED int s_flag;
    if (lane == 0) {
        PdBuf pdb;
        const double* pd = pd_at(pdata_of(a, b), grid_time(a.T, N, N), pdb);
        Model::term2(a.X + ((size_t)b * (N + 1) + N) * NX, theta_of(a, b), pd, s_hxx, s_hxe);
        PM::term2_pd(a.X + ((size_t)b * (N + 1) + N) * NX, theta_of(a, b), pd, s_G);     // hxp, parked in G
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
    for (int q = lane; q < NX * NP; q += DISC_THREADS) s_W[(q / NP) * NPSQ + q % NP] = s_hxe[q];
    for (int q = lane; q < NX * XQ; q += DISC_THREADS) s_W[(q / XQ) * NPSQ + NP + q % XQ] = s_G[q];     // W^pd starts at hxp
    NWT_SYNC();
    for (int k = N - 1; k >= 0; --k) {
        const double* ABg = a.AB + (ib + k) * NX * NZ;
        const double* Hg = a.H + (ib + k) * NZ * NZ;
        const double* Eg = d.E + (ib + k) * NX * NP;
        const double* Htg = d.Hth + (ib + k) * NZ * NP;
        const double* Epg = pw.Epd + (ib + k) * NX * XQ;
        const double* Hpg = pw.Hpd + (ib + k) * NZ * XQ;
        for (int c = lane; c < DCOLQ; c += DISC_THREADS) {
            NWT_UNROLL for (int e = 0; e < NX; ++e)
                s_G[e * DCSQ + c] = (c < NZ) ? ABg[e * NZ + c] : (c < NZ + NP) ? Eg[e * NP + c - NZ] : Epg[e * XQ + c - NZ - NP];
        }
        NWT_SYNC();
        for (int c = lane; c < DCOLQ; c += DISC_THREADS) {
            double y[NX];
            NWT_UNROLL for (int i = 0; i < NX; ++i) y[i] = (c < NZ) ? 0.0 : s_W[i * NPSQ + c - NZ];
            nwt_mac<NX>(s_V, NXS, s_G + c, DCSQ, NX, y);                    // (V symmetric: row e of V is column e)
            NWT_UNROLL for (int i = 0; i < NX; ++i) s_Y[i * DCSQ + c] = y[i];
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
            nwt_mac<NZ>(s_G, DCSQ, s_Y + c, DCSQ, NX, q);                    // (my own column of Y: no barrier needed)
            NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) s_Q[r_ * DCSQ + c] = q[r_];
        }
        NWT_SYNC();
        if (lane == 0) {
            for (int r_ = 0; r_ < NU; ++r_)
                for (int c = 0; c < NU; ++c)
                    s_L[r_ * NU + c] = 0.5 * (s_Q[(NX + r_) * DCSQ + NX + c] + s_Q[(NX + c) * DCSQ + NX + r_]);
            if (!chol_inplace<NU>(s_L)) s_flag = 1;
        }
        NWT_SYNC();
        if (s_flag) break;
        // gain columns: c < NX feedback (Qux symmetrised), c >= NZ feed-forward
        for (int c = lane; c < DCOLQ; c += DISC_THREADS) {
            if (c >= NX && c < NZ) continue;
            double rhs[NU];
            NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_)
                rhs[r_] = (c < NX) ? 0.5 * (s_Q[(NX + r_) * DCSQ + c] + s_Q[c * DCSQ + NX + r_]) : s_Q[(NX + r_) * DCSQ + c];
            chol_solve<NU>(s_L, rhs);
            NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) {
                s_K[r_ * DCSQ + c] = -rhs[r_];
                if (c < NX) a.Kf[(ib + k) * NU * NX + r_ * NX + c] = -rhs[r_];
                else if (c < NZ + NP) d.Kth[(ib + k) * NU * NP + r_ * NP + c - NZ] = -rhs[r_];
                else pw.Kpd[(ib + k) * NU * XQ + r_ * XQ + c - NZ - NP] = -rhs[r_];
            }
        }
        NWT_SYNC();
        // V = Qxx + Qxu K (exactly symmetric, as in k_newton_step), W = Qx,theta + Qxu Kth
        for (int c = lane; c < DCOLQ; c += DISC_THREADS) {
            if (c >= NX && c < NZ) continue;
            double vnew[NX];
            NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) {
                if (c < NX) {
                    const double acc = 0.5 * (s_Q[r_ * DCSQ + c] + s_Q[c * DCSQ + r_]);
                    double a1 = 0.0, a2 = 0.0;
                    NWT_UNROLL for (int e = 0; e < NU; ++e) {
                        a1 += 0.5 * (s_Q[r_ * DCSQ + NX + e] + s_Q[(NX + e) * DCSQ + r_]) * s_K[e * DCSQ + c];
                        a2 += 0.5 * (s_Q[c * DCSQ + NX + e] + s_Q[(NX + e) * DCSQ + c]) * s_K[e * DCSQ + r_];
                    }
                    vnew[r_] = acc + 0.5 * (a1 + a2);
                } else {
                    double acc = s_Q[r_ * DCSQ + c];
                    NWT_UNROLL for (int e = 0; e < NU; ++e)
                        acc += 0.5 * (s_Q[r_ * DCSQ + NX + e] + s_Q[(NX + e) * DCSQ + r_]) * s_K[e * DCSQ + c];
                    vnew[r_] = acc;
                }
            }
            // (every read of the old V and W of this stage lies before the barriers above)
            if (c < NX) { NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) s_V[r_ * NXS + c] = vnew[r_]; }
            else { NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) s_W[r_ * NPSQ + c - NZ] = vnew[r_]; }
        }
        NWT_SYNC();
    }
    if (s_flag && lane == 0) x.aux_status[b] = 4;
}

template <class PM>
CPDP_GLOBAL void __launch_bounds__(ADJ_THREADS) k_aux_adjoint_pd(AuxArgs x, SolveArgs a, DiscWs d, AdjArgs j, PdWs pw,
                                                                 double* pdata_bar) {
    adjoint_body<PM>(x, a, d, j, pw, pdata_bar);
}

}  // namespace CPDP_NS
