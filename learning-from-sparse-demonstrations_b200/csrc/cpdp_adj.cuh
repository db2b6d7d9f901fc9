// Adjoint of mode 2 (cpdp_aux_adjoint): theta_bar = (dX/dtheta)' Xbar + (dU/dtheta)' Ubar and x0_bar = (dX/dx0)' Xbar + (dU/dx0)' Ubar
// for per-problem cotangents (Xbar, Ubar) of the trajectory, in one reverse sweep over the gains mode 2's phase 1 leaves in the
// workspace (DESIGN.md §3.9).  Phase 2 of k_aux_discrete is the linear map (dtheta, dx0) -> (dX, dU)
//     x_0 = dx0,   u_k = K_k x_k + Kth_k dtheta,   x_{k+1} = A_k x_k + B_k u_k + E_k dtheta,   u_N = u_{N-1}   (CPDP.py:191)
// (mode 2 itself runs it with dx0 = 0, one column per parameter); its transpose, one vector per problem:
//     Ubar'_{N-1} = Ubar_{N-1} + Ubar_N,   p = Xbar_N,   theta_bar = 0
//     k = N-1 .. 0:   g = Ubar'_k + B_k' p,   theta_bar += Kth_k' g + E_k' p,   p = Xbar_k + A_k' p + K_k' g
//     x0_bar = p
// The NQ per-problem constants pdata enter the KKT system exactly as theta does (cpdp_aux_adjoint_pd, DESIGN.md §3.11), so they
// ride along as NQ extra parameter columns of mode 2's phase 1 and of this sweep, PM = ModelPd of the companion header
// model_<name>_pd.cuh (codegen.py generate_pdata_header):  pdata_bar += K^pd' g + E^pd' p.  A library instantiates the kernels on
// ModelPd only when the model has constants and NZ + NP + NQ <= 32 (the columns fit the idle lanes and threads).
#pragma once
#include "cpdp_disc.cuh"

namespace CPDP_NS {

struct AdjArgs {
    const double* Xbar;    // [B][N+1][NX] or null (zero)
    const double* Ubar;    // [B][N+1][NU] or null (zero)
    double* theta_bar;     // [B][NP]
    double* x0_bar;        // [B][NX] or null
};

// ------------------------------------------------------------------------------------------------
// k_aux_adjoint<PM>: one warp per problem (grid = B).  p and g live in shared memory; lane i forms row i of A'p + K'g (rows i,
// i + 32, ...), lane j forms g_j, lane q accumulates theta_bar_q in registers.  Every global operand of stage k - 1 (the columns of
// [A B], K, Kth, E this lane contracts and its entries of Xbar, Ubar) is fetched in one batch of independent loads while stage k
// is computed.  The summation order depends on N only (no atomics): a problem's row does not depend on the batch around it.
// Rows are zero for a problem with aux_status != 0 or a solve that did not end CPDP_CONVERGED (the rule of k_pack_rows).
// ------------------------------------------------------------------------------------------------
constexpr int ADJ_THREADS = 32;
constexpr int ADJ_RX = (NX + ADJ_THREADS - 1) / ADJ_THREADS;      // state rows per lane
constexpr int ADJ_RU = (NU + ADJ_THREADS - 1) / ADJ_THREADS;      // control rows per lane
constexpr int ADJ_RP = (NP + ADJ_THREADS - 1) / ADJ_THREADS;      // parameters per lane

struct AdjStage {
    double a[ADJ_RX][NX], k[ADJ_RX][NU], xb[ADJ_RX];   // column i of A and of K, Xbar_k[i]
    double bc[ADJ_RU][NX], ub[ADJ_RU];                  // column j of B, Ubar'_k[j]
    double e[ADJ_RP][NX], kt[ADJ_RP][NU];               // column q of E and of Kth
};

// PM::NQ > 0 (cpdp_aux_adjoint_pd): lane l owns column l of [theta | pdata], i.e. column l of [E | E^pd] and [Kth | K^pd]
// (NP + NQ <= 32, so that the stage operands do not grow).
template <class PM>
CPDP_D void adj_fetch(const SolveArgs& a, const DiscWs& d, const PdWs& pw, const AdjArgs& j, int b, int k, int lane,
                      AdjStage& s) {
    const int N = a.N;
    const size_t g = (size_t)b * N + k;
    const double* ABg = a.AB + g * NX * NZ;
    const double* Kk = a.Kf + g * NU * NX;
    const double* Eg = d.E + g * NX * NP;
    const double* Ktk = d.Kth + g * NU * NP;
    NWT_UNROLL for (int t = 0; t < ADJ_RX; ++t) {
        const int i0 = lane + t * ADJ_THREADS, i = i0 < NX ? i0 : 0;    // (lanes past the end load a valid column and ignore it)
        NWT_UNROLL for (int e = 0; e < NX; ++e) s.a[t][e] = ABg[e * NZ + i];
        NWT_UNROLL for (int c = 0; c < NU; ++c) s.k[t][c] = Kk[c * NX + i];
        s.xb[t] = j.Xbar ? j.Xbar[((size_t)b * (N + 1) + k) * NX + i] : 0.0;
    }
    NWT_UNROLL for (int t = 0; t < ADJ_RU; ++t) {
        const int u0 = lane + t * ADJ_THREADS, u = u0 < NU ? u0 : 0;
        NWT_UNROLL for (int e = 0; e < NX; ++e) s.bc[t][e] = ABg[e * NZ + NX + u];
        double v = 0.0;
        if (j.Ubar) {
            v = j.Ubar[((size_t)b * (N + 1) + k) * NU + u];
            if (k == N - 1) v += j.Ubar[((size_t)b * (N + 1) + N) * NU + u];      // u_N = u_{N-1}
        }
        s.ub[t] = v;
    }
    if constexpr (PM::NQ > 0) {
        constexpr int XQ = PM::NQ;
        static_assert(ADJ_RP == 1 && NP + XQ <= ADJ_THREADS, "one column of [theta | pdata] per lane");
        const int l = lane < NP + XQ ? lane : 0;
        const bool th = l < NP;
        const double* Ec = th ? Eg + l : pw.Epd + g * NX * XQ + (l - NP);
        const double* Kc = th ? Ktk + l : pw.Kpd + g * NU * XQ + (l - NP);
        const int ld = th ? NP : XQ;
        NWT_UNROLL for (int e = 0; e < NX; ++e) s.e[0][e] = Ec[e * ld];
        NWT_UNROLL for (int c = 0; c < NU; ++c) s.kt[0][c] = Kc[c * ld];
    } else {
        NWT_UNROLL for (int t = 0; t < ADJ_RP; ++t) {
            const int q0 = lane + t * ADJ_THREADS, q = q0 < NP ? q0 : 0;
            NWT_UNROLL for (int e = 0; e < NX; ++e) s.e[t][e] = Eg[e * NP + q];
            NWT_UNROLL for (int c = 0; c < NU; ++c) s.kt[t][c] = Ktk[c * NP + q];
        }
    }
}

// PM::NQ > 0: the same sweep with pdata_bar[B][NQ] += K^pd' g + E^pd' p accumulated by lanes NP .. NP + NQ - 1.
template <class PM>
CPDP_GLOBAL void __launch_bounds__(ADJ_THREADS) k_aux_adjoint(AuxArgs x, SolveArgs a, DiscWs d, AdjArgs j, PdWs pw,
                                                              double* pdata_bar) {
    constexpr int XQ = PM::NQ;
    const int b = blockIdx.x, lane = threadIdx.x;
    const int N = a.N;
    if (x.aux_status[b] != 0 || (x.solve_status && x.solve_status[b] != ST_CONVERGED)) {
        for (int q = lane; q < NP; q += ADJ_THREADS) j.theta_bar[(size_t)b * NP + q] = 0.0;
        for (int q = lane; q < XQ; q += ADJ_THREADS) pdata_bar[(size_t)b * XQ + q] = 0.0;
        if (j.x0_bar) for (int i = lane; i < NX; i += ADJ_THREADS) j.x0_bar[(size_t)b * NX + i] = 0.0;
        return;
    }
    CPDP_SHARED double s_p[NX], s_g[NU];
    for (int i = lane; i < NX; i += ADJ_THREADS) s_p[i] = j.Xbar ? j.Xbar[((size_t)b * (N + 1) + N) * NX + i] : 0.0;
    double tb[ADJ_RP];
    NWT_UNROLL for (int t = 0; t < ADJ_RP; ++t) tb[t] = 0.0;
    AdjStage cur, nxt;
    adj_fetch<PM>(a, d, pw, j, b, N - 1, lane, nxt);
    NWT_SYNC();
    CPDP_LOOP for (int k = N - 1; k >= 0; --k) {
        cur = nxt;
        if (k > 0) adj_fetch<PM>(a, d, pw, j, b, k - 1, lane, nxt);
        // g = Ubar'_k + B_k' p
        NWT_UNROLL for (int t = 0; t < ADJ_RU; ++t) {
            const int u = lane + t * ADJ_THREADS;
            if (u < NU) {
                double acc = cur.ub[t];
                NWT_UNROLL for (int e = 0; e < NX; ++e) acc += cur.bc[t][e] * s_p[e];
                s_g[u] = acc;
            }
        }
        NWT_SYNC();
        // theta_bar += Kth_k' g + E_k' p;   p <- Xbar_k + A_k' p + K_k' g
        NWT_UNROLL for (int t = 0; t < ADJ_RP; ++t) {
            double acc = 0.0;
            NWT_UNROLL for (int c = 0; c < NU; ++c) acc += cur.kt[t][c] * s_g[c];
            NWT_UNROLL for (int e = 0; e < NX; ++e) acc += cur.e[t][e] * s_p[e];
            tb[t] += acc;
        }
        double pn[ADJ_RX];
        NWT_UNROLL for (int t = 0; t < ADJ_RX; ++t) {
            double acc = cur.xb[t];
            NWT_UNROLL for (int e = 0; e < NX; ++e) acc += cur.a[t][e] * s_p[e];
            NWT_UNROLL for (int c = 0; c < NU; ++c) acc += cur.k[t][c] * s_g[c];
            pn[t] = acc;
        }
        NWT_SYNC();                                        // every read of p and g of this stage is done
        NWT_UNROLL for (int t = 0; t < ADJ_RX; ++t) {
            const int i = lane + t * ADJ_THREADS;
            if (i < NX) s_p[i] = pn[t];
        }
        NWT_SYNC();
    }
    NWT_UNROLL for (int t = 0; t < ADJ_RP; ++t) {
        const int q = lane + t * ADJ_THREADS;
        if (q < NP) j.theta_bar[(size_t)b * NP + q] = tb[t];
        else if (XQ > 0 && q < NP + XQ) pdata_bar[(size_t)b * XQ + q - NP] = tb[t];
    }
    if (j.x0_bar) for (int i = lane; i < NX; i += ADJ_THREADS) j.x0_bar[(size_t)b * NX + i] = s_p[i];
}

}  // namespace CPDP_NS
