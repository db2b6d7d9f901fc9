// Warm start of the batched solve (cpdp_solve_warm, DESIGN.md §3.10): k_solve_init_warm takes the place of k_solve_init and starts
// each problem's Newton iteration from a caller's trajectory (X, U, Lam and, for a bounded model, z_L, z_U) instead of the zero
// seed.  Everything after the start -- stage kernels, Newton step, filter line search, convergence test -- is the cold solve's.
//   shift = 0:  row k of each array takes row k of the guess;
//   shift = 1:  row k takes row min(k + 1, last row of that quantity) (receding horizon: the previous solution one interval on);
//               X, Lam and the states' z repeat row N, U and the controls' z repeat row N-1.
//   X_0 = x0 in both modes, and U_N = U_{N-1} (CPDP.py:191).
// Bounded models follow IPOPT's warm_start_init_point: the primal is pushed into the interior by warm_start_bound_push =
// warm_start_bound_frac = 1e-3, z = max(z guess, warm_start_mult_bound_push = 1e-3) (z = mu_init / slack without a z guess), and
// mu = mu_init.  A problem whose init_status is not CPDP_CONVERGED gets k_solve_init's cold seed, bit for bit.
#pragma once
#include "cpdp_kernels.cuh"

namespace CPDP_NS {

// Guess of k_solve_init_warm (a separate parameter: SolveArgs, and with it every other kernel's parameters, stay as they are).
struct WarmArgs {
    const double* Xg;            // [B][N+1][NX]  may alias X
    const double* Ug;            // [B][N+1][NU]  may alias U
    const double* Lg;            // [B][N+1][NX]  may alias Lam
    const double* Zlg;           // [B][N+1][NZ]  or null (bounded models; may alias the workspace's z_L)
    const double* Zug;           // [B][N+1][NZ]  or null
    const int* init_status;      // [B] or null; may alias status
    int shift;                   // 0 or 1
    double mu_init;              // barrier parameter of a warm-started problem (bounded models)
};

constexpr double WARM_PUSH = 1e-3;        // IPOPT's warm_start_bound_push = warm_start_bound_frac
constexpr double WARM_MULT_PUSH = 1e-3;   // IPOPT's warm_start_mult_bound_push

// ------------------------------------------------------------------------------------------------
// k_solve_init_warm: one warp per problem (grid = B).  Lane l owns the whole columns j = l, l + 32, ... of the problem (X, Lam and
// z column j for a state, U and z column j for a control) and walks k upward, reading guess row k + shift before it writes row
// k; no other thread touches the column, so the guess may alias the outputs.
// ------------------------------------------------------------------------------------------------
constexpr int WARM_THREADS = 32;

// Starting value of component j in row k for a warm-started problem (bounded models: pushed, z from the guess or mu_init / s).
CPDP_D void warm_value(const WarmArgs& g, int j, const double* pd, bool var, double v, double zlg, double zug, double& w, double& zl,
                       double& zu) {
    if constexpr (!HAS_BOUNDS) {
        w = v; zl = 0.0; zu = 0.0;
    } else {
        const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
        const bool fl = var && bnd_finite(lb), fu = var && bnd_finite(ub);
        w = bnd_push(lb, ub, fl, fu, v, WARM_PUSH);
        if (g.Zlg) { zl = fl ? fmax(zlg, WARM_MULT_PUSH) : 0.0; zu = fu ? fmax(zug, WARM_MULT_PUSH) : 0.0; }
        else { zl = fl ? g.mu_init / (w - lb) : 0.0; zu = fu ? g.mu_init / (ub - w) : 0.0; }
    }
}

CPDP_GLOBAL void __launch_bounds__(WARM_THREADS) k_solve_init_warm(SolveArgs a, WarmArgs g) {
    const int b = blockIdx.x, lane = threadIdx.x;
    const int N = a.N;
    const bool cold = g.init_status && g.init_status[b] != ST_CONVERGED;
    NWT_SYNC();                                        // every lane has read init_status[b] before lane 0 writes status[b]
    const size_t rx = (size_t)b * (N + 1) * NX, ru = (size_t)b * (N + 1) * NU, rz = (size_t)b * (N + 1) * NZ;
    const double* pd = pdata_of(a, b);
    for (int j = lane; j < NZ; j += WARM_THREADS) {
        const bool isx = j < NX;
        const int c = isx ? j : j - NX, nc = isx ? NX : NU;
        const int last = isx ? N : N - 1;             // last row of the quantity (U_N is not a variable)
        const double* src = isx ? g.Xg : g.Ug;
        double* dst = isx ? a.X : a.U;
        const size_t r0 = isx ? rx : ru;
        double w = 0.0, zl = 0.0, zu = 0.0;
        for (int k = 0; k <= N; ++k) {
            const bool var = k <= last;
            const int ks = (k + g.shift < last) ? k + g.shift : last;
            double lam = 0.0;
            if (cold) {
                cold_seed(j, pd, var, w, zl, zu);
            } else if (var) {
                const double v = (isx && k == 0) ? a.x0[(size_t)b * NX + c] : src[r0 + (size_t)ks * nc + c];
                const double zlg = g.Zlg ? g.Zlg[rz + (size_t)ks * NZ + j] : 0.0, zug = g.Zug ? g.Zug[rz + (size_t)ks * NZ + j] : 0.0;
                if (isx) lam = g.Lg[rx + (size_t)ks * NX + c];
                warm_value(g, j, pd, true, v, zlg, zug, w, zl, zu);
            } else {
                zl = 0.0; zu = 0.0;                    // U_N = U_{N-1}: w keeps row N-1's value
            }
            dst[r0 + (size_t)k * nc + c] = w;
            if (isx) a.Lam[rx + (size_t)k * NX + c] = lam;
            if constexpr (HAS_BOUNDS) { a.zL[rz + (size_t)k * NZ + j] = zl; a.zU[rz + (size_t)k * NZ + j] = zu; }
        }
    }
    if (lane == 0) {
        start_state(a, b);
        if constexpr (HAS_BOUNDS) {
            a.bmu[b] = cold ? MU_COLD : g.mu_init;
            check_x0(a, b);
        }
    }
}

}  // namespace CPDP_NS
