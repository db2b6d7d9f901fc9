// CPDP gradient-iteration kernels (fp64, sm_100a).  Included AFTER a generated model header that defines
// `struct Model` (see codegen.py).  One shared library is built per model.
//
// Path and reference mapping (SURVEY.md §8a):
//   forward solve  : k_stage_adjoint + k_stage_hessian + k_newton_step   <- COCSys.cocSolver   CPDP.py:92-198
//   Riccati sweep  : k_riccati_rk45 / k_riccati_bdf                      <- auxSysSolver       CPDP.py:316-338
//   forward sweep  : k_aux_forward (+ fused loss / dL/dtheta)            <- auxSysSolver       CPDP.py:341-381
//                                                                           loss closures QuadAlgorithm.py:616-639
//   reduction      : k_reduce_tree                                        (new: cross-problem sum, fixed order)
// No tensor cores: per-step matrices are <= 13x13 (+ sparse), fp64.  Bound: FP64 pipe / latency, not HBM.
#pragma once
#include <type_traits>
#include "cpdp_port.h"

namespace CPDP_NS {

constexpr int NX = Model::NX;
constexpr int NU = Model::NU;
constexpr int NP = Model::NP;
constexpr int NZ = NX + NU;
constexpr int NQ = Model::NQ;          // per-problem constants (not learnable)
constexpr int HAS_TIME = Model::HAS_TIME;   // COCSys_TimeVarying (CPDP.py:394-787): f, c, h depend on the time t explicitly;
constexpr int NQT = NQ + HAS_TIME;          // the generated model code reads t as one more constant, pd[NQ]

constexpr int FILTER_CAP = 256;        // filter entries per problem (one is added per h-type iteration at most)

enum Status { ST_RUNNING = 0, ST_CONVERGED = 1, ST_MAXITER = 2, ST_LINESEARCH = 3, ST_NUMERIC = 4, ST_INFEASIBLE = 5 };

// Box bounds on the states and controls (DESIGN.md §3.8).  A model header defines HAS_BOUNDS and XLB / XUB / ULB / UUB only when
// some bound is finite; every other model takes the unbounded code path unchanged.  A model with BOUNDS_PD = 1 (DESIGN.md §3.12)
// has bounds that are expressions of its per-problem constants: XLB(i, pd) ...; every call site passes its problem's constants pd
// (the user constants, never the time slot), which lo(j, pd) / hi(j, pd) of a constant-bound model ignore.
template <class M, class = void> struct ModelBoundsPd { static constexpr int PD = 0; };
template <class M> struct ModelBoundsPd<M, std::void_t<decltype(M::BOUNDS_PD)>> { static constexpr int PD = M::BOUNDS_PD; };

template <class M, class = void> struct ModelBounds {
    static constexpr int HAS = 0;
    static constexpr int PD = 0;
    CPDP_HD static double lo(int) { return -1e20; }
    CPDP_HD static double hi(int) { return 1e20; }
    CPDP_HD static double lo(int, const double*) { return -1e20; }
    CPDP_HD static double hi(int, const double*) { return 1e20; }
};
template <class M> struct ModelBounds<M, std::void_t<decltype(M::HAS_BOUNDS)>> {
    static constexpr int HAS = M::HAS_BOUNDS;
    static constexpr int PD = ModelBoundsPd<M>::PD;
    // bound of component j of z = [x; u] (a chain of selects: no local-memory table for a lane-dependent j)
    CPDP_HD static double lo(int j) {
        double v = 0.0;
        CPDP_PRAGMA_UNROLL(NX) for (int i = 0; i < NX; ++i) if (i == j) v = M::XLB(i);
        CPDP_PRAGMA_UNROLL(NU) for (int i = 0; i < NU; ++i) if (NX + i == j) v = M::ULB(i);
        return v;
    }
    CPDP_HD static double hi(int j) {
        double v = 0.0;
        CPDP_PRAGMA_UNROLL(NX) for (int i = 0; i < NX; ++i) if (i == j) v = M::XUB(i);
        CPDP_PRAGMA_UNROLL(NU) for (int i = 0; i < NU; ++i) if (NX + i == j) v = M::UUB(i);
        return v;
    }
    // the bound of problem constants pd (the same select chain over the model's expressions of pd)
    CPDP_HD static double lo(int j, const double* pd) {
        if constexpr (!PD) {
            return lo(j);
        } else {
            double v = 0.0;
            CPDP_PRAGMA_UNROLL(NX) for (int i = 0; i < NX; ++i) if (i == j) v = M::XLB(i, pd);
            CPDP_PRAGMA_UNROLL(NU) for (int i = 0; i < NU; ++i) if (NX + i == j) v = M::ULB(i, pd);
            return v;
        }
    }
    CPDP_HD static double hi(int j, const double* pd) {
        if constexpr (!PD) {
            return hi(j);
        } else {
            double v = 0.0;
            CPDP_PRAGMA_UNROLL(NX) for (int i = 0; i < NX; ++i) if (i == j) v = M::XUB(i, pd);
            CPDP_PRAGMA_UNROLL(NU) for (int i = 0; i < NU; ++i) if (NX + i == j) v = M::UUB(i, pd);
            return v;
        }
    }
};
constexpr int HAS_BOUNDS = ModelBounds<Model>::HAS;
constexpr int BOUNDS_PD = ModelBounds<Model>::PD;      // bounds that depend on the per-problem constants
CPDP_HD bool bnd_finite(double v) { return fabs(v) < 1e19; }

// Barrier terms of component j (value w, multipliers zl, zu of its lower / upper bound, barrier parameter mu):
// sig = zl/sl + zu/su (the diagonal Sigma), bg = -mu/sl + mu/su (the barrier's gradient), sl = w - lb, su = ub - w; pd: the
// problem's constants.
CPDP_HD void bnd_terms(int j, const double* pd, double w, double zl, double zu, double mu, double& sig, double& bg) {
    const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
    sig = 0.0; bg = 0.0;
    if (bnd_finite(lb)) { const double s = w - lb; sig += zl / s; bg -= mu / s; }
    if (bnd_finite(ub)) { const double s = ub - w; sig += zu / s; bg += mu / s; }
}
// The two parts of bnd_terms' Sigma: sgl = zl/sl of the lower bound, sgu = zu/su of the upper one (0 for no finite bound).
CPDP_HD void bnd_sigmas(int j, const double* pd, double w, double zl, double zu, double& sgl, double& sgu) {
    const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
    sgl = bnd_finite(lb) ? zl / (w - lb) : 0.0;
    sgu = bnd_finite(ub) ? zu / (ub - w) : 0.0;
}

// Newton step of a bound multiplier z with slack s whose step is ds:  dz = mu/s - z - (z/s) ds.
CPDP_HD double bnd_dz(double s, double z, double mu, double ds) { return mu / s - z - (z / s) * ds; }
// ln of the slacks of component j at value w (the barrier's log terms; 0 for no finite bound)
CPDP_HD double bnd_log(int j, const double* pd, double w) {
    const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
    double v = 0.0;
    if (bnd_finite(lb)) v += log(w - lb);
    if (bnd_finite(ub)) v += log(ub - w);
    return v;
}

// Workspace of the barrier method.  An unbounded model's SolveArgs gets an empty base (static null pointers), so that its layout --
// and with it the kernel parameters of every kernel -- is the same as without bound support.
template <int H> struct BoundPtrs {
    double* zL;                  // [B][N+1][NZ]  multipliers of the lower bounds (row N: states only; 0 where no bound)
    double* zU;                  // [B][N+1][NZ]  multipliers of the upper bounds
    double* bmu;                 // [B]  barrier parameter
};
template <> struct BoundPtrs<0> {
    static constexpr double* zL = nullptr;
    static constexpr double* zU = nullptr;
    static constexpr double* bmu = nullptr;
};
CPDP_HD void bind_bounds(BoundPtrs<1>& p, double* zl, double* zu, double* mu) { p.zL = zl; p.zU = zu; p.bmu = mu; }
CPDP_HD void bind_bounds(BoundPtrs<0>&, double*, double*, double*) {}

// ------------------------------------------------------------------------------------------------
// Arguments of the forward-solve kernels (passed by value).
// ------------------------------------------------------------------------------------------------
struct SolveArgs : BoundPtrs<HAS_BOUNDS> {
    int B, N, S;                 // problems, grid intervals, RK4 substeps per interval
    double T;                    // horizon
    double tol;                  // KKT tolerance
    int max_iter;
    const double* x0;            // [B][NX]
    const double* theta;         // [B or 1][NP]
    int theta_stride;            // NP or 0
    const double* pdata;         // [B][NQ] per-problem constants (may be null if NQ == 0)
    double* X;                   // [B][N+1][NX]   NLP states (in/out)
    double* U;                   // [B][N+1][NU]   NLP controls, row N := row N-1 on exit
    double* Lam;                 // [B][N+1][NX]   multipliers of [x0-X0, F_k-X_{k+1}]
    int* status;                 // [B]
    int* iters;                  // [B]
    // workspace
    double* xs;                  // [B*N][4S][NX]  RK4 stage states
    double* mu;                  // [B*N][4S][NX]  stage adjoints
    double* AB;                  // [B*N][NX][NZ]  dF/d(x,u)
    double* H;                   // [B*N][NZ][NZ]  Hess (q + lam'F)
    double* gL;                  // [B*N][NZ]      grad (q + lam'F)
    double* dfc;                 // [B][N+1][NX]   defects (row 0 unused here)
    double* cost;                // [B*N]
    double* Vs;                  // [B][N+1][NX*NX]
    double* vs;                  // [B][N+1][NX]
    double* Kf;                  // [B*N][NU][NX]
    double* kf;                  // [B*N][NU]
    double* gq;                  // [B*N][NZ]
    double* dX;                  // [B][N+1][NX]
    double* dU;                  // [B][N][NU]
    double* lamn;                // [B][N+1][NX]
    double* th_init;             // [B]  max(1, theta(x0)): scale of the filter's theta_min / theta_max
    double* filt;                // [B][FILTER_CAP][2]  filter corners (theta, phi)
    int* nfilt;                  // [B]  filter entries in use
    double* dlast;               // [B]  last inertia-correction delta
    double* J;                   // [B]  objective at the current iterate
    double* kkt;                 // [B]  KKT error at the current iterate
    int* act;                    // [B]  compacted list of problems still iterating
    int* nact;                   // [1]
};

CPDP_HD const double* theta_of(const SolveArgs& a, int b) { return a.theta + (size_t)b * a.theta_stride; }
CPDP_HD const double* pdata_of(const SolveArgs& a, int b) { return a.pdata + (size_t)b * NQ; }

// [per-problem constants | t] for a time-varying model; the constants themselves otherwise (no copy)
struct PdBuf { double v[NQT > 0 ? NQT : 1]; };
CPDP_HD const double* pd_at(const double* pd, double t, PdBuf& buf) {
    if (!HAS_TIME) return pd;
    for (int i = 0; i < NQ; ++i) buf.v[i] = pd[i];
    buf.v[NQ] = t;
    return buf.v;
}
// node k of numpy.linspace(0, T, N + 1) (CPDP.py:544; the last node is T exactly) -- COCSys' [T / N * k] (CPDP.py:192) has the same bits
CPDP_HD double grid_time(double T, int N, int k) { return (k == N) ? T : (T / N) * k; }

// One classical RK4 step of (f, c) with frozen control (CPDP.py:117-123).
CPDP_HD void rk4_step(const double* x, const double* u, const double* th, const double* pd, double DT, double* xn, double& q) {
    double k[NX], xt[NX], c;
    Model::fc(x, u, th, pd, k, c);
    double qa = c;
    for (int i = 0; i < NX; ++i) { xn[i] = x[i] + DT / 6 * k[i]; xt[i] = x[i] + DT / 2 * k[i]; }
    Model::fc(xt, u, th, pd, k, c);
    qa += 2 * c;
    for (int i = 0; i < NX; ++i) { xn[i] += DT / 3 * k[i]; xt[i] = x[i] + DT / 2 * k[i]; }
    Model::fc(xt, u, th, pd, k, c);
    qa += 2 * c;
    for (int i = 0; i < NX; ++i) { xn[i] += DT / 3 * k[i]; xt[i] = x[i] + DT * k[i]; }
    Model::fc(xt, u, th, pd, k, c);
    qa += c;
    for (int i = 0; i < NX; ++i) xn[i] += DT / 6 * k[i];
    q += DT / 6 * qa;
}

// S RK4 steps over one grid interval: x -> x_end, q = integral of the path cost.
CPDP_HD void rk4_interval(const double* x, const double* u, const double* th, const double* pd, double DT, int S, double* xe, double& q) {
    double xa[NX], xb[NX];
    for (int i = 0; i < NX; ++i) xa[i] = x[i];
    q = 0.0;
    for (int s = 0; s < S; ++s) {
        rk4_step(xa, u, th, pd, DT, xb, q);
        for (int i = 0; i < NX; ++i) xa[i] = xb[i];
    }
    for (int i = 0; i < NX; ++i) xe[i] = xa[i];
}

// Layout of the stage states / stage adjoints handed from k_stage_adjoint to k_stage_hessian: tiles of STAGE_TILE intervals,
// element (stage row, e) of the tile's intervals contiguous -- [tile][row][e][interval in tile].  k_stage_adjoint runs one thread
// per interval, so a warp's store of one element is 256 contiguous bytes (the plain [interval][row][e] layout made it 32 separate
// sectors per store instruction: the kernel sat on a full load/store queue, lg_throttle 22 per issued instruction).
constexpr int STAGE_TILE = 32;
CPDP_HD size_t stage_off(int idx, int row, int nrows, int e) {
    return (((size_t)(idx / STAGE_TILE) * nrows + row) * NX + e) * STAGE_TILE + (idx % STAGE_TILE);
}

// ------------------------------------------------------------------------------------------------
// k_stage_adjoint: one thread per (problem, interval).
// Forward RK4 rollout storing the 4S stage states, defect and cost; then the discrete adjoint of the interval map
// seeded with lam_{k+1}, storing the 4S stage adjoints and grad_z (q_k + lam_{k+1}' F_k).
// ------------------------------------------------------------------------------------------------
CPDP_D void stage_adjoint_item(const SolveArgs& a, int b, int k);

#ifndef CPDP_ADJ_MINB
#define CPDP_ADJ_MINB 1
#endif
CPDP_GLOBAL void __launch_bounds__(128, CPDP_ADJ_MINB) k_stage_adjoint(SolveArgs a) {
    const int total = *a.nact * a.N;
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < total; item += gridDim.x * blockDim.x)
        stage_adjoint_item(a, a.act[item / a.N], item % a.N);
}

CPDP_D void stage_adjoint_item(const SolveArgs& a, int b, int k) {
    const int idx = b * a.N + k;
    const double DT = a.T / a.N / a.S;
    const double* th = theta_of(a, b);
    PdBuf pdb;
    const double* pd = pd_at(pdata_of(a, b), grid_time(a.T, a.N, k), pdb);      // the time is frozen at t_k over the interval (CPDP.py:512-519,554)
    double x[NX], u[NU];
    {
        const double* xk = a.X + ((size_t)b * (a.N + 1) + k) * NX;
        const double* uk = a.U + ((size_t)b * (a.N + 1) + k) * NU;
        for (int i = 0; i < NX; ++i) x[i] = xk[i];
        for (int i = 0; i < NU; ++i) u[i] = uk[i];
    }
    const int nrows = 4 * a.S;
    double* xs = a.xs + stage_off(idx, 0, nrows, 0);           // element (row, e) of this interval: xs[(row * NX + e) * STAGE_TILE]
    double* mus = a.mu + stage_off(idx, 0, nrows, 0);
    double q = 0.0;
    {   // forward
        double kk[NX], xt[NX], xn[NX], c;
        for (int s = 0; s < a.S; ++s) {
            double* st = xs + (size_t)s * 4 * NX * STAGE_TILE;
            for (int i = 0; i < NX; ++i) st[i * STAGE_TILE] = x[i];
            Model::fc(x, u, th, pd, kk, c);
            double qa = c;
            for (int i = 0; i < NX; ++i) { xn[i] = x[i] + DT / 6 * kk[i]; xt[i] = x[i] + DT / 2 * kk[i]; st[(NX + i) * STAGE_TILE] = xt[i]; }
            Model::fc(xt, u, th, pd, kk, c);
            qa += 2 * c;
            for (int i = 0; i < NX; ++i) { xn[i] += DT / 3 * kk[i]; xt[i] = x[i] + DT / 2 * kk[i]; st[(2 * NX + i) * STAGE_TILE] = xt[i]; }
            Model::fc(xt, u, th, pd, kk, c);
            qa += 2 * c;
            for (int i = 0; i < NX; ++i) { xn[i] += DT / 3 * kk[i]; xt[i] = x[i] + DT * kk[i]; st[(3 * NX + i) * STAGE_TILE] = xt[i]; }
            Model::fc(xt, u, th, pd, kk, c);
            qa += c;
            for (int i = 0; i < NX; ++i) x[i] = xn[i] + DT / 6 * kk[i];
            q += DT / 6 * qa;
        }
    }
    {
        const double* xn = a.X + ((size_t)b * (a.N + 1) + k + 1) * NX;
        double* d = a.dfc + ((size_t)b * (a.N + 1) + k + 1) * NX;
        for (int i = 0; i < NX; ++i) d[i] = x[i] - xn[i];
        a.cost[idx] = q;
    }
    // backward (adjoint) sweep
    double adj[NX], gu[NU];
    {
        const double* ln = a.Lam + ((size_t)b * (a.N + 1) + k + 1) * NX;
        for (int i = 0; i < NX; ++i) adj[i] = ln[i];
        for (int i = 0; i < NU; ++i) gu[i] = 0.0;
    }
    const double bco[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
    const double aco[4] = {0.0, 0.5, 0.5, 1.0};
    for (int s = a.S - 1; s >= 0; --s) {
        double ax[NX], xi[NX], kap[NX], g_u[NU], xst[NX];
        for (int i = 0; i < NX; ++i) { ax[i] = 0.0; xi[i] = 0.0; }
        for (int st = 3; st >= 0; --st) {
            const double* xsp = xs + ((size_t)s * 4 + st) * NX * STAGE_TILE;
            for (int i = 0; i < NX; ++i) xst[i] = xsp[i * STAGE_TILE];
            const double cnext = (st < 3) ? aco[st + 1] * DT : 0.0;
            for (int i = 0; i < NX; ++i) kap[i] = bco[st] * DT * adj[i] + cnext * xi[i];
            double* mp = mus + ((size_t)s * 4 + st) * NX * STAGE_TILE;
            for (int i = 0; i < NX; ++i) mp[i * STAGE_TILE] = kap[i];
            Model::hgrad(xst, u, th, pd, kap, bco[st] * DT, xi, g_u);
            for (int i = 0; i < NX; ++i) ax[i] += xi[i];
            for (int i = 0; i < NU; ++i) gu[i] += g_u[i];
        }
        for (int i = 0; i < NX; ++i) adj[i] += ax[i];
    }
    double* g = a.gL + (size_t)idx * NZ;
    for (int i = 0; i < NX; ++i) g[i] = adj[i];
    for (int i = 0; i < NU; ++i) g[NX + i] = gu[i];
}

// ------------------------------------------------------------------------------------------------
// k_stage_hessian: NZ threads per (problem, interval), KPC intervals per CTA.
// Thread j propagates column j of the forward sensitivity d(stage state)/d(x_k,u_k) through the 4S stages and
// accumulates column j of  Hess = sum_s Sz_s' Hess_z(mu_s'f + w_s c) Sz_s ; writes [A B] and Hess.
// ------------------------------------------------------------------------------------------------
// CTA size: the kernel needs ~250 registers per thread, so an SM holds 256 threads of it whatever their grouping; small CTAs
// (64 threads, four per SM) run out of phase with each other and overlap the arithmetic-bound model code of one with the
// shared-memory-bound accumulation of another, which one 256-thread CTA serialises behind its barriers (41.5 -> 38.3 ms / solve)
#ifndef CPDP_HESS_THREADS
#define CPDP_HESS_THREADS 64
#endif
#ifndef CPDP_HESS_GRID_MULT
#define CPDP_HESS_GRID_MULT (4 * (256 / CPDP_HESS_THREADS))     // CTAs per SM in the grid (grid-stride loop over the interval groups)
#endif
constexpr int HESS_THREADS = CPDP_HESS_THREADS;
constexpr int KPC = HESS_THREADS / NZ;          // intervals per CTA
static_assert(KPC >= 1, "k_stage_hessian: a CTA must hold at least one interval (NZ threads)");

#ifndef CPDP_HESS_MINB
#define CPDP_HESS_MINB (256 / CPDP_HESS_THREADS)
#endif
CPDP_GLOBAL void __launch_bounds__(HESS_THREADS, CPDP_HESS_MINB) k_stage_hessian(SolveArgs a) {
    CPDP_SHARED double s_x[2][KPC][NX];        // double-buffered: the next stage's states / adjoints are fetched while this one computes
    CPDP_SHARED double s_mu[2][KPC][NX];
    CPDP_SHARED double s_u[KPC][NU];
    CPDP_SHARED double s_th[KPC][NP];
    CPDP_SHARED double s_pd[KPC][NQT > 0 ? NQT : 1];
    constexpr int SXS = (NX + 1) & ~1;                 // even row length: the Hessian accumulation reads the rows with 128-bit loads
    // rows 0 .. NZ-1 = the NZ sensitivity columns; rows NZ .. NZ+HW-2 repeat rows 0 .. HW-2, so that thread j reads rows j .. j+HW-1
    // without wrapping: consecutive lanes then read consecutive rows (7 x 16 bytes apart: a quarter-warp covers all banks)
    CPDP_SHARED __align__(16) double s_S[KPC][NZ + NZ / 2][SXS];
    CPDP_SHARED double s_hzu[KPC][NZ][NU];     // control rows of each thread's Hessian-vector product (dynamic index in the accumulation)
    CPDP_SHARED int s_gi[KPC];                 // global interval index b*N+k of each slot, -1 if none
    constexpr int HW = NZ / 2 + 1;
    const int tid = threadIdx.x;
    const int kk = tid / NZ, j = tid % NZ;
    const int total = *a.nact * a.N;
    const int ngroups = (total + KPC - 1) / KPC;
    const double DT = a.T / a.N / a.S;
    const double bco[4] = {1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6};
    const double aco[4] = {0.0, 0.5, 0.5, 1.0};

    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
        __syncthreads();
        for (int t = tid; t < KPC; t += HESS_THREADS) {
            const int li = grp * KPC + t;
            s_gi[t] = (li < total) ? a.act[li / a.N] * a.N + li % a.N : -1;
        }
        __syncthreads();
        for (int t = tid; t < KPC * (NU + NP + NQ); t += HESS_THREADS) {
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
            for (int t = tid; t < KPC; t += HESS_THREADS) if (s_gi[t] >= 0) s_pd[t][NQ] = grid_time(a.T, a.N, s_gi[t] % a.N);
        }
        const bool mine = (kk < KPC) && (s_gi[kk < KPC ? kk : 0] >= 0);
        const int gi = mine ? s_gi[kk] : -1;

        // The Hessian is symmetric: thread j accumulates the HW entries (i, j), i = (j + w) mod NZ, w < HW, and mirrors them at
        // the end -- every unordered pair {i, j} is covered once (for even NZ the pairs at distance NZ/2 twice: the lower thread writes them).
        double Sx[NX], Sn[NX], dX[NX], df[NX], du[NU], hz[NZ], Hc[HW];
        const double* rowp[HW];                    // row i of this interval's stage sensitivities
        int rowu[HW];                              // i - NX for the control rows, -1 for the state rows
        for (int w = 0; w < HW; ++w) {
            const int i = (j + w) % NZ;
            rowp[w] = s_S[kk < KPC ? kk : 0][j + w];
            rowu[w] = i >= NX ? i - NX : -1;
            Hc[w] = 0.0;
        }
        for (int i = 0; i < NX; ++i) { Sx[i] = (i == j) ? 1.0 : 0.0; df[i] = 0.0; }
        for (int i = 0; i < NU; ++i) du[i] = (NX + i == j) ? 1.0 : 0.0;

        // stage states + adjoints of every interval of this group: fetched one stage ahead into registers, parked in the other
        // shared-memory buffer after the Hessian accumulation (the global-load latency hides behind the model code)
        constexpr int NPRE = (KPC * 2 * NX + HESS_THREADS - 1) / HESS_THREADS;
        double pre[NPRE];
        const int nstage = 4 * a.S;
#define HESS_FETCH(sidx)                                                                                        \
        for (int p_ = 0; p_ < NPRE; ++p_) {                                                                     \
            const int t = tid + p_ * HESS_THREADS;                                                              \
            pre[p_] = 0.0;                                                                                      \
            if (t < KPC * 2 * NX) {                                                                             \
                const int q = t % KPC, e = t / KPC;     /* intervals fastest: neighbours share sectors of the tiled arrays */  \
                const int g2 = s_gi[q];                                                                         \
                if (g2 >= 0) {                                                                                  \
                    pre[p_] = (e < NX) ? a.xs[stage_off(g2, (sidx), nstage, e)] : a.mu[stage_off(g2, (sidx), nstage, e - NX)];  \
                }                                                                                               \
            }                                                                                                   \
        }
#define HESS_STASH(buf)                                                                                         \
        for (int p_ = 0; p_ < NPRE; ++p_) {                                                                     \
            const int t = tid + p_ * HESS_THREADS;                                                              \
            if (t < KPC * 2 * NX) {                                                                             \
                const int q = t % KPC, e = t / KPC;     /* intervals fastest: neighbours share sectors of the tiled arrays */  \
                if (e < NX) s_x[buf][q][e] = pre[p_]; else s_mu[buf][q][e - NX] = pre[p_];                      \
            }                                                                                                   \
        }
        HESS_FETCH(0)
        HESS_STASH(0)
        __syncthreads();
        for (int s = 0; s < a.S; ++s) {
            for (int i = 0; i < NX; ++i) Sn[i] = Sx[i];
            for (int st = 0; st < 4; ++st) {
                const int sidx = s * 4 + st, cur = sidx & 1;
                if (sidx + 1 < nstage) { HESS_FETCH(sidx + 1) }
                if (mine) {
                    const double ca = aco[st] * DT;
                    for (int i = 0; i < NX; ++i) dX[i] = Sx[i] + ca * df[i];
                    Model::dir(s_x[cur][kk], s_u[kk], s_th[kk], s_pd[kk], s_mu[cur][kk], bco[st] * DT, dX, du, df, hz);
                    for (int i = 0; i < NX; ++i) s_S[kk][j][i] = dX[i];
                    if (j < NZ / 2) { for (int i = 0; i < NX; ++i) s_S[kk][NZ + j][i] = dX[i]; }
                    for (int i = 0; i < NU; ++i) s_hzu[kk][j][i] = hz[NX + i];      // (read back by this thread only)
                }
                __syncthreads();
                if (mine) {
                    // Hc[w] += hz[i] (control rows) + sum_e S[i][e] hz[e],  i = (j + w) mod NZ, e ascending.  The HW rows advance
                    // together through e: their loads are issued back to back and the rows are independent sums, so neither the
                    // shared-memory latency nor the add latency of one row's chain is exposed.
                    double acc[HW];
                    CPDP_PRAGMA_UNROLL(HW) for (int w = 0; w < HW; ++w) acc[w] = rowu[w] >= 0 ? s_hzu[kk][j][rowu[w] >= 0 ? rowu[w] : 0] : 0.0;
#ifdef __CUDACC__
#pragma unroll
                    for (int e = 0; e + 1 < NX; e += 2) {
                        double2 c2[HW];
#pragma unroll
                        for (int w = 0; w < HW; ++w) c2[w] = *reinterpret_cast<const double2*>(rowp[w] + e);
#pragma unroll
                        for (int w = 0; w < HW; ++w) { acc[w] += c2[w].x * hz[e]; acc[w] += c2[w].y * hz[e + 1]; }
                    }
                    if (NX & 1) {                                          // (last element through a 128-bit load as well: the 64-bit form conflicts two-way)
#pragma unroll
                        for (int w = 0; w < HW; ++w) acc[w] += reinterpret_cast<const double2*>(rowp[w] + NX - 1)->x * hz[NX - 1];
                    }
#else
                    for (int w = 0; w < HW; ++w) { for (int e = 0; e < NX; ++e) acc[w] += rowp[w][e] * hz[e]; }
#endif
                    CPDP_PRAGMA_UNROLL(HW) for (int w = 0; w < HW; ++w) Hc[w] += acc[w];
                    const double cb = bco[st] * DT;
                    for (int i = 0; i < NX; ++i) Sn[i] += cb * df[i];
                }
                if (sidx + 1 < nstage) { HESS_STASH(cur ^ 1) }     // (the other buffer was last read by the previous stage's model code)
                __syncthreads();
            }
            for (int i = 0; i < NX; ++i) Sx[i] = Sn[i];
        }
#undef HESS_FETCH
#undef HESS_STASH
        if (mine) {
            double* AB = a.AB + (size_t)gi * NX * NZ;
            for (int i = 0; i < NX; ++i) AB[i * NZ + j] = Sx[i];
            double* H = a.H + (size_t)gi * NZ * NZ;
            for (int w = 0; w < HW; ++w) {
                const int i = (j + w) % NZ;
                // (even NZ: the pairs at distance NZ/2 are computed by both of their threads; the lower one writes them)
                if ((NZ % 2 == 0) && w == NZ / 2 && j >= NZ / 2) continue;
                H[i * NZ + j] = Hc[w];
                if (w != 0) H[j * NZ + i] = Hc[w];                     // exactly symmetric: k_newton_step reads one triangle's worth
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// small dense helpers used by one CTA (all threads call; results valid after the trailing barrier)
// ------------------------------------------------------------------------------------------------
// Block-wide sum / max returned to every thread.  Order of operations (identical on the GPU and in the host
// emulation, so both produce the same bits): xor-butterfly inside each group of 32 threads, then the group results
// are combined sequentially in group order by every thread.  blockDim.x must be a multiple of 32; `red` needs
// blockDim.x doubles (emulation) / blockDim.x/32 doubles (GPU).  All threads of the CTA must call it.
CPDP_D double block_reduce(double v, double* red, bool is_max) {
    const int tid = threadIdx.x, nt = blockDim.x;
#ifdef __CUDACC__
    for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(0xffffffffu, v, o);
        v = is_max ? fmax(v, x) : (v + x);
    }
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double r = red[0];
    for (int i = 1; i < (nt >> 5); ++i) r = is_max ? fmax(r, red[i]) : (r + red[i]);
    return r;
#else
    for (int o = 16; o > 0; o >>= 1) {
        __syncthreads();
        red[tid] = v;
        __syncthreads();
        const double x = red[tid ^ o];
        v = is_max ? fmax(v, x) : (v + x);
    }
    __syncthreads();
    red[tid] = v;
    __syncthreads();
    double r = red[0];
    for (int i = 32; i < nt; i += 32) r = is_max ? fmax(r, red[i]) : (r + red[i]);
    return r;
#endif
}

// In-place Cholesky of an n x n SPD matrix (row-major, lower triangle used). Returns false if not PD.
template <int n>
CPDP_HD bool chol_inplace(double* A) {
    for (int j = 0; j < n; ++j) {
        double d = A[j * n + j];
        for (int k = 0; k < j; ++k) d -= A[j * n + k] * A[j * n + k];
        if (!(d > 0.0)) return false;
        d = sqrt(d);
        A[j * n + j] = d;
        for (int i = j + 1; i < n; ++i) {
            double s = A[i * n + j];
            for (int k = 0; k < j; ++k) s -= A[i * n + k] * A[j * n + k];
            A[i * n + j] = s / d;
        }
    }
    return true;
}

// Solve L L' x = b in place (L from chol_inplace).
template <int n>
CPDP_HD void chol_solve(const double* L, double* b) {
    for (int i = 0; i < n; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i * n + k] * b[k];
        b[i] = s / L[i * n + i];
    }
    for (int i = n - 1; i >= 0; --i) {
        double s = b[i];
        for (int k = i + 1; k < n; ++k) s -= L[k * n + i] * b[k];
        b[i] = s / L[i * n + i];
    }
}

// ------------------------------------------------------------------------------------------------
// k_newton_step: one CTA per problem.
//  1. KKT error of the current iterate (stop test, IPOPT-style: max(|grad L|, |g|)).
//  2. Newton step of the equality-constrained NLP by the Riccati recursion on the stage-wise KKT system, with
//     IPOPT's inertia-correction schedule when some Quu block is not positive definite.
//  3. IPOPT filter line search (one thread per interval re-integrates the RK4 map).
//  4. Primal / dual update.
// ------------------------------------------------------------------------------------------------
// Shape (round 2): ONE WARP per problem; lane j < NZ owns column j of the stage matrices ([A B], T = V [A B], Q) in
// registers, every product is "matrix in shared memory (broadcast loads, contraction index rolled) times my column" with NX / NZ
// independent accumulators -- the first version ran 64-thread CTAs through rolled shared-memory dot products with ten CTA
// barriers per stage (1.2 ms per round at any batch size: latency bound).  All sums are taken in the first version's order.
constexpr int NEWTON_THREADS = 32;
static_assert(NZ <= 32, "k_newton_step maps one lane per column of the stage-wise KKT blocks");
constexpr int NZS = NZ | 1;              // odd row strides: conflict-free row reads by lane
constexpr int NXS = NX | 1;

#ifdef __CUDACC__
#define NWT_SYNC() __syncwarp()
#define NWT_UNROLL _Pragma("unroll")
#else
#define NWT_SYNC() __syncthreads()
#define NWT_UNROLL
#endif

// out[i] += sum_k AT[k * as + i] * x[k * xs], i < NOUT: contraction rolled, NOUT independent accumulators (ascending k)
template <int NOUT>
CPDP_D void nwt_mac(const double* __restrict__ AT, const int as, const double* __restrict__ x, const int xs, const int nk, double (&out)[NOUT]) {
    CPDP_LOOP for (int k = 0; k < nk; ++k) {
        const double xk = x[k * xs];
        NWT_UNROLL for (int i = 0; i < NOUT; ++i) out[i] += AT[k * as + i] * xk;
    }
}

CPDP_D double nwt_reduce(double v, double* red, bool is_max) {
#ifdef __CUDACC__
    (void)red;
    NWT_UNROLL for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(0xffffffffu, v, o);
        v = is_max ? fmax(v, x) : (v + x);
    }
    return v;
#else
    return block_reduce(v, red, is_max);
#endif
}

CPDP_D void newton_step_problem(const SolveArgs& a, const int b) {
    const int lane = threadIdx.x, nt = NEWTON_THREADS;
    const int N = a.N;
    const double DT = a.T / a.N / a.S;
    const double* th = theta_of(a, b);
    const double* pd0 = pdata_of(a, b);
    double* X = a.X + (size_t)b * (N + 1) * NX;
    double* U = a.U + (size_t)b * (N + 1) * NU;
    double* Lam = a.Lam + (size_t)b * (N + 1) * NX;
    double* dfc = a.dfc + (size_t)b * (N + 1) * NX;
    double* dX = a.dX + (size_t)b * (N + 1) * NX;
    double* dU = a.dU + (size_t)b * N * NU;
    double* lamn = a.lamn + (size_t)b * (N + 1) * NX;
    double* Vs = a.Vs + (size_t)b * (N + 1) * NX * NX;
    double* vs = a.vs + (size_t)b * (N + 1) * NX;
    const size_t ib = (size_t)b * N;

    CPDP_SHARED double red[66];
    CPDP_SHARED double s_hx[NX], s_hxx[NX * NX], s_hxe[NX * NP];
    CPDP_SHARED double s_V[NX * NXS], s_v[NX], s_vt[NX];          // value function of the stage being eliminated (V symmetric)
    CPDP_SHARED double s_AB[NX * NZS], s_T[NX * NZS], s_Q[NZ * NZS];
    CPDP_SHARED double s_L[NU * NU], s_K[NU * NXS], s_kf[NU], s_dx[NX], s_du[NU], s_dk[NX], s_lk[NX];
    CPDP_SHARED double s_h;
    CPDP_SHARED int s_flag;
    const bool isZ = lane < NZ, isX = lane < NX;
    const int jz = isZ ? lane : 0, jx = isX ? lane : 0;

    // ---- terminal cost derivatives, defect of the initial condition
    if (lane == 0) {
        double h;
        PdBuf pdb;
        const double* pd = pd_at(pd0, grid_time(a.T, N, N), pdb);
        Model::term(X + (size_t)N * NX, th, pd, h, s_hx);
        Model::term2(X + (size_t)N * NX, th, pd, s_hxx, s_hxe);
        s_h = h;
    }
    for (int i = lane; i < NX; i += nt) dfc[i] = a.x0[(size_t)b * NX + i] - X[i];
    NWT_SYNC();

    // ---- KKT error and objective
    double e = 0.0, Jp = 0.0, g1 = 0.0;
    double* zL = nullptr;
    double* zU = nullptr;
    if constexpr (!HAS_BOUNDS) {
        for (int k = lane; k < N; k += nt) {
            const double* g = a.gL + (ib + k) * NZ;
            for (int i = 0; i < NX; ++i) e = fmax(e, fabs(g[i] - Lam[(size_t)k * NX + i]));
            for (int i = 0; i < NU; ++i) e = fmax(e, fabs(g[NX + i]));
            Jp += a.cost[ib + k];
        }
    } else {
        // gradient of the Lagrangian with the bound multipliers: grad L - z_L + z_U
        zL = a.zL + (size_t)b * (N + 1) * NZ;
        zU = a.zU + (size_t)b * (N + 1) * NZ;
        for (int k = lane; k < N; k += nt) {
            const double* g = a.gL + (ib + k) * NZ;
            for (int i = 0; i < NX; ++i) e = fmax(e, fabs(g[i] - Lam[(size_t)k * NX + i] - zL[(size_t)k * NZ + i] + zU[(size_t)k * NZ + i]));
            for (int i = 0; i < NU; ++i) e = fmax(e, fabs(g[NX + i] - zL[(size_t)k * NZ + NX + i] + zU[(size_t)k * NZ + NX + i]));
            Jp += a.cost[ib + k];
        }
    }
    for (int i = lane; i < (N + 1) * NX; i += nt) { e = fmax(e, fabs(dfc[i])); g1 += fabs(dfc[i]); }
    if constexpr (!HAS_BOUNDS) {
        for (int i = lane; i < NX; i += nt) e = fmax(e, fabs(s_hx[i] - Lam[(size_t)N * NX + i]));
    } else {
        for (int i = lane; i < NX; i += nt) e = fmax(e, fabs(s_hx[i] - Lam[(size_t)N * NX + i] - zL[(size_t)N * NZ + i] + zU[(size_t)N * NZ + i]));
    }
    double kkt = nwt_reduce(e, red, true);
    const double J0 = nwt_reduce(Jp, red, false) + s_h;
    g1 = nwt_reduce(g1, red, false);
    // Barrier method (IPOPT's monotone mode, Waechter & Biegler 2006, §2-3; unscaled): the stop test is E_0 < tol, and while
    // E_mu <= 10 mu the barrier parameter drops to max(tol/10, min(0.2 mu, mu^1.5)) and the filter is emptied.
    // E_mu = max(|grad L - z_L + z_U|, |c|, |S z - mu|): the complementarity enters through max(S z) and min(S z).
    double mu = 0.0, P0 = J0;                     // barrier parameter, barrier objective phi_mu at the current iterate
    bool freset = false;
    if constexpr (HAS_BOUNDS) {
        mu = a.bmu[b];                              // (read before the reductions: lane 0 writes it back below)
        double szmax = 0.0, nszmin = -1e300, lg = 0.0;
        for (int idx = lane; idx < (N + 1) * NZ; idx += nt) {
            const int k = idx / NZ, j = idx % NZ;
            if (k == N && j >= NX) continue;
            const double w = (j < NX) ? X[(size_t)k * NX + j] : U[(size_t)k * NU + j - NX];
            const double lb = ModelBounds<Model>::lo(j, pd0), ub = ModelBounds<Model>::hi(j, pd0);
            if (bnd_finite(lb)) { const double sl = w - lb, p = sl * zL[idx]; szmax = fmax(szmax, p); nszmin = fmax(nszmin, -p); lg += log(sl); }
            if (bnd_finite(ub)) { const double su = ub - w, p = su * zU[idx]; szmax = fmax(szmax, p); nszmin = fmax(nszmin, -p); lg += log(su); }
        }
        szmax = nwt_reduce(szmax, red, true);
        nszmin = nwt_reduce(nszmin, red, true);
        lg = nwt_reduce(lg, red, false);
        const double est = kkt;
        kkt = fmax(est, szmax);
        if (kkt >= a.tol) {
            while (fmax(est, fmax(szmax - mu, mu + nszmin)) <= 10.0 * mu) {
                const double mn = fmax(a.tol / 10.0, fmin(0.2 * mu, pow(mu, 1.5)));
                if (!(mn < mu)) break;
                mu = mn;
                freset = true;
            }
        }
        P0 = J0 - mu * lg;
    }
    if (lane == 0) { a.kkt[b] = kkt; a.J[b] = J0; }
    if constexpr (HAS_BOUNDS) {
        if (lane == 0) { a.bmu[b] = mu; if (freset) a.nfilt[b] = 0; }
    }
    const int it = a.iters[b];
    if (!(kkt == kkt)) { if (lane == 0) a.status[b] = ST_NUMERIC; }
    if (kkt < a.tol || it >= a.max_iter || !(kkt == kkt)) {
        if (lane == 0 && kkt == kkt) a.status[b] = (kkt < a.tol) ? ST_CONVERGED : ST_MAXITER;
        for (int i = lane; i < NU; i += nt) U[(size_t)N * NU + i] = U[(size_t)(N - 1) * NU + i];   // CPDP.py:191
        return;
    }

    // barrier terms of the final state (lane i: component i)
    double sgN = 0.0, bgN = 0.0;
    if constexpr (HAS_BOUNDS) {
        if (isX) bnd_terms(jx, pd0, X[(size_t)N * NX + jx], zL[(size_t)N * NZ + jx], zU[(size_t)N * NZ + jx], mu, sgN, bgN);
    }

    // ---- Riccati factorisation with inertia correction (IPOPT Alg. IC)
    const double dlast = a.dlast[b];
    double delta = 0.0;
    int attempt = 0;
    while (true) {
        if (isX) {
            const double dN = HAS_BOUNDS ? delta + sgN : delta;          // (+ Sigma of the final state)
            NWT_UNROLL for (int i = 0; i < NX; ++i) {
                const double v = s_hxx[i * NX + jx] + ((i == jx) ? dN : 0.0);
                s_V[i * NXS + jx] = v;
                Vs[(size_t)N * NX * NX + i * NX + jx] = v;
            }
            const double hN = HAS_BOUNDS ? s_hx[jx] + bgN : s_hx[jx];      // (+ barrier gradient)
            s_v[jx] = hN;
            vs[(size_t)N * NX + jx] = hN;
        }
        if (lane == 0) s_flag = 0;
        NWT_SYNC();
        for (int k = N - 1; k >= 0; --k) {
            const double* ABg = a.AB + (ib + k) * NX * NZ;
            const double* Hg = a.H + (ib + k) * NZ * NZ;
            const double* gLg = a.gL + (ib + k) * NZ;
            const double* dk1 = dfc + (size_t)(k + 1) * NX;
            const double* lk1 = Lam + (size_t)(k + 1) * NX;
            // my column of [A B]; vt = v + V d_{k+1}
            // (every global operand of the stage is fetched up front, in one batch of independent loads: the stage loop is a
            //  chain of short dependent phases, an L2 round trip inside any of them is paid 50 times per problem and round)
            double ab[NX], hq[NZ];
            NWT_UNROLL for (int e2 = 0; e2 < NX; ++e2) ab[e2] = isZ ? ABg[e2 * NZ + jz] : 0.0;
            NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) hq[r_] = isZ ? Hg[r_ * NZ + jz] : 0.0;     // (k_stage_hessian writes H exactly symmetric: 0.5 (H + H') = H)
            const double gl = isZ ? gLg[jz] : 0.0;
            double sgk = 0.0, bgk = 0.0;                 // barrier terms of my component of z_k
            if constexpr (HAS_BOUNDS) {
                if (isZ) bnd_terms(jz, pd0, jz < NX ? X[(size_t)k * NX + jz] : U[(size_t)k * NU + jz - NX], zL[(size_t)k * NZ + jz],
                                   zU[(size_t)k * NZ + jz], mu, sgk, bgk);
            }
            if (isX) { s_dk[jx] = dk1[jx]; s_lk[jx] = lk1[jx]; }
            NWT_UNROLL for (int e2 = 0; e2 < NX; ++e2) if (isZ) s_AB[e2 * NZS + jz] = ab[e2];
            NWT_SYNC();
            if (isX) {
                double acc = s_v[jx];
                NWT_UNROLL for (int c = 0; c < NX; ++c) acc += s_V[jx * NXS + c] * s_dk[c];
                s_vt[jx] = acc;
            }
            NWT_SYNC();
            // T[:, j] = V [A B][:, j]   (V symmetric: V[e][i] = V[i][e] is its own contraction-major operand)
            double t[NX];
            NWT_UNROLL for (int i = 0; i < NX; ++i) t[i] = 0.0;
            if (isZ) nwt_mac<NX>(s_V, NXS, s_AB + jz, NZS, NX, t);
            // gq[j] = gL[j] - [A B][:, j]' lam_{k+1};  qv[j] = gq[j] + [A B][:, j]' vt
            double gqj = gl;
            NWT_UNROLL for (int e2 = 0; e2 < NX; ++e2) gqj -= ab[e2] * s_lk[e2];
            if constexpr (HAS_BOUNDS) gqj += bgk;       // gradient of the barrier objective
            double qvj = gqj;
            NWT_UNROLL for (int e2 = 0; e2 < NX; ++e2) qvj += ab[e2] * s_vt[e2];
            if (isZ) { NWT_UNROLL for (int e2 = 0; e2 < NX; ++e2) s_T[e2 * NZS + jz] = t[e2]; a.gq[(ib + k) * NZ + jz] = gqj; }
            // Q[:, j] = sym(H)[:, j] + (delta + Sigma_j) e_j + [A B]' T[:, j]
            double q[NZ];
            const double dk = HAS_BOUNDS ? delta + sgk : delta;
            NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) q[r_] = hq[r_] + ((isZ && r_ == jz) ? dk : 0.0);
            if (isZ) nwt_mac<NZ>(s_AB, NZS, s_T + jz, NZS, NX, q);          // (reads my own column of T: no barrier needed)
            if (isZ) { NWT_UNROLL for (int r_ = 0; r_ < NZ; ++r_) s_Q[r_ * NZS + jz] = q[r_]; }
            NWT_SYNC();
            // Quu = L L'
            if (lane == 0) {
                for (int r_ = 0; r_ < NU; ++r_)
                    for (int c = 0; c < NU; ++c)
                        s_L[r_ * NU + c] = 0.5 * (s_Q[(NX + r_) * NZS + NX + c] + s_Q[(NX + c) * NZS + NX + r_]);
                if (!chol_inplace<NU>(s_L)) s_flag = 1;
            }
            NWT_SYNC();
            if (s_flag) break;
            // K = -Quu^{-1} Qux (my column), kf = -Quu^{-1} qu (lane NX, which holds qv[NX..] below)
            if (isX) {
                double rhs[NU];
                NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) rhs[r_] = 0.5 * (q[NX + r_] + s_Q[jx * NZS + NX + r_]);
                chol_solve<NU>(s_L, rhs);
                NWT_UNROLL for (int r_ = 0; r_ < NU; ++r_) { s_K[r_ * NXS + jx] = -rhs[r_]; a.Kf[(ib + k) * NU * NX + r_ * NX + jx] = -rhs[r_]; }
            }
            // qv of the control rows travels through shared memory to one lane
            if (lane >= NX && lane < NZ) s_du[lane - NX] = qvj;
            NWT_SYNC();
            if (lane == 0) {
                double rhs[NU];
                for (int r_ = 0; r_ < NU; ++r_) rhs[r_] = s_du[r_];
                chol_solve<NU>(s_L, rhs);
                for (int r_ = 0; r_ < NU; ++r_) { s_kf[r_] = -rhs[r_]; a.kf[(ib + k) * NU + r_] = -rhs[r_]; }
            }
            NWT_SYNC();
            // V = Qxx + Qxu K (symmetrised), v = qx + Qxu kf
            if (isX) {
                const int c = jx;
                double vnew[NX];
                NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) {
                    const double acc = 0.5 * (s_Q[r_ * NZS + c] + s_Q[c * NZS + r_]);
                    double a1 = 0.0, a2 = 0.0;
                    NWT_UNROLL for (int e2 = 0; e2 < NU; ++e2) {
                        a1 += 0.5 * (s_Q[r_ * NZS + NX + e2] + s_Q[(NX + e2) * NZS + r_]) * s_K[e2 * NXS + c];
                        a2 += 0.5 * (s_Q[c * NZS + NX + e2] + s_Q[(NX + e2) * NZS + c]) * s_K[e2 * NXS + r_];
                    }
                    vnew[r_] = acc + 0.5 * (a1 + a2);
                }
                double acc = qvj;
                NWT_UNROLL for (int e2 = 0; e2 < NU; ++e2) acc += 0.5 * (s_Q[c * NZS + NX + e2] + s_Q[(NX + e2) * NZS + c]) * s_kf[e2];
                // (every read of the old V of this stage -- T and vt -- lies before the barriers above)
                NWT_UNROLL for (int r_ = 0; r_ < NX; ++r_) { s_V[r_ * NXS + c] = vnew[r_]; Vs[(size_t)k * NX * NX + r_ * NX + c] = vnew[r_]; }
                s_v[c] = acc;
                vs[(size_t)k * NX + c] = acc;
            }
            NWT_SYNC();
        }
        NWT_SYNC();
        if (!s_flag) break;
        // wrong inertia: next delta
        if (attempt == 0) delta = (dlast == 0.0) ? 1e-4 : fmax(1e-20, dlast / 3.0);
        else delta *= (dlast == 0.0) ? 100.0 : 8.0;
        ++attempt;
        if (delta > 1e40) {
            if (lane == 0) a.status[b] = ST_NUMERIC;
            for (int i = lane; i < NU; i += nt) U[(size_t)N * NU + i] = U[(size_t)(N - 1) * NU + i];   // CPDP.py:191 holds whatever the solver returned
            return;
        }
        NWT_SYNC();
    }
    if (lane == 0 && delta > 0.0) a.dlast[b] = delta;
#ifdef __CUDACC__
    __threadfence_block();
#endif
    NWT_SYNC();

    // ---- forward pass: step (dX, dU) and new multipliers (lane i < NX: row i)
    if (isX) { s_dx[jx] = dfc[jx]; dX[jx] = dfc[jx]; }
    NWT_SYNC();
    for (int k = 0; k < N; ++k) {
        const double* Kk = a.Kf + (ib + k) * NU * NX;
        const double* kfk = a.kf + (ib + k) * NU;
        const double* ABg = a.AB + (ib + k) * NX * NZ;
        // rows of K, V, [A B] for this lane: one batch of independent loads
        double kr[NX], vr[NX], ar[NZ];
        const int lu = (lane < NU) ? lane : 0;
        NWT_UNROLL for (int c = 0; c < NX; ++c) { kr[c] = Kk[lu * NX + c]; vr[c] = Vs[(size_t)k * NX * NX + c * NX + jx]; }   // (V is exactly symmetric: column jx = row jx, read coalesced)
        NWT_UNROLL for (int c = 0; c < NZ; ++c) ar[c] = ABg[jx * NZ + c];
        const double kf0 = kfk[lu], vs0 = vs[(size_t)k * NX + jx], df0 = dfc[(size_t)(k + 1) * NX + jx];
        if (lane < NU) {
            double acc = kf0;
            NWT_UNROLL for (int c = 0; c < NX; ++c) acc += kr[c] * s_dx[c];
            s_du[lane] = acc;
            dU[(size_t)k * NU + lane] = acc;
        }
        if (isX) {
            double acc = vs0;
            NWT_UNROLL for (int c = 0; c < NX; ++c) acc += vr[c] * s_dx[c];
            lamn[(size_t)k * NX + jx] = acc;
        }
        NWT_SYNC();
        double nx = 0.0;
        if (isX) {
            double acc = df0;
            NWT_UNROLL for (int c = 0; c < NX; ++c) acc += ar[c] * s_dx[c];
            NWT_UNROLL for (int c = 0; c < NU; ++c) acc += ar[NX + c] * s_du[c];
            nx = acc;
        }
        NWT_SYNC();
        if (isX) { s_dx[jx] = nx; dX[(size_t)(k + 1) * NX + jx] = nx; }
        NWT_SYNC();
    }
    if (isX) {
        double acc = vs[(size_t)N * NX + jx];
        NWT_UNROLL for (int c = 0; c < NX; ++c) acc += Vs[(size_t)N * NX * NX + jx * NX + c] * s_dx[c];
        lamn[(size_t)N * NX + jx] = acc;
    }
#ifdef __CUDACC__
    __threadfence_block();
#endif
    NWT_SYNC();

    // ---- directional derivative of the objective along the step
    double gd = 0.0, bad = 0.0;
    for (int i = lane; i < (N + 1) * NX; i += nt) if (!(fabs(lamn[i]) < 1e300)) bad = 1.0;
    for (int k = lane; k < N; k += nt) {
        const double* g = a.gq + (ib + k) * NZ;
        for (int i = 0; i < NX; ++i) gd += g[i] * dX[(size_t)k * NX + i];
        for (int i = 0; i < NU; ++i) gd += g[NX + i] * dU[(size_t)k * NU + i];
    }
    if constexpr (!HAS_BOUNDS) {
        for (int i = lane; i < NX; i += nt) gd += s_hx[i] * dX[(size_t)N * NX + i];
    } else {
        if (isX) gd += (s_hx[jx] + bgN) * dX[(size_t)N * NX + jx];
    }
    bad = nwt_reduce(bad, red, true);
    gd = nwt_reduce(gd, red, false);
    if (bad != 0.0 || !(gd == gd)) {
        if (lane == 0) a.status[b] = ST_NUMERIC;
        for (int i = lane; i < NU; i += nt) U[(size_t)N * NU + i] = U[(size_t)(N - 1) * NU + i];
        return;
    }

    // ---- fraction to the boundary, tau = max(0.99, 1 - mu): the largest primal step alpha_max and dual step alpha_z in (0, 1]
    //      that keep every slack / bound multiplier above (1 - tau) times its value
    double amax = 1.0, az = 1.0;
    if constexpr (HAS_BOUNDS) {
        const double tau = fmax(0.99, 1.0 - mu);
        double na = -1.0, nz = -1.0;               // -alpha_max, -alpha_z
        for (int idx = lane; idx < (N + 1) * NZ; idx += nt) {
            const int k = idx / NZ, j = idx % NZ;
            if (k == N && j >= NX) continue;
            const double w = (j < NX) ? X[(size_t)k * NX + j] : U[(size_t)k * NU + j - NX];
            const double dw = (j < NX) ? dX[(size_t)k * NX + j] : dU[(size_t)k * NU + j - NX];
            const double lb = ModelBounds<Model>::lo(j, pd0), ub = ModelBounds<Model>::hi(j, pd0);
            if (bnd_finite(lb)) {
                const double sl = w - lb, dz = bnd_dz(sl, zL[idx], mu, dw);
                if (dw < 0.0) na = fmax(na, tau * sl / dw);
                if (dz < 0.0) nz = fmax(nz, tau * zL[idx] / dz);
            }
            if (bnd_finite(ub)) {
                const double su = ub - w, dz = bnd_dz(su, zU[idx], mu, -dw);
                if (dw > 0.0) na = fmax(na, -(tau * su / dw));
                if (dz < 0.0) nz = fmax(nz, tau * zU[idx] / dz);
            }
        }
        amax = -nwt_reduce(na, red, true);
        az = -nwt_reduce(nz, red, true);
    }

    // ---- IPOPT filter line search (Waechter & Biegler 2006, Sec. 2.3; phi = J, theta = |g|_1, default constants
    //      gamma_theta 1e-5, gamma_phi 1e-8, delta 1, s_theta 1.1, s_phi 2.3, eta_phi 1e-8; no second-order
    //      correction, no restoration phase).  One lane per interval re-integrates the RK4 map at each trial point.
    const double th0 = g1;
    if (it == 0 && lane == 0) a.th_init[b] = fmax(1.0, th0);
#ifdef __CUDACC__
    __threadfence_block();
#endif
    NWT_SYNC();
    const double theta_min = 1e-4 * a.th_init[b], theta_max = 1e4 * a.th_init[b];
    int nf = a.nfilt[b];
    if constexpr (HAS_BOUNDS) { if (freset) nf = 0; }
    const double* filt = a.filt + (size_t)b * FILTER_CAP * 2;
    const double sw_rhs = pow(th0, 1.1);
    const double sw_lhs = (gd < 0) ? pow(-gd, 2.3) : 0.0;
    double alpha = amax;
    bool ok = false, ftype = false;
    for (int ls = 0; ls <= 30; ++ls) {
        double Jt = 0.0, gt = 0.0, lt = 0.0;
        for (int k = lane; k <= N; k += nt) {
            double xk[NX];
            PdBuf pdb;
            const double* pd = pd_at(pd0, grid_time(a.T, N, k), pdb);
            for (int i = 0; i < NX; ++i) xk[i] = X[(size_t)k * NX + i] + alpha * dX[(size_t)k * NX + i];
            if constexpr (HAS_BOUNDS) { NWT_UNROLL for (int i = 0; i < NX; ++i) lt += bnd_log(i, pd0, xk[i]); }
            if (k < N) {
                double uk[NU], xe[NX], q;
                for (int i = 0; i < NU; ++i) uk[i] = U[(size_t)k * NU + i] + alpha * dU[(size_t)k * NU + i];
                if constexpr (HAS_BOUNDS) { NWT_UNROLL for (int i = 0; i < NU; ++i) lt += bnd_log(NX + i, pd0, uk[i]); }
                rk4_interval(xk, uk, th, pd, DT, a.S, xe, q);
                Jt += q;
                for (int i = 0; i < NX; ++i)
                    gt += fabs(xe[i] - (X[(size_t)(k + 1) * NX + i] + alpha * dX[(size_t)(k + 1) * NX + i]));
            } else {
                double h, hx[NX];
                Model::term(xk, th, pd, h, hx);
                Jt += h;
            }
            if (k == 0) for (int i = 0; i < NX; ++i) gt += fabs(a.x0[(size_t)b * NX + i] - xk[i]);
        }
        Jt = nwt_reduce(Jt, red, false);
        gt = nwt_reduce(gt, red, false);
        if constexpr (HAS_BOUNDS) Jt -= mu * nwt_reduce(lt, red, false);        // barrier objective at the trial point
        bool acc = (Jt == Jt) && (gt == gt) && fabs(Jt) < 1e300 && gt <= theta_max;
        for (int e2 = 0; acc && e2 < nf; ++e2) if (gt >= filt[2 * e2] && Jt >= filt[2 * e2 + 1]) acc = false;
        if (acc) {
            const bool switching = (gd < 0) && (alpha * sw_lhs > sw_rhs);
            if (switching && th0 <= theta_min) {
                acc = (Jt <= P0 + 1e-8 * alpha * gd);
                ftype = acc;
            } else {
                acc = (gt <= (1 - 1e-5) * th0) || (Jt <= P0 - 1e-8 * th0);
            }
        }
        if (acc) { ok = true; break; }
        alpha *= 0.5;
    }
    if (!ok) {
        if (lane == 0) a.status[b] = ST_LINESEARCH;
        for (int i = lane; i < NU; i += nt) U[(size_t)N * NU + i] = U[(size_t)(N - 1) * NU + i];
        return;
    }
    if (!ftype && lane == 0 && nf < FILTER_CAP) {
        a.filt[((size_t)b * FILTER_CAP + nf) * 2] = (1 - 1e-5) * th0;
        a.filt[((size_t)b * FILTER_CAP + nf) * 2 + 1] = P0 - 1e-8 * th0;
        a.nfilt[b] = nf + 1;
    }

    // ---- update
    if constexpr (HAS_BOUNDS) {
        // z += alpha_z dz, then IPOPT's safeguard: z_L within [mu / (kappa_Sigma s_L), kappa_Sigma mu / s_L] at the new slack s_L,
        // kappa_Sigma = 1e10 (before the primal update below: the new slacks are formed here from the old values)
        for (int idx = lane; idx < (N + 1) * NZ; idx += nt) {
            const int k = idx / NZ, j = idx % NZ;
            if (k == N && j >= NX) continue;
            const double w = (j < NX) ? X[(size_t)k * NX + j] : U[(size_t)k * NU + j - NX];
            const double dw = (j < NX) ? dX[(size_t)k * NX + j] : dU[(size_t)k * NU + j - NX];
            const double wn = w + alpha * dw;
            const double lb = ModelBounds<Model>::lo(j, pd0), ub = ModelBounds<Model>::hi(j, pd0);
            if (bnd_finite(lb)) {
                const double z = zL[idx] + az * bnd_dz(w - lb, zL[idx], mu, dw), sn = wn - lb;
                zL[idx] = fmax(fmin(z, 1e10 * mu / sn), mu / (1e10 * sn));
            }
            if (bnd_finite(ub)) {
                const double z = zU[idx] + az * bnd_dz(ub - w, zU[idx], mu, -dw), sn = ub - wn;
                zU[idx] = fmax(fmin(z, 1e10 * mu / sn), mu / (1e10 * sn));
            }
        }
        NWT_SYNC();
    }
    for (int i = lane; i < (N + 1) * NX; i += nt) {
        X[i] += alpha * dX[i];
        Lam[i] += alpha * (lamn[i] - Lam[i]);
    }
    for (int i = lane; i < N * NU; i += nt) U[i] += alpha * dU[i];
    if (lane == 0) a.iters[b] = it + 1;
}

// One warp per problem walks the N stages serially (block LDL' of the KKT matrix, then the line search); a persistent grid
// strides over the compacted list of problems still iterating.
#ifndef CPDP_NEWTON_MINB
#define CPDP_NEWTON_MINB 8
#endif
CPDP_GLOBAL void __launch_bounds__(NEWTON_THREADS, CPDP_NEWTON_MINB) k_newton_step(SolveArgs a) {
    const int nact = *a.nact;
    for (int pi = blockIdx.x; pi < nact; pi += gridDim.x) {
        newton_step_problem(a, a.act[pi]);
        NWT_SYNC();
    }
}

// ---- starting point of the solve: the cold seed of k_solve_init and the pieces k_solve_init_warm (cpdp_warm.cuh) shares with it
constexpr double MU_COLD = 0.1;        // IPOPT's mu_init: barrier parameter of the cold start
constexpr double COLD_PUSH = 1e-2;     // IPOPT's bound_push = bound_frac of the cold start

// Per-problem solver state of a fresh solve (both starts).
CPDP_HD void start_state(const SolveArgs& a, size_t i) {
    a.status[i] = ST_RUNNING; a.iters[i] = 0; a.th_init[i] = 1.0; a.nfilt[i] = 0; a.dlast[i] = 0.0; a.J[i] = 0.0; a.kkt[i] = 0.0;
}

// IPOPT's projection of value w into the interior of its bounds lb, ub (fl, fu: the bound is finite and applies), with
// bound_push = bound_frac = kappa (Waechter & Biegler 2006, §3.6).
CPDP_HD double bnd_push(double lb, double ub, bool fl, bool fu, double w, double kappa) {
    const double pl = fl ? (fu ? fmin(kappa * fmax(1.0, fabs(lb)), kappa * (ub - lb)) : kappa * fmax(1.0, fabs(lb))) : 0.0;
    const double pu = fu ? (fl ? fmin(kappa * fmax(1.0, fabs(ub)), kappa * (ub - lb)) : kappa * fmax(1.0, fabs(ub))) : 0.0;
    if (fl && w < lb + pl) w = lb + pl;
    else if (fu && w > ub - pu) w = ub - pu;
    return w;
}

// Cold seed of component j of z = [x; u] in a row where it is a variable (var; row N holds the final state only): the zero seed
// (CPDP.py:139,155,167) pushed into the interior by bound_push = bound_frac = 1e-2, and z = 1 for every finite bound (0 else).
// k_solve_init spells out the same three statements: routing its stores through this helper changes its generated code.
CPDP_HD void cold_seed(int j, const double* pd, bool var, double& w, double& zl, double& zu) {
    const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
    const bool fl = var && bnd_finite(lb), fu = var && bnd_finite(ub);
    w = bnd_push(lb, ub, fl, fu, 0.0, COLD_PUSH);
    zl = fl ? 1.0 : 0.0;
    zu = fu ? 1.0 : 0.0;
}

// x0 outside a finite state bound cannot be reached: status CPDP_INFEASIBLE (both starts).  Bounds that depend on the problem's
// constants: also a component whose lb(pd) >= ub(pd) (or NaN), an empty box for that problem.
CPDP_HD void check_x0(const SolveArgs& a, size_t i) {
    const double* pd = pdata_of(a, (int)i);
    for (int j = 0; j < NX; ++j) {
        const double v = a.x0[i * NX + j], lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
        if ((bnd_finite(lb) && !(v > lb)) || (bnd_finite(ub) && !(v < ub))) a.status[i] = ST_INFEASIBLE;
    }
    if constexpr (BOUNDS_PD) {
        for (int j = 0; j < NZ; ++j)
            if (!(ModelBounds<Model>::lo(j, pd) < ModelBounds<Model>::hi(j, pd))) a.status[i] = ST_INFEASIBLE;
    }
}

// k_solve_init: zero seed (CPDP.py:139,155,167), multipliers 0, per-problem solver state.
CPDP_GLOBAL void k_solve_init(SolveArgs a) {
    const size_t tot = (size_t)a.B * (a.N + 1);
    const size_t gs = (size_t)gridDim.x * blockDim.x;
    if constexpr (!HAS_BOUNDS) {
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot * NX; i += gs) { a.X[i] = 0.0; a.Lam[i] = 0.0; }
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot * NU; i += gs) a.U[i] = 0.0;
    } else {
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot * NX; i += gs) a.Lam[i] = 0.0;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)a.B; i += gs) start_state(a, i);
    if constexpr (HAS_BOUNDS) {
        // IPOPT's start (Waechter & Biegler 2006, §3.6): cold_seed, mu = 0.1, check_x0
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot * NZ; i += gs) {
            const int j = (int)(i % NZ);
            const size_t k = i / NZ;
            const bool var = (k % (a.N + 1)) < (size_t)a.N || j < NX;           // (row N holds the final state only)
            const double* pd = pdata_of(a, (int)(k / (a.N + 1)));
            const double lb = ModelBounds<Model>::lo(j, pd), ub = ModelBounds<Model>::hi(j, pd);
            const bool fl = var && bnd_finite(lb), fu = var && bnd_finite(ub);
            const double w = bnd_push(lb, ub, fl, fu, 0.0, COLD_PUSH);
            if (j < NX) a.X[k * NX + j] = w; else a.U[k * NU + j - NX] = w;
            a.zL[i] = fl ? 1.0 : 0.0;
            a.zU[i] = fu ? 1.0 : 0.0;
        }
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)a.B; i += gs) {
            a.bmu[i] = MU_COLD;
            check_x0(a, i);
        }
    }
}

// k_dfma_probe: 8 independent DFMA chains per thread (FP64 pipe throughput probe for the bench roofline).
CPDP_GLOBAL void __launch_bounds__(256) k_dfma_probe(double* sink, int iters) {
    double a0 = 1.0 + threadIdx.x * 1e-9, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3, a4 = a0 + 4e-3, a5 = a0 + 5e-3,
           a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double m = 0.999999, c = 1e-7;
    for (int i = 0; i < iters; ++i) {
        a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
        a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
    }
    const double r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123.456) sink[0] = r;          // never true: keeps the chains alive
}

// k_compact: ordered list of the problems that are still iterating (single CTA).
constexpr int COMPACT_THREADS = 256;
CPDP_GLOBAL void __launch_bounds__(COMPACT_THREADS) k_compact(SolveArgs a) {
    CPDP_SHARED int s_cnt[COMPACT_THREADS + 1];
    const int tid = threadIdx.x;
    const int chunk = (a.B + COMPACT_THREADS - 1) / COMPACT_THREADS;
    const int lo = tid * chunk, hi = (lo + chunk < a.B) ? lo + chunk : a.B;
    int c = 0;
    for (int i = lo; i < hi; ++i) c += (a.status[i] == ST_RUNNING);
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
    for (int i = lo; i < hi; ++i) if (a.status[i] == ST_RUNNING) a.act[o++] = i;
}

}  // namespace CPDP_NS
