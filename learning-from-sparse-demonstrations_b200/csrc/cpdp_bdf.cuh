// Backward Riccati sweep with the integrator of the as-shipped reference: COCSys.auxSysSolver calls
// scipy.integrate.solve_ivp(method='BDF') once per grid interval at scipy's default tolerances
// (/root/reference/CPDP/CPDP.py:333-336).  This file re-implements that solver's control logic per problem, following
// scipy/integrate/_ivp/bdf.py of the scipy the oracle runs (1.18.1; the control flow is unchanged since the 1.6.1 the
// reference pins):
//   variable-order (1..5) NDF in quasi-constant-step form on the differences array D   bdf.py:314-453
//   change_D / compute_R on every step-size change                                       bdf.py:18-33
//   simplified Newton, <= 4 iterations, rate test, tol = max(10 eps/rtol, min(.03, sqrt(rtol)))   bdf.py:36-75,217
//   select_initial_step with order 1                                                     common.py:68-134
//   RMS error norm over the full vec(P), vec(W) state                                    common.py:63-65
//   LU kept across an error-test rejection, dropped on Newton failure / order change     bdf.py:377-407
//
// One deliberate difference.  scipy approximates the Jacobian of the right-hand side by finite differences (num_jac) and
// factorises the dense (n^2+nr)^2 matrix I - cJ.  The Riccati right-hand side is quadratic, so its Jacobian is known in
// closed form and has Kronecker structure: with L = A' - P R and C = R W - r_,
//     d(Pdot)[dP] = -(L dP + dP L')          d(Wdot)[dP, dW] = dP C - L dW .
// The Newton systems (I - cJ) dy = b are therefore solved exactly as
//     X + c (L X + X L') = B_P        (Bartels-Stewart through ONE Schur form L = Z T Z^H per Jacobian)
//     (I + c L) dW = B_W + c X C      (n x n inverse, rebuilt from the Schur form when c changes)
// i.e. with the same matrix the reference factorises up to its finite-difference error (~1e-8 relative).  Measured with
// scipy itself (jac = closed form vs jac = None on the stored quadrotor run): dL/dtheta moves by 2.2e-7 relative.
//
// SHAPE ON THE SM (round 2).  One warp per problem; lane c < NX + NP owns COLUMN c of the n x (n+r) state S = [P | W] in
// REGISTERS (full storage, as the reference's vec(P), vec(W)), and so do the Newton iterate, the correction d, psi and the
// error scale.  Every small product is then "matrix in shared memory (broadcast loads) times my register column" with NX
// independent accumulators: straight-line DFMA streams instead of the rolled, index-table driven shared-memory loops of the
// first version, whose lone-warp latency was 16 k cycles per right-hand side and 28 k per Newton solve (measured with
// clock64, tools/prof_bdf_phases.py).  Sparse model matrices (fx, fu, fe) are walked through compile-time COO lists that
// fold into the unrolled code.  Two-sided transforms A B A' are two applications of "multiply from the left, transpose
// through shared memory".  P is kept bitwise symmetric (commutative sums of separately rounded products, explicit
// symmetrisation of the Newton correction).  The differences array lives in an L2-resident workspace, [row][i][lane].
#pragma once
#include "cpdp_aux.cuh"

namespace CPDP_NS {

constexpr int BDF_THREADS = 32;
constexpr int NC = NX + NP;                      // columns of S = [P | W]: one lane each
static_assert(NC <= 32, "k_riccati_bdf maps one lane per column of [P | W]");
static_assert(NX <= 15 && NP <= 16, "warp sections map one lane per row/column and 16 + lane for the second half / the rows of Z; lane 31 must stay free for the bulge-chase fix-up");
#ifndef CPDP_BDF_MINB
#define CPDP_BDF_MINB 8
#endif
constexpr int BDF_MAX_ORDER = 5;
constexpr int BDF_NEWTON_MAXITER = 4;
constexpr int BDF_NROWS = BDF_MAX_ORDER + 3;
constexpr int BDF_WS_DOUBLES = BDF_NROWS * NX * NC;      // differences array of one problem, [row][i][c]

// code-size / instruction-level-parallelism knobs of the hot loop.  Measured (tools/prof_bdf_phases.py, 4096 OCPs / one OCP per SM):
// fully unrolled product + stencils x4: 183 ms / 20.0 ms; rolled: 141 ms / 21.1 ms -- eight warps per SM at different phases of
// the integrator share a 32 KB instruction cache, so code size beats instruction-level parallelism.
#ifndef CPDP_BDF_LMUL_UNROLL
#define CPDP_BDF_LMUL_UNROLL 1
#endif
#ifndef CPDP_BDF_STENCIL_UNROLL
#define CPDP_BDF_STENCIL_UNROLL 1
#endif
// Newton solves in the eigenbasis of L (bdf_eig_basis): taken for a Jacobian whose real eigenvector basis V has
// ||V||_F ||V^{-1}||_F <= CPDP_BDF_EIG_KAPPA; 0 compiles the eigen path out (every solve runs the Bartels-Stewart sweep).
#ifndef CPDP_BDF_EIG_KAPPA
#define CPDP_BDF_EIG_KAPPA 1e4
#endif
constexpr double BDF_EIG_KAPPA = CPDP_BDF_EIG_KAPPA;
// Warm start of the eigen path (bdf_eig_refine): a Jacobian that follows one on the eigen path first refines the previous
// eigenbasis and runs bdf_schur only when that is rejected; 0 compiles the refinement out (every Jacobian runs bdf_schur).
#ifndef CPDP_BDF_EIG_WARM
#define CPDP_BDF_EIG_WARM 1
#endif
#ifdef __CUDACC__
#define BDF_SYNC() __syncwarp()
#define BDF_UNROLL _Pragma("unroll")
#define BDF_PRAGMA_STR(x) _Pragma(#x)
#define BDF_PRAGMA_UNROLL(n) BDF_PRAGMA_STR(unroll n)
#else
#define BDF_SYNC() __syncthreads()
#define BDF_UNROLL
#define BDF_PRAGMA_UNROLL(n)
#endif

CPDP_HD double bdf_kappa(int k) { const double v[6] = {0.0, -0.1850, -1.0 / 9, -0.0823, -0.0415, 0.0}; return v[k]; }
// gamma_k = cumsum(1 / (1..k)) in double precision, as numpy accumulates it (bdf.py:244)
CPDP_HD double bdf_gamma(int k) { const double v[6] = {0.0, 1.0, 1.5, 1.8333333333333333, 2.083333333333333, 2.283333333333333}; return v[k]; }
CPDP_HD double bdf_alpha(int k) { return (1.0 - bdf_kappa(k)) * bdf_gamma(k); }
CPDP_HD double bdf_error_const(int k) { return bdf_kappa(k) * bdf_gamma(k) + 1.0 / (k + 1); }

// separately rounded product (keeps a*b + c*d commutative in its two terms: no FMA contraction)
#ifdef __CUDACC__
CPDP_D double bdf_mul(double a, double b) { return __dmul_rn(a, b); }
#else
CPDP_D double bdf_mul(double a, double b) { volatile double r = a * b; return r; }
#endif

// Shared-memory layout of one problem: compile-time offsets (in doubles) into the dynamic block.
constexpr int QS = (NX + 1) & ~1;                // row stride of the k-major product operands
constexpr int NCS = NC | 1;                      // odd row stride of the column exchange buffers (conflict-free transposes)
constexpr int SWQ = NX > 1 ? (NX - 1 + 3) / 4 : 1;   // Lyapunov sweep: terms per lane and sum (4 lanes per entry; >= 1: the eigen
                                                 // path's scratch in T2S needs a nonzero TW, and at NX = 1 every term is a stored zero)
constexpr int TW = 4 * SWQ;                      // row width of the skewed T: T2S[r][t] = T[r][r + 1 + t], zero beyond the matrix
constexpr int NH = (NX + 1) / 2;                 // rows per half in the two-halves products (lanes c and 16 + c)
namespace bo {
constexpr int M = 0;                             // PMP matrices at the current time + inverse of Huu
constexpr int XUL = M + ((MSZ + 1) & ~1);        // interpolated (x, u, lambda)
constexpr int RED = XUL + ((2 * NX + NU + 1) & ~1);   // reduction scratch (host emulation of the warp butterfly)
constexpr int Q = RED + 66;                      // real Schur vectors Q[k][i], row stride QS: k-major operand of Q' x
constexpr int QT = Q + NX * QS;                  // Q'[k][i] = Q[i][k]: k-major operand of Q x
constexpr int WT = QT + NX * QS;                 // ((I + c L)^{-1})'[k][i]: k-major operand of (I + cL)^{-1} x
constexpr int LM = WT + NX * QS;                 // L = A' - P R at the Jacobian point, row-major (kept for the "LU" events)
constexpr int Y2 = LM + ((NX * NX + 1) & ~1);    // Lyapunov sweep: right-hand side in, Hermitian solution out; complex, [k][j]
constexpr int T2S = Y2 + 2 * NX * NX;            // T = Z^H L Z above the diagonal, complex, skewed rows of width TW.  MUST follow
                                                 // Y2: the sweep's zero-weighted reads past Y2 land here (finite values)
constexpr int TD = T2S + 2 * NX * TW;            // diagonal of T, complex
constexpr int PV = TD + 2 * NX;                  // Lyapunov pivots 1 / (1 + c (t_ii + conj t_jj)), complex, [i][j], i <= j;
                                                 // during the Schur iteration: the plain n x n work arrays Tr | Ti
constexpr int CM = PV + 2 * NX * NX;             // C = R W - r_ at the Jacobian point, [NX][NP]
constexpr int XA = CM + ((NX * NP + 1) & ~1);    // column exchange buffers, [NX][NCS]
constexpr int XB = XA + NX * NCS;
constexpr int GHM = XB + NX * NCS;               // fu Huu^{-1}, [NX][NU]
constexpr int YPM = GHM + NX * NU;               // Huu^{-1} Y, [NU][NX]
constexpr int ROT = YPM + NU * NX;               // block rotations G: ga | gbr | gbi | partner   (4 x NX)
constexpr int RU = (ROT + 4 * NX + 1) & ~1;                 // change_D: RU | R | U, 6 x 6 each (also Householder vector scratch, sweep store dump: 128)
constexpr int FLAG = RU + 128;                   // 4 ints: prepare ok | Schur ok | first node row held in NODE | eigen path
constexpr int NODE = FLAG + 2;                   // the two node rows (x, u, lambda) bracketing the current grid interval
constexpr int NODE_W = 2 * NX + NU;
#ifdef CPDP_BDF_TIMING
constexpr int TS = NODE + ((2 * NODE_W + 1) & ~1);   // developer timing build: Schur sub-phase clocks (8; 6: warm refinement)
constexpr int END = TS + 8;
#else
constexpr int END = NODE + ((2 * NODE_W + 1) & ~1);
#endif
static_assert(Y2 % 2 == 0 && T2S % 2 == 0 && TD % 2 == 0 && PV % 2 == 0 && RU % 2 == 0, "complex arrays are read with 128-bit loads");
// eigen path (flag 3): Y2 holds V | Im x while the basis is built, then the coefficients k3 | k4 of the block solve; T2S holds
// V^{-1} while the basis is built, then the block solution Z (row stride QS); PV the coefficients k1 | k2; TD (a, b) per index
static_assert(2 * NX * NX <= T2S - Y2 && NX * NX <= 2 * NX * TW && NX * QS <= 2 * NX * TW, "eigen path scratch");
}  // namespace bo
constexpr int BDF_SMEM_DOUBLES = bo::END;
constexpr size_t BDF_SMEM_BYTES = (size_t)BDF_SMEM_DOUBLES * sizeof(double);

struct cplx { double x, y; };                    // (host emulation has no double2)
#ifdef __CUDACC__
#define BDF_LD2(p) (*reinterpret_cast<const double2*>(p))
#define BDF_ST2(p, a, b) (*reinterpret_cast<double2*>(p) = make_double2((a), (b)))
#else
#define BDF_LD2(p) (*reinterpret_cast<const cplx*>(p))
#define BDF_ST2(p, a, b) do { (p)[0] = (a); (p)[1] = (b); } while (0)
#endif

#define BDF_SM() CPDP_DYN_SMEM(sm)

// warp-wide sum / max returned to every lane (xor butterfly; the host emulation walks the same tree through shared memory)
CPDP_D_NOINLINE double bdf_reduce(double v, bool is_max) {
#ifdef __CUDACC__
    BDF_UNROLL for (int o = 16; o > 0; o >>= 1) {
        const double x = __shfl_xor_sync(0xffffffffu, v, o);
        v = is_max ? fmax(v, x) : (v + x);
    }
    return v;
#else
    BDF_SM();
    return block_reduce(v, sm + bo::RED, is_max);
#endif
}
CPDP_D_NOINLINE double bdf_pow(double x, double y) { return pow(x, y); }
// reciprocal of a positive, normal number to ~1 ulp: hardware seed + two Newton steps (5 instructions instead of the 20+ of an
// IEEE division; used for the error scale 1 / (atol + rtol |y|), where the last bit does not matter)
CPDP_D double bdf_rcp(double x) {
#ifdef __CUDACC__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
#else
    return 1.0 / x;
#endif
}

// Developer instrumentation (-DCPDP_BDF_TIMING): per-phase clock64() totals of each problem, written over the Ua rows of
// the problem at kernel end (phases = 1 runs only; tools/prof_bdf_phases.py).  Off in the shipped library.
#ifdef CPDP_BDF_TIMING
#define BDF_T(ph, ...) do { const long long t0__ = clock64(); __VA_ARGS__; tp[ph] += clock64() - t0__; } while (0)
#define BDF_TB(ph, var, expr) do { const long long t0__ = clock64(); var = (expr); tp[ph] += clock64() - t0__; } while (0)
#define BDF_TP_PARAM , long long* tp
#define BDF_TP_ARG , tp
#define BDF_TS0() const long long ts0__ = clock64()
#define BDF_TS(i) do { if (threadIdx.x == 0) sm[bo::TS + (i)] += (double)(clock64() - ts0__); } while (0)
#else
#define BDF_T(ph, ...) do { __VA_ARGS__; } while (0)
#define BDF_TB(ph, var, expr) do { var = (expr); } while (0)
#define BDF_TP_PARAM
#define BDF_TP_ARG
#define BDF_TS0()
#define BDF_TS(i)
#endif
// Developer path counts (-DCPDP_BDF_PATH_COUNTS, implied by the timing build): Newton solves on the eigen path | on the
// sweep, Jacobians on the eigen path | on the sweep, Jacobians whose warm refinement was accepted | rejected, written over
// Ua[24..29] of the problem at kernel end.
#ifdef CPDP_BDF_TIMING
#define CPDP_BDF_PATH_COUNTS
#endif
#ifdef CPDP_BDF_PATH_COUNTS
#define BDF_PATH(sm, k) do { cnt[4 + (k) + ((BDF_EIG_KAPPA > 0.0 && ((const int*)((sm) + bo::FLAG))[3]) ? 0 : 1)] += 1; } while (0)
#define BDF_WARM(dk) do { cnt[8] += (dk) == 2; cnt[9] += (dk) == 3; } while (0)
#else
#define BDF_PATH(sm, k) do { } while (0)
#define BDF_WARM(dk) do { } while (0)
#endif

// THE product of the hot loop, one out-of-line instance:  dst[(i0 + i) * ds] = sum_k AT[k][i0 + i] x[k * xs],  i < NH.
// All operands in shared memory; AT is k-major with row stride `as` (broadcast loads), x a column (stride NCS) or a row
// (stride 1) of an exchange buffer.  Two lanes share one output column (rows [0, NH) and [NX - NH, NX)), so a 13 x 13 product
// occupies 26 lanes with 7 independent accumulator chains each; k is fully unrolled (every load in flight at once) --
// affordable because this is the only copy.  Summation order: ascending k.
template <int AS>
CPDP_D_NOINLINE void bdf_lmul_t(const double* __restrict__ AT, const double* __restrict__ x, const int xs,
                                double* __restrict__ dst, const int ds, const int i0) {
    double out[NH];
    BDF_UNROLL for (int i = 0; i < NH; ++i) out[i] = 0.0;
    const double* A0 = AT + i0;
    BDF_PRAGMA_UNROLL(CPDP_BDF_LMUL_UNROLL) for (int k = 0; k < NX; ++k) {
        const double xk = x[k * xs];
        if constexpr (AS % 2 == 0 && (NX - NH) % 2 == 0) {           // rows of A start 16-byte aligned in both halves
            double a[NH + 1];
            BDF_UNROLL for (int i = 0; i + 1 < NH + 1; i += 2) { const auto v = BDF_LD2(A0 + k * AS + i); a[i] = v.x; a[i + 1] = v.y; }
            BDF_UNROLL for (int i = 0; i < NH; ++i) out[i] += a[i] * xk;
        } else {
            BDF_UNROLL for (int i = 0; i < NH; ++i) out[i] += A0[k * AS + i] * xk;
        }
    }
    // (for odd NX the two halves overlap in one row: the second half leaves it to the first)
    const int first = (i0 > 0) ? 2 * NH - NX : 0;
    BDF_UNROLL for (int i = 0; i < NH; ++i) if (i >= first) dst[(i0 + i) * ds] = out[i];
}
CPDP_D void bdf_lmul_to(const double* AT, const int as, const double* x, const int xs, double* dst, const int ds, const int i0) {
    if (as == QS) bdf_lmul_t<QS>(AT, x, xs, dst, ds, i0);        // (as is a literal at every call site: one branch survives)
    else bdf_lmul_t<NCS>(AT, x, xs, dst, ds, i0);
}
// lane -> (column, first row) of the two-halves mapping; false for idle lanes
CPDP_D bool bdf_half(const int lane, int& col, int& i0) {
    col = lane & 15;
    i0 = (lane >> 4) ? NX - NH : 0;
    return col < NX;
}
// column exchange helpers: buf is [NX][NCS]
CPDP_D void bdf_put(double* buf, int c, const double (&v)[NX]) {
    BDF_UNROLL for (int i = 0; i < NX; ++i) buf[i * NCS + c] = v[i];
}
CPDP_D void bdf_get_col(const double* buf, int c, double (&v)[NX]) {
    BDF_UNROLL for (int i = 0; i < NX; ++i) v[i] = buf[i * NCS + c];
}

// ------------------------------------------------------------------------------------------------
// PMP matrices at time t (CPDP.py:317-323: opt_sol(t) by linear interp1d, then the derivative set of diffPMP)
// ------------------------------------------------------------------------------------------------
// rows lo, lo + 1 of the node tables X, U, Lam for the grid interval that starts (backwards) at t0: one batch of loads per
// interval instead of two dependent global loads per lane in every step's bdf_prepare
CPDP_D void bdf_stage_nodes(double* sm, const AuxProblem& p, const double t0) {
    const int lane = threadIdx.x;
    const int lo = interp_lo(t0, p.dt, p.N);
    BDF_SYNC();
    CPDP_LOOP for (int q = lane; q < 2 * bo::NODE_W; q += BDF_THREADS) {
        const int row = lo + q / bo::NODE_W, e = q % bo::NODE_W;
        sm[bo::NODE + q] = (e < NX) ? p.X[(size_t)row * NX + e]
                         : (e < NX + NU) ? p.U[(size_t)row * NU + e - NX] : p.Lam[(size_t)row * NX + e - NX - NU];
    }
    if (lane == 0) ((int*)(sm + bo::FLAG))[2] = lo;
    BDF_SYNC();
}
CPDP_D_NOINLINE bool bdf_prepare(const AuxProblem p, const double t) {
    BDF_SM();
    const int lane = threadIdx.x;
    BDF_SYNC();
    int* flag = (int*)(sm + bo::FLAG);
    {   // xul_at through the interval's staged node rows (bdf_stage_nodes); a time outside them (the interval's end point belongs
        // to the previous pair of rows under interp1d's rule) reads global memory.  Same arithmetic either way.
        const int lo = interp_lo(t, p.dt, p.N);
        const bool hit = lo == flag[2];
        const double xlo = p.dt * lo, xhi = p.dt * (lo + 1);
        CPDP_LOOP for (int q = lane; q < bo::NODE_W; q += BDF_THREADS) {
            double v;
            if (hit) v = interp_val(sm[bo::NODE + q], sm[bo::NODE + bo::NODE_W + q], xlo, xhi, t);
            else v = xul_at(p, t, q);
            sm[bo::XUL + q] = v;
        }
    }
    BDF_SYNC();
    if (lane == 0) flag[0] = pmp_eval(p, sm + bo::XUL, sm + bo::M, t) ? 1 : 0;
    BDF_SYNC();
    return flag[0] != 0;
}

// ------------------------------------------------------------------------------------------------
// Riccati right-hand side (CPDP.py:262-274) on register columns, written without forming A, R, Q:
//   YZ = fu'[P|W] + [Hux|Hue],  Yp = Huu^{-1} Y
//   Pdot = -(Hxx + fx'P + (fx'P)' - sym(Y' Huu^{-1} Y))          Wdot = -fx'W - P fe - Hxe + Yp' Z
// ------------------------------------------------------------------------------------------------
CPDP_D void bdf_rhs_cols(double* sm, const double (&y)[NX], double (&f)[NX], const bool SYM) {
    const int c = threadIdx.x;
    const bool isP = c < NX, isW = (c >= NX) && (c < NC);
    const int k = isW ? c - NX : 0, cp = isP ? c : 0;
    const double* M = sm + bo::M;
    const double* fx = M + Model::PMP_FX; const double* fu = M + Model::PMP_FU; const double* fe = M + Model::PMP_FE;
    const double* Hxx = M + Model::PMP_HXX; const double* Hxu = M + Model::PMP_HXU; const double* Hxe = M + Model::PMP_HXE;
    const double* Hue = M + Model::PMP_HUE; const double* Hinv = M + Model::PMP_SIZE;
    double yz[NU], ypz[NU];
    BDF_UNROLL for (int a = 0; a < NU; ++a) yz[a] = isP ? Hxu[cp * NU + a] : Hue[a * NP + k];
    BDF_UNROLL for (int p = 0; p < Model::FU_nnz; ++p) yz[Model::FU_cooc(p)] += fu[Model::FU_coor(p) * NU + Model::FU_cooc(p)] * y[Model::FU_coor(p)];
    BDF_UNROLL for (int a = 0; a < NU; ++a) {
        double acc = 0.0;
        BDF_UNROLL for (int b2 = 0; b2 < NU; ++b2) acc += Hinv[a * NU + b2] * yz[b2];
        ypz[a] = acc;
    }
    double g[NX];
    BDF_UNROLL for (int i = 0; i < NX; ++i) g[i] = 0.0;
    BDF_UNROLL for (int p = 0; p < Model::FX_nnz; ++p) g[Model::FX_cooc(p)] += fx[Model::FX_coor(p) * NX + Model::FX_cooc(p)] * y[Model::FX_coor(p)];
    if (isP) {
        BDF_UNROLL for (int a = 0; a < NU; ++a) sm[bo::YPM + a * NX + c] = ypz[a];
        bdf_put(sm + bo::XA, c, g);                                      // XA[i][c] = (fx'P)[i][c]
        double pf[NP];                                                   // row c of P fe (P symmetric: P[c][a] = y[a])
        BDF_UNROLL for (int q = 0; q < NP; ++q) pf[q] = 0.0;
        BDF_UNROLL for (int p = 0; p < Model::FE_nnz; ++p) pf[Model::FE_cooc(p)] += y[Model::FE_coor(p)] * fe[Model::FE_coor(p) * NP + Model::FE_cooc(p)];
        BDF_UNROLL for (int q = 0; q < NP; ++q) sm[bo::XA + c * NCS + NX + q] = pf[q];
    }
    BDF_SYNC();
    // f[:, c] = -( [Hxx | Hxe][:, c] + (fx'S)[:, c] + [ (fx'P)' | P fe ][:, c] - Yp' YZ[:, c] )
    // (Hxx is emitted from one symbolic Hessian: entries (i, j) and (j, i) are the same expression, bitwise equal)
    const double* gb = sm + bo::XA + (isP ? c * NCS : c);              // (fx'P)[c][i]  |  (P fe)[i][k]
    const int gs = isP ? 1 : NCS;
    const double* hb = isP ? Hxx + cp : Hxe + k;
    const int hs = isP ? NX : NP;
    const double* yp = sm + bo::YPM;
    BDF_UNROLL for (int i = 0; i < NX; ++i) {
        double yy = 0.0;
        BDF_UNROLL for (int a = 0; a < NU; ++a) yy += yp[a * NX + i] * yz[a];
        f[i] = -(((g[i] + gb[i * gs]) + hb[i * hs]) - yy);
    }
    BDF_SYNC();
    if (SYM) {                                                           // bitwise symmetric P block
        if (isP) bdf_put(sm + bo::XA, c, f);
        BDF_SYNC();
        if (isP) { BDF_UNROLL for (int i = 0; i < NX; ++i) f[i] = 0.5 * (f[i] + sm[bo::XA + c * NCS + i]); }
        BDF_SYNC();
    }
}

// ------------------------------------------------------------------------------------------------
// Closed-form Jacobian data at (PMP matrices in shared memory, state columns y):  L = A' - P R -> LM (row-major),
// C = R W - r_ -> CM, with A = fx - G Hxu', R = G fu', r_ = fe - G Hue, G = fu Huu^{-1}   (CPDP.py:262-270)
// ------------------------------------------------------------------------------------------------
CPDP_D_NOINLINE void bdf_jacobian() {
    BDF_SM();
    const int c = threadIdx.x;
    const bool isP = c < NX, isW = (c >= NX) && (c < NC);
    const int k = isW ? c - NX : 0, cp = isP ? c : 0;
    const double* M = sm + bo::M;
    const double* fx = M + Model::PMP_FX; const double* fu = M + Model::PMP_FU; const double* fe = M + Model::PMP_FE;
    const double* Hxu = M + Model::PMP_HXU; const double* Hue = M + Model::PMP_HUE; const double* Hinv = M + Model::PMP_SIZE;
    double y[NX];
    bdf_get_col(sm + bo::XA, c < NC ? c : 0, y);                         // the caller parked the state columns in XA
    BDF_SYNC();
    if (isP) {                                                           // row c of G = fu Hinv
        CPDP_LOOP for (int a = 0; a < NU; ++a) {
            double acc = 0.0;
            BDF_UNROLL for (int b2 = 0; b2 < NU; ++b2) acc += fu[c * NU + b2] * Hinv[b2 * NU + a];
            sm[bo::GHM + c * NU + a] = acc;
        }
    }
    BDF_SYNC();
    const double* G = sm + bo::GHM;
    if (isP) {
        double pg[NU];                                                   // row c of P G
        BDF_UNROLL for (int a = 0; a < NU; ++a) {
            double acc = 0.0;
            BDF_UNROLL for (int b2 = 0; b2 < NX; ++b2) acc += y[b2] * G[b2 * NU + a];
            pg[a] = acc;
        }
        CPDP_LOOP for (int j = 0; j < NX; ++j) {                         // L[c][j] = A[j][c] - (P R)[c][j]
            double a1 = fx[j * NX + c];
            BDF_UNROLL for (int a = 0; a < NU; ++a) a1 -= G[j * NU + a] * Hxu[c * NU + a];
            double pr = 0.0;
            BDF_UNROLL for (int a = 0; a < NU; ++a) pr += pg[a] * fu[j * NU + a];
            sm[bo::LM + c * NX + j] = a1 - pr;
        }
    } else if (isW) {
        double z[NU];                                                    // column k of Z = fu'W + Hue
        BDF_UNROLL for (int a = 0; a < NU; ++a) {
            double acc = Hue[a * NP + k];
            BDF_UNROLL for (int b2 = 0; b2 < NX; ++b2) acc += fu[b2 * NU + a] * y[b2];
            z[a] = acc;
        }
        CPDP_LOOP for (int i = 0; i < NX; ++i) {                         // C[i][k] = sum_a G[i][a] z[a] - fe[i][k]
            double acc = -fe[i * NP + k];
            BDF_UNROLL for (int a = 0; a < NU; ++a) acc += G[i * NU + a] * z[a];
            sm[bo::CM + i * NP + k] = acc;
        }
    }
    (void)cp;
    BDF_SYNC();
}

// ------------------------------------------------------------------------------------------------
// Schur form by the warp: Givens reduction to Hessenberg form, Francis double-shift QR in real arithmetic (2 x 2 blocks left
// as they come), then one complex Givens rotation per 2 x 2 block.
// H: in L, out quasi-upper-triangular T (exact zeros below the sub-diagonal); Z: out orthogonal, L = Z T Z'.
// ------------------------------------------------------------------------------------------------
// warp vote / broadcast (host emulation: through the reduction scratch)
CPDP_D unsigned bdf_ballot(double* sm, bool pred) {
#ifdef __CUDACC__
    (void)sm;
    return __ballot_sync(0xffffffffu, pred);
#else
    unsigned* w = (unsigned*)(sm + bo::RED);
    __syncthreads();
    w[threadIdx.x] = pred ? 1u : 0u;
    __syncthreads();
    unsigned m = 0;
    for (int i = 0; i < 32; ++i) m |= w[i] << i;
    __syncthreads();
    return m;
#endif
}
CPDP_D double bdf_bcast(double* sm, double v, int src) {
#ifdef __CUDACC__
    (void)sm;
    return __shfl_sync(0xffffffffu, v, src);
#else
    double* w = sm + bo::RED;
    __syncthreads();
    w[threadIdx.x] = v;
    __syncthreads();
    const double r = w[src];
    __syncthreads();
    return r;
#endif
}
// lane holding the largest key among the lanes with pred (ties: the highest lane); key = 0 everywhere -> -1
CPDP_D int bdf_argmax(double* sm, double v, bool pred) {
#ifdef __CUDACC__
    (void)sm;
    const unsigned key = pred ? (unsigned)__double2hiint(fabs(v)) : 0u;      // high word: monotonic for non-negative doubles
    const unsigned mx = __reduce_max_sync(0xffffffffu, key);
    if (mx == 0u) return -1;
    return 31 - __clz((int)__ballot_sync(0xffffffffu, key == mx));
#else
    double* w = sm + bo::RED;
    __syncthreads();
    w[threadIdx.x] = pred ? fabs(v) : -1.0;
    __syncthreads();
    int best = -1; unsigned bk = 0;
    for (int i = 0; i < 32; ++i) {
        if (w[i] < 0.0) continue;
        unsigned long long bits; memcpy(&bits, &w[i], 8);
        const unsigned key = (unsigned)(bits >> 32);
        if (key != 0u && key >= bk) { bk = key; best = i; }
    }
    __syncthreads();
    return best;
#endif
}
CPDP_D int bdf_top_bit(unsigned m) {            // index of the highest set bit (m != 0)
#ifdef __CUDACC__
    return 31 - __clz((int)m);
#else
    int b = 31;
    while (!((m >> b) & 1u)) --b;
    return b;
#endif
}
// 1 / sqrt(x) for a positive, normal x to ~1 ulp: hardware seed + two Newton steps (the reflectors of the bulge chase are built
// from it: any consistent scaling gives an orthogonal reflector to rounding)
CPDP_D double bdf_rsqrt(double x) {
#ifdef __CUDACC__
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double hx = 0.5 * x;
    r = fma(r, fma(-hx * r, r, 0.5), r);
    r = fma(r, fma(-hx * r, r, 0.5), r);
    return r;
#else
    return 1.0 / sqrt(x);
#endif
}

// Real Schur form by the warp.  H: in L, out quasi-upper-triangular T (exact zeros below the sub-diagonal); Z: out
// orthogonal, L = Z T Z'.  vb: NX doubles of scratch.
//   Hessenberg form by Householder reflections (column-owned left application, row-owned right application);
//   Francis double-shift QR (EISPACK hqr2 control flow) with the deflation / start-row scans done by all lanes in parallel
//   (one vote each) and reflectors from one rsqrt + one reciprocal; two warp barriers per bulge step.
#ifdef CPDP_SCHUR_STATS
#include <cstdio>
struct SchurStats { long long calls = 0, sweeps = 0, steps = 0, exc = 0, maxits = 0; ~SchurStats() { fprintf(stderr, "SCHUR calls %lld sweeps %lld steps %lld exceptional %lld max its %lld\n", calls, sweeps, steps, exc, maxits); } };
static SchurStats g_ss;
#define SS(...) do { if (threadIdx.x == 0) { __VA_ARGS__; } } while (0)
#else
#define SS(...)
#endif
CPDP_D bool schur_real_w0(double* sm, double* H, double* Z, double* vb) {
    SS(g_ss.calls++);
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const double EPS = 2.220446049250313e-16;
#define h_(i, j) H[(i) * n + (j)]
    const int rw = lane & 15;                                      // lanes 0..15: row rw of H, lanes 16..31: row rw of Z
    double* const Mrow = (rw < n) ? ((lane < 16) ? H : Z) + rw * n : vb;      // (lanes without a row: scratch nobody writes in the chase)
    for (int i = lane; i < n * n; i += 32) Z[i] = (i / n == i % n) ? 1.0 : 0.0;
    BDF_SYNC();
    // ---- Hessenberg form
    { BDF_TS0();
    CPDP_LOOP for (int j = 0; j < n - 2; ++j) {
        double sig = 0.0;
        BDF_UNROLL for (int i = 0; i < n; ++i) { const double v = h_(i, j); sig += (i >= j + 2) ? v * v : 0.0; }
        if (sig == 0.0) continue;                                  // (uniform: every lane read the same values)
        const double alpha = h_(j + 1, j);
        const double nrm = sqrt(alpha * alpha + sig);
        const double beta_ = (alpha >= 0.0) ? -nrm : nrm;
        const double v0 = alpha - beta_;
        const double tau = 2.0 / (v0 * v0 + sig);
        BDF_SYNC();
        if (lane < n) vb[lane] = (lane <= j) ? 0.0 : (lane == j + 1 ? v0 : h_(lane, j));
        BDF_SYNC();
        if (lane >= j && lane < n) {                               // H <- (I - tau v v') H, my column
            double w = 0.0;
            BDF_UNROLL for (int i = 0; i < n; ++i) w += vb[i] * h_(i, lane);
            w *= tau;
            if (lane == j) {
                BDF_UNROLL for (int i = 0; i < n; ++i) if (i > j) h_(i, j) = (i == j + 1) ? beta_ : 0.0;
            } else {
                BDF_UNROLL for (int i = 0; i < n; ++i) h_(i, lane) -= vb[i] * w;
            }
        }
        BDF_SYNC();
        if (rw < n) {                                              // H <- H (I - tau v v') and Z <- Z (I - tau v v'): my row of H / of Z,
            double u = 0.0;                                        // one instruction stream for both halves of the warp
            BDF_UNROLL for (int k = 0; k < n; ++k) u += Mrow[k] * vb[k];
            u *= tau;
            BDF_UNROLL for (int k = 0; k < n; ++k) Mrow[k] -= u * vb[k];
        }
        BDF_SYNC();
    }
    BDF_TS(0); }
    double norm = 0.0;
    if (lane < n) { BDF_UNROLL for (int jj = 0; jj < n; ++jj) norm += (jj + 1 >= lane) ? fabs(h_(lane, jj)) : 0.0; }
    norm = bdf_reduce(norm, false);
    // ---- Francis double-shift QR sweeps, full Schur form (rows / columns updated over the whole matrix)
    int en = n - 1;
    while (en >= 0) {
        int its = 0;
        while (true) {
            BDF_TS0();
            int l = 0;
            {
                bool small = false;
                if (lane >= 1 && lane <= en) {
                    double s = fabs(h_(lane - 1, lane - 1)) + fabs(h_(lane, lane));
                    if (s == 0.0) s = norm;
                    small = fabs(h_(lane, lane - 1)) <= EPS * s;
                }
                const unsigned mk = bdf_ballot(sm, small);
                if (mk) l = bdf_top_bit(mk);
            }
            if (l == en) { BDF_SYNC(); if (lane == 0 && l >= 1) h_(l, l - 1) = 0.0; BDF_SYNC(); en -= 1; break; }
            if (l == en - 1) { BDF_SYNC(); if (lane == 0 && l >= 1) h_(l, l - 1) = 0.0; BDF_SYNC(); en -= 2; break; }
            if (its >= 600) return false;
            double x = h_(en, en), y = h_(en - 1, en - 1), w = h_(en, en - 1) * h_(en - 1, en);
            // exceptional shift every 14th sweep: blocks holding two nearly identical complex pairs (the x/y symmetry
            // of the quadrotor) converge only linearly under the standard shifts and can need > 100 sweeps
            SS(g_ss.sweeps++; if (its + 1 > g_ss.maxits) g_ss.maxits = its + 1);
            if (its > 0 && its % 14 == 0) {
                SS(g_ss.exc++);
                const double s = fabs(h_(en, en - 1)) + fabs(h_(en - 1, en - 2));
                x = y = 0.75 * s + h_(en, en);
                w = -0.4375 * s * s;
            }
            ++its;
            // start row m of the bulge: the largest m in [l, en-2] passing hqr2's small-subdiagonal test (m = l always does)
            int m;
            double p = 0.0, q = 0.0, r = 0.0;
            {
                bool pass = false;
                if (lane >= l && lane <= en - 2) {
                    const int mm = lane;
                    const double z = h_(mm, mm), r0 = x - z, s0 = y - z;
                    p = (r0 * s0 - w) / h_(mm + 1, mm) + h_(mm, mm + 1);
                    q = h_(mm + 1, mm + 1) - z - r0 - s0;
                    r = h_(mm + 2, mm + 1);
                    const double s = fabs(p) + fabs(q) + fabs(r);
                    if (s != 0.0) { const double is = 1.0 / s; p *= is; q *= is; r *= is; }
                    if (mm == l) pass = true;
                    else {
                        const double u = fabs(h_(mm, mm - 1)) * (fabs(q) + fabs(r));
                        const double v = fabs(p) * (fabs(h_(mm - 1, mm - 1)) + fabs(z) + fabs(h_(mm + 1, mm + 1)));
                        pass = (u <= EPS * v);
                    }
                }
                m = bdf_top_bit(bdf_ballot(sm, pass));
                p = bdf_bcast(sm, p, m); q = bdf_bcast(sm, q, m); r = bdf_bcast(sm, r, m);
            }
            BDF_SYNC();
            if (lane == 0 && l >= 1) h_(l, l - 1) = 0.0;
            BDF_TS(1);
            CPDP_LOOP for (int k = m; k <= en - 1; ++k) {
                const bool notlast = (k != en - 1);
                SS(g_ss.steps++);
                if (k != m) { p = h_(k, k - 1); q = h_(k + 1, k - 1); r = notlast ? h_(k + 2, k - 1) : 0.0; }
                const double sig = p * p + q * q + r * r;
                if (sig == 0.0) continue;                             // (uniform)
                const double rs = bdf_rsqrt(sig);
                const double sgn = (p < 0.0) ? -1.0 : 1.0;
                const double s = sgn * (sig * rs);
                const double xx = 1.0 + fabs(p) * rs, yy = q * rs * sgn, zz = r * rs * sgn;
                const double ixx = bdf_rcp(xx);                          // xx in [1, 2]
                const double qn = yy * ixx, rn = zz * ixx;
                {   // rows k .. k+2 of my column (columns >= k).  Branch-free: idle lanes compute on column k and store nothing
                    const bool on = lane >= k && lane < n;
                    double* const col = on ? H + lane : Z;             // (idle lanes: column 0 of Z, which this phase does not write)
                    const double a0 = col[k * n], a1 = col[(k + 1) * n], a2 = notlast ? col[(k + 2) * n] : 0.0;
                    const double pp = (a0 + qn * a1) + rn * a2;         // (a2 = 0 in the last step: adds an exact zero)
                    if (on && notlast) col[(k + 2) * n] = a2 - pp * zz;
                    if (on) col[k * n] = a0 - pp * xx;
                    if (on) col[(k + 1) * n] = a1 - pp * yy;
                }
                BDF_SYNC();
                {   // columns k .. k+2 of my row of H (rows <= imax) / of Z: one stream, branch-free
                    const int imax = (en < k + 3) ? en : k + 3;
                    const bool on = lane < 16 ? (rw <= imax) : (rw < n);
                    const double z0 = Mrow[k], z1 = Mrow[k + 1], z2 = notlast ? Mrow[k + 2] : 0.0;
                    const double pp = (xx * z0 + yy * z1) + zz * z2;
                    if (on && notlast) Mrow[k + 2] = z2 - pp * rn;
                    if (on) Mrow[k] = z0 - pp;
                    if (on) Mrow[k + 1] = z1 - pp * qn;
                    // column k-1 below the diagonal (every lane read it above, before the barrier; the two updates do not touch it)
                    if (lane == 31) {
                        if (k != m) { h_(k, k - 1) = -s; h_(k + 1, k - 1) = 0.0; if (notlast) h_(k + 2, k - 1) = 0.0; }
                        else if (l != m) h_(k, k - 1) = -h_(k, k - 1);
                    }
                }
                BDF_SYNC();
            }
            BDF_TS(2);                                                   // (scans + bulge chase of this sweep)
        }
    }
#undef h_
    return true;
}

// Real eigenvector basis of the quasi-triangular T of L = Q T Q' (row stride NX):  T = V D V^{-1}, D block diagonal with
// 1 x 1 blocks [lambda] and 2 x 2 blocks [[a, b], [-b, a]] on the columns [Re x, Im x] of the eigenvector x of a + ib (b > 0);
// a 2 x 2 block of T with real eigenvalues gives two 1 x 1 blocks.  V is block upper triangular on T's blocks, so V (complex
// back-substitution per eigenvalue, columns normalised) and V^{-1} (real back-substitution) take one column per lane, as
// LAPACK's dtrevc does.  Nothing is perturbed: a defective or nearly defective T shows as a non-finite or large
// ||V||_F ||V^{-1}||_F, and then nothing the sweep path reads is touched and the result is false (uniformly).  Otherwise
// G = Q V and H = V^{-1} Q' replace Q and Q' in the product slots (k-major H' in Q, G' in QT), TD holds (a, b) per index
// (b = 0 for a real eigenvalue) and ROT's partner row the other index of each complex pair.  The Q / QT slots hold Q on entry.
CPDP_D bool bdf_eig_basis(double* sm, const double* T) {
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool own = lane < n;
    const int j = own ? lane : 0;
    double* Vr = sm + bo::Y2; double* Vi = Vr + n * n; double* W = sm + bo::T2S;        // row stride n
    const bool up = j + 1 < n && T[(j + 1) * n + j] != 0.0, dn = j >= 1 && T[j * n + j - 1] != 0.0;
    const int bs = dn ? j - 1 : j, be = up ? j + 1 : j;                // my block of T
    double lr = T[j * n + j], li = 0.0;                                // my eigenvalue lr + i li
    double x0r = 1.0, x0i = 0.0, x1r = 0.0;                            // x on rows bs, be (x1 is real)
    bool cpx = false;
    if (bs != be) {
        const double p = T[bs * n + bs], q = T[bs * n + be], r = T[be * n + bs], s = T[be * n + be];
        const double hd = 0.5 * (p - s), disc = hd * hd + q * r;
        if (disc < 0.0) { cpx = true; li = sqrt(-disc); lr = s + hd; x0r = hd; x0i = li; x1r = r; }      // (lambda - s, r)
        else {
            const double sq = (hd >= 0.0) ? sqrt(disc) : -sqrt(disc);
            if (j == bs) { lr = s + (hd + sq); x0r = hd + sq; x1r = r; }                                 // (lambda - s, r)
            else { lr = p - (hd + sq); x0r = q; x1r = -(hd + sq); }                                        // (q, lambda - p)
        }
    }
    if (own) {
        CPDP_LOOP for (int i = 0; i < n; ++i) { Vr[i * n + j] = 0.0; Vi[i * n + j] = 0.0; }
        Vr[bs * n + j] = x0r; Vi[bs * n + j] = x0i;
        if (be != bs) Vr[be * n + j] = x1r;
    }
    // rows above my block, row blocks of T bottom-up: (T_II - lambda) x_I = -sum_{m > I} T_Im x_m
    for (int i = n - 1; i >= 0;) {
        const bool two = i >= 1 && T[i * n + i - 1] != 0.0;
        const int i0 = two ? i - 1 : i;
        if (own && i < bs) {
            double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;
            CPDP_LOOP for (int m = i + 1; m < n; ++m) {
                const double xr = Vr[m * n + j], xi = Vi[m * n + j], ta = T[i0 * n + m], tb = T[i * n + m];
                ar -= ta * xr; ai -= ta * xi; br -= tb * xr; bi -= tb * xi;
            }
            const double dr = T[i0 * n + i0] - lr, di = -li;
            double yr, yi;
            if (two) {                                                 // 2 x 2 complex system by Cramer's rule
                const double er = T[i * n + i] - lr, t01 = T[i0 * n + i], t10 = T[i * n + i0];
                const double gr = (dr * er - di * di) - t01 * t10, gi = dr * di + di * er;          // det
                const double ig = 1.0 / (gr * gr + gi * gi);
                const double ur = (ar * er - ai * di) - t01 * br, ui = (ar * di + ai * er) - t01 * bi;
                const double wr = (dr * br - di * bi) - t10 * ar, wi = (dr * bi + di * br) - t10 * ai;
                Vr[i0 * n + j] = (ur * gr + ui * gi) * ig; Vi[i0 * n + j] = (ui * gr - ur * gi) * ig;
                yr = (wr * gr + wi * gi) * ig; yi = (wi * gr - wr * gi) * ig;
            } else {
                const double ig = 1.0 / (dr * dr + di * di);
                yr = (ar * dr + ai * di) * ig; yi = (ai * dr - ar * di) * ig;
            }
            Vr[i * n + j] = yr; Vi[i * n + j] = yi;
        }
        i = i0 - 1;
    }
    if (own) {                                                         // column j of V: Re x, or Im x for the second of a pair
        double s2 = 0.0;
        CPDP_LOOP for (int m = 0; m < n; ++m) s2 += Vr[m * n + j] * Vr[m * n + j] + Vi[m * n + j] * Vi[m * n + j];
        const double sc = 1.0 / sqrt(s2);
        const double* src = (cpx && j == be) ? Vi : Vr;
        CPDP_LOOP for (int m = 0; m < n; ++m) Vr[m * n + j] = src[m * n + j] * sc;
    }
    BDF_SYNC();
    // column j of V^{-1}: V w = e_j, row blocks bottom-up
    for (int i = n - 1; i >= 0;) {
        const bool two = i >= 1 && T[i * n + i - 1] != 0.0;
        const int i0 = two ? i - 1 : i;
        if (own) {
            double a = (i0 == j) ? 1.0 : 0.0, b = (i == j) ? 1.0 : 0.0;
            CPDP_LOOP for (int m = i + 1; m < n; ++m) { const double w = W[m * n + j]; a -= Vr[i0 * n + m] * w; b -= Vr[i * n + m] * w; }
            if (two) {
                const double v00 = Vr[i0 * n + i0], v01 = Vr[i0 * n + i], v10 = Vr[i * n + i0], v11 = Vr[i * n + i];
                const double ig = 1.0 / (v00 * v11 - v01 * v10);
                W[i0 * n + j] = (a * v11 - v01 * b) * ig;
                W[i * n + j] = (v00 * b - v10 * a) * ig;
            } else {
                W[i * n + j] = a / Vr[i * n + i];
            }
        }
        i = i0 - 1;
    }
    double nv = 0.0, nw = 0.0;
    if (own) { CPDP_LOOP for (int m = 0; m < n; ++m) { nv += Vr[m * n + j] * Vr[m * n + j]; nw += W[m * n + j] * W[m * n + j]; } }
    nv = bdf_reduce(nv, false);
    nw = bdf_reduce(nw, false);
    if (!(nv * nw <= BDF_EIG_KAPPA * BDF_EIG_KAPPA)) return false;     // (NaN / inf fail the test too)
    // G = Q V -> XA[i][c];  H' = Q (V^{-1})' -> XB[k][i] = H[i][k]
    double* XA = sm + bo::XA; double* XB = sm + bo::XB;
    int hc, hi0;
    if (bdf_half(lane, hc, hi0)) {
        bdf_lmul_to(sm + bo::QT, QS, Vr + hc, n, XA + hc, NCS, hi0);
        bdf_lmul_to(sm + bo::QT, QS, W + hc * n, 1, XB + hc, NCS, hi0);
    }
    BDF_SYNC();
    CPDP_LOOP for (int e = lane; e < n * n; e += BDF_THREADS) {
        const int k = e / n, i = e % n;
        sm[bo::Q + k * QS + i] = XB[k * NCS + i];
        sm[bo::QT + k * QS + i] = XA[i * NCS + k];
    }
    if (own) {
        BDF_ST2(sm + bo::TD + 2 * j, lr, li);
        sm[bo::ROT + 3 * n + j] = (double)(cpx ? (j == bs ? be : bs) : j);
    }
    BDF_SYNC();
    return true;
}

// Complex Schur form L = Z T Z^H of the matrix in TR; result: T in (TR, TI), the real Schur vectors Q (and Q'), the block
// rotations G (Z = Q G^H) as per-row coefficients.  Returns false (uniformly) if the QR iteration did not converge.
CPDP_D_NOINLINE bool bdf_schur() {
    BDF_SM();
    constexpr int n = NX;
    const int lane = threadIdx.x;
    double* Tr = sm + bo::PV; double* Ti = Tr + n * n;                 // plain work arrays (the pivots are rebuilt by bdf_factor)
    double* Zm = sm + bo::Y2;                                          // Schur vectors, row stride n (scratch)
    double* ga = sm + bo::ROT; double* gbr = ga + n; double* gbi = gbr + n; double* pi = gbi + n;
    int* flag = (int*)(sm + bo::FLAG);
    BDF_SYNC();
    CPDP_LOOP for (int e = lane; e < n * n; e += BDF_THREADS) { Tr[e] = sm[bo::LM + e]; Ti[e] = 0.0; }
    if (lane == 0) flag[1] = 1;
    BDF_SYNC();
    const bool ok = schur_real_w0(sm, Tr, Zm, sm + bo::RU);
    BDF_SYNC();
    if (!ok && lane == 0) flag[1] = 0;
    // k-major product operands Q[k][i] (for Q' x) and QT[k][i] = Q[i][k] (for Q x)
    CPDP_LOOP for (int e = lane; e < n * n; e += BDF_THREADS) {
        const int r_ = e / n, c_ = e % n;
        const double v = Zm[e];
        sm[bo::Q + r_ * QS + c_] = v;
        sm[bo::QT + c_ * QS + r_] = v;
    }
    BDF_SYNC();
    if (BDF_EIG_KAPPA > 0.0) {
        BDF_TS0();
        const bool eig = ok && bdf_eig_basis(sm, Tr);
        if (lane == 0) flag[3] = eig ? 1 : 0;
        BDF_SYNC();
        BDF_TS(5);
        if (eig) return true;
    }
    BDF_TS0();
    // ---- one unitary rotation per 2 x 2 block:  G = [[c, s], [-conj(s), c]],  T <- G T G^H.  The Schur vectors stay REAL;
    //      the block-diagonal unitary factor is kept as per-index coefficients (Z = Q G^H):
    //      G[i][i] = ga[i] (real), G[i][pi[i]] = gb[i] (complex), pi[i] = the other index of i's block (or i).
    if (lane < n) { ga[lane] = 1.0; gbr[lane] = 0.0; gbi[lane] = 0.0; pi[lane] = (double)lane; }
    BDF_SYNC();
    CPDP_LOOP for (int j = 0; ok && j < n - 1; ++j) {
        const double cc = Tr[(j + 1) * n + j];
        if (cc == 0.0) continue;
        const double a = Tr[j * n + j], b = Tr[j * n + j + 1], d = Tr[(j + 1) * n + j + 1];
        const double hd = 0.5 * (a - d), disc = hd * hd + b * cc;
        double v1r, v1i;                                           // eigenvector [lambda - d, cc]
        if (disc >= 0.0) { v1r = hd + (hd >= 0.0 ? sqrt(disc) : -sqrt(disc)); v1i = 0.0; }
        else { v1r = hd; v1i = sqrt(-disc); }
        const double av1 = sqrt(v1r * v1r + v1i * v1i);
        const double rho = sqrt(av1 * av1 + cc * cc);
        double cr, sr, si;
        if (av1 == 0.0) { cr = 0.0; sr = (cc >= 0.0) ? 1.0 : -1.0; si = 0.0; }
        else { cr = av1 / rho; sr = v1r * cc / (av1 * rho); si = v1i * cc / (av1 * rho); }
        BDF_SYNC();
        if (lane >= j && lane < n) {                               // rows j, j+1
            const int k = lane;
            const double xr = Tr[j * n + k], xi = Ti[j * n + k], yr = Tr[(j + 1) * n + k], yi = Ti[(j + 1) * n + k];
            Tr[j * n + k] = cr * xr + (sr * yr - si * yi);
            Ti[j * n + k] = cr * xi + (sr * yi + si * yr);
            Tr[(j + 1) * n + k] = cr * yr - (sr * xr + si * xi);
            Ti[(j + 1) * n + k] = cr * yi - (sr * xi - si * xr);
        }
        BDF_SYNC();
        if (lane <= j + 1) {                                       // columns j, j+1 of T
            const int k = lane;
            const double xr = Tr[k * n + j], xi = Ti[k * n + j], yr = Tr[k * n + j + 1], yi = Ti[k * n + j + 1];
            Tr[k * n + j] = cr * xr + (sr * yr + si * yi);
            Ti[k * n + j] = cr * xi + (sr * yi - si * yr);
            Tr[k * n + j + 1] = cr * yr - (sr * xr - si * xi);
            Ti[k * n + j + 1] = cr * yi - (sr * xi + si * xr);
        } else if (lane == 16) {
            ga[j] = cr; gbr[j] = sr; gbi[j] = si; pi[j] = (double)(j + 1);
            ga[j + 1] = cr; gbr[j + 1] = -sr; gbi[j + 1] = si; pi[j + 1] = (double)j;      // -conj(s)
        }
        BDF_SYNC();
        if (lane == 0) { Tr[(j + 1) * n + j] = 0.0; Ti[(j + 1) * n + j] = 0.0; }
        BDF_SYNC();
    }
    BDF_SYNC();
    BDF_TS(3);
    // T packed for the sweep
    CPDP_LOOP for (int e = lane; e < n * TW; e += BDF_THREADS) {
        const int r_ = e / TW, k = r_ + 1 + e % TW;
        BDF_ST2(sm + bo::T2S + 2 * e, k < n ? Tr[r_ * n + k] : 0.0, k < n ? Ti[r_ * n + k] : 0.0);
    }
    if (lane < n) BDF_ST2(sm + bo::TD + 2 * lane, Tr[lane * n + lane], Ti[lane * n + lane]);
    BDF_SYNC();
    BDF_TS(4);                                                           // (rotations + packing)
    return flag[1] != 0;
}

// 2 x 2 stencils of the block rotations on a matrix held in shared memory:
//   (G E G^H)[i][j]  for real symmetric E (row stride st)  ->  complex
CPDP_D void bdf_stencil_GEGh(const double* rot, const double* E, const int st, const int i, const int j, double& cr, double& ci) {
    constexpr int n = NX;
    const int pi = (int)rot[3 * n + i], pj = (int)rot[3 * n + j];
    const double gi_a = rot[i], gi_br = rot[n + i], gi_bi = rot[2 * n + i];            // G[i][i], G[i][pi]
    const double gj_a = rot[j], gj_br = rot[n + j], gj_bi = -rot[2 * n + j];           // conj(G[j][j]), conj(G[j][pj])
    const double c1 = E[i * st + j], c2 = E[pi * st + j], c3 = E[i * st + pj], c4 = E[pi * st + pj];
    const double ujr = gi_a * c1 + gi_br * c2, uji = gi_bi * c2;                       // u_b = G[i][i] E[i][b] + G[i][pi] E[pi][b]
    const double upr = gi_a * c3 + gi_br * c4, upi = gi_bi * c4;
    cr = ujr * gj_a + (upr * gj_br - upi * gj_bi);
    ci = uji * gj_a + (upr * gj_bi + upi * gj_br);
}
//   Re (G^H Y G)[i][j]  for the complex Y of the sweep
CPDP_D double bdf_stencil_GhYG(const double* rot, const double* Y, const int i, const int j) {
    constexpr int n = NX;
    const int pi = (int)rot[3 * n + i], pj = (int)rot[3 * n + j];
    const double ai_r = rot[i], ap_r = rot[n + pi], ap_i = -rot[2 * n + pi];           // conj(G[i][i]), conj(G[pi][i])
    const double bj_r = rot[j], bp_r = rot[n + pj], bp_i = rot[2 * n + pj];            // G[j][j], G[pj][j]
    const bool hi = (pi != i), hj = (pj != j);
    const auto y1 = BDF_LD2(Y + 2 * (i * n + j)), y2 = BDF_LD2(Y + 2 * (pi * n + j));
    const auto y3 = BDF_LD2(Y + 2 * (i * n + pj)), y4 = BDF_LD2(Y + 2 * (pi * n + pj));
    const double tjr = ai_r * y1.x + (hi ? (ap_r * y2.x - ap_i * y2.y) : 0.0);
    const double tpr = ai_r * y3.x + (hi ? (ap_r * y4.x - ap_i * y4.y) : 0.0), tpi = ai_r * y3.y + (hi ? (ap_r * y4.y + ap_i * y4.x) : 0.0);
    return tjr * bj_r + (hj ? (tpr * bp_r - tpi * bp_i) : 0.0);
}

// scipy's "LU" event on the eigen path.  In the eigenbasis the Lyapunov operator Z + c (D Z + Z D') splits into the blocks of
// D: for the index blocks I, J with eigenvalues a_I + i b_I (b = 0 for a real one) the parts of Z_IJ that commute and
// anticommute with the rotation generator are scaled by  w+ = 1 / (1 + c (l_I + conj l_J))  and  w- = 1 / (1 + c conj(l_I + l_J)),
// which gives every entry as  Z_ij = k1 B_ij + k2 B_pi,j + k3 B_i,pj + k4 B_pi,pj  (p: partner index, s = +1 / -1 for the
// first / second index of a pair, 0 for a real eigenvalue):
//   k1 = Re(w+ + w-) / 2,  k2 = s_i Im(w+ - w-) / 2,  k3 = -s_j Im(w+ + w-) / 2,  k4 = s_i s_j Re(w+ - w-) / 2.
// (I + c L)^{-1} = G (I + c D)^{-1} H: H's rows scaled block by block, one product with G.  Zero pivots: false, as below.
CPDP_D bool bdf_factor_eig(double* sm, const double c) {
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool own = lane < n;
    const int j = own ? lane : 0;
    const double* TD = sm + bo::TD; const double* part = sm + bo::ROT + 3 * n;
    double* s1 = sm + bo::ROT; double* s2 = s1 + n;                    // row scaling of (I + cD)^{-1}: own row | partner row
    double* XA = sm + bo::XA;
    BDF_SYNC();
    double bad = 0.0;
    if (own) {
        const auto lj = BDF_LD2(TD + 2 * j);
        const int pj = (int)part[j];
        const double sj = (pj > j) ? 1.0 : ((pj < j) ? -1.0 : 0.0);
        CPDP_LOOP for (int i = 0; i < n; ++i) {
            const auto li = BDF_LD2(TD + 2 * i);
            const int pi = (int)part[i];
            const double si = (pi > i) ? 1.0 : ((pi < i) ? -1.0 : 0.0);
            const double er = 1.0 + c * (li.x + lj.x), ep = c * (li.y - lj.y), em = -c * (li.y + lj.y);
            const double mp = er * er + ep * ep, mm = er * er + em * em;
            if (!(mp > 0.0) || !(mm > 0.0)) bad = 1.0;
            const double ip = 1.0 / mp, im = 1.0 / mm;
            const double u = er * ip, v = -ep * ip, w = er * im, t = -em * im;       // w+ = u + iv, w- = w + it
            BDF_ST2(sm + bo::PV + 2 * (i * n + j), 0.5 * (u + w), si * (0.5 * (v - t)));
            BDF_ST2(sm + bo::Y2 + 2 * (i * n + j), -sj * (0.5 * (v + t)), (si * sj) * (0.5 * (u - w)));
        }
        const double dr = 1.0 + c * lj.x, di = c * lj.y, md = dr * dr + di * di;      // 1 / (1 + c (a + ib))
        if (!(md > 0.0)) bad = 1.0;
        s1[j] = dr / md; s2[j] = sj * (-di / md);
    }
    BDF_SYNC();
    if (own) {                                                         // XA[i][k] = ((I + cD)^{-1} H)[i][k], my column k
        CPDP_LOOP for (int i = 0; i < n; ++i) XA[i * NCS + j] = s1[i] * sm[bo::Q + j * QS + i] + s2[i] * sm[bo::Q + j * QS + (int)part[i]];
    }
    BDF_SYNC();
    int hc, hi0;
    if (bdf_half(lane, hc, hi0)) bdf_lmul_to(sm + bo::QT, QS, XA + hc, NCS, sm + bo::WT + hc * QS, 1, hi0);     // WT[k][i] = Winv[i][k]
    BDF_SYNC();
    return !bdf_ballot(sm, bad != 0.0);
}

// A^{-1} by Gauss-Jordan elimination with partial pivoting on [A | I]: lane c < n owns column c of the left half (A in XA,
// written by the caller), lane 16 + c column c of the right half (XB).  Out: dstT[k][i] = A^{-1}[i][k] (row stride QS), XA
// and XB overwritten.  False (uniformly, dstT untouched) when a pivot column is zero.
CPDP_D_NOINLINE bool bdf_gauss_jordan(double* dstT) {
    BDF_SM();
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool isP = lane < n, isB = (lane >= 16) && (lane < 16 + n);
    double* XA = sm + bo::XA; double* XB = sm + bo::XB;
    if (isB) { BDF_UNROLL for (int i = 0; i < n; ++i) XB[i * NCS + lane - 16] = (i == lane - 16) ? 1.0 : 0.0; }
    double* mine = isP ? XA + lane : XB + (isB ? lane - 16 : 0);
    const bool own = isP || isB;
    BDF_SYNC();
    CPDP_LOOP for (int k = 0; k < n; ++k) {
        const int p = bdf_argmax(sm, (isP && lane >= k) ? XA[lane * NCS + k] : 0.0, isP && lane >= k);     // lane = candidate row
        if (p < 0) return false;                                 // (uniform)
        if (own && p != k) { const double a = mine[k * NCS], b = mine[p * NCS]; mine[k * NCS] = b; mine[p * NCS] = a; }
        BDF_SYNC();
        double ak[n];
        BDF_UNROLL for (int i = 0; i < n; ++i) ak[i] = XA[i * NCS + k];
        const double ip = bdf_rcp(XA[k * NCS + k]);              // (either sign; the argmax above made it the largest of its column)
        BDF_SYNC();
        if (own) {
            const double t = mine[k * NCS] * ip;
            BDF_UNROLL for (int i = 0; i < n; ++i) mine[i * NCS] -= ak[i] * t;
            mine[k * NCS] = t;                                   // (row k itself: the scaled pivot row)
        }
        BDF_SYNC();
    }
    if (isB) { BDF_UNROLL for (int i = 0; i < n; ++i) dstT[(lane - 16) * QS + i] = XB[i * NCS + lane - 16]; }
    BDF_SYNC();
    return true;
}

// scipy's "LU" event for a new c: the Lyapunov pivots of the sweep and (I + c L)^{-1} by Gauss-Jordan elimination on [I + cL | I]
CPDP_D_NOINLINE bool bdf_factor(const double c) {
    BDF_SM();
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool isP = lane < n;
    const double* TD = sm + bo::TD;
    double* XA = sm + bo::XA;
    if (BDF_EIG_KAPPA > 0.0 && ((const int*)(sm + bo::FLAG))[3]) return bdf_factor_eig(sm, c);
    BDF_SYNC();
    double bad = 0.0;
    if (isP) {
        const int j = lane;
        const auto tj = BDF_LD2(TD + 2 * j);
        CPDP_LOOP for (int i = 0; i <= j; ++i) {                 // 1 / ((1/2 + c t_ii) + conj(1/2 + c t_jj))
            const auto ti = BDF_LD2(TD + 2 * i);
            const double er = 1.0 + c * (ti.x + tj.x), ei = c * (ti.y - tj.y);
            const double ee = er * er + ei * ei;
            if (!(ee > 0.0)) bad = 1.0;
            const double ie = 1.0 / ee;
            BDF_ST2(sm + bo::PV + 2 * (i * n + j), er * ie, -ei * ie);
        }
        BDF_UNROLL for (int i = 0; i < n; ++i) XA[i * NCS + j] = ((i == j) ? 1.0 : 0.0) + c * sm[bo::LM + i * n + j];
    }
    if (!bdf_gauss_jordan(sm + bo::WT)) return false;           // WT[k][i] = Winv[i][k]
    return !bdf_ballot(sm, bad != 0.0);
}

// Warm start of the eigen path: L = G D H (H = G^{-1}, D real block diagonal as bdf_eig_basis leaves it) from the previous
// Jacobian's G, by Newton refinement of the similarity instead of a new Schur form.  One step:
//   H = G^{-1} (bdf_gauss_jordan),  M = H L G,  D = the part of M's diagonal blocks that commutes with the rotation
//   generator J = [[0, 1], [-1, 0]] (a = mean of the diagonal, b = (m01 - m10) / 2), and F from  D_I F_IJ - F_IJ D_J = -M_IJ
//   on every block pair: the parts of M_IJ that commute / anticommute with J are scaled by 1 / (l_I - l_J) and
//   1 / (l_I - conj l_J) (l = a + ib), which gives every entry as  F_ij = -(k1 M_ij + k2 M_pi,j + k3 M_i,pj + k4 M_pi,pj)
//   (p: partner index, s = +1 / -1 for the first / second index of a pair, 0 for a real eigenvalue):
//     k1 = Re(w+ + w-) / 2,  k2 = s_i Im(w+ + w-) / 2,  k3 = s_j Im(w- - w+) / 2,  k4 = s_i s_j Re(w+ - w-) / 2
//   with w+ = 1 / (l_I - l_J) (0 inside a block: its commuting part is D's) and w- = 1 / (l_I - conj l_J) (0 for a real
//   diagonal entry);  then G <- G + G F.
// The columns of G are first scaled by powers of two (exact; both columns of a pair by one factor) to unit norm within a factor
// of two.  Accepted when ||M - D||_F <= BDF_REFINE_TOL ||L||_F and ||G||_F ||H||_F <= CPDP_BDF_EIG_KAPPA (the cold path's
// conditions), with every pair still complex (b > 0); rejected, uniformly, when a step has max |F| > BDF_REFINE_FMAX or a
// non-finite F, or after BDF_REFINE_STEPS steps.  On accept H' (Q), G' (QT) and TD hold what bdf_eig_basis leaves there; the
// pair structure (ROT's partner row) is the previous Jacobian's.  On reject Q, QT, TD are garbage: bdf_schur rebuilds them from LM.
// Scratch: L' in PV, the products in XA / XB.
constexpr int BDF_REFINE_STEPS = 5;
constexpr double BDF_REFINE_FMAX = 0.5;
#ifndef CPDP_BDF_REFINE_TOL
#define CPDP_BDF_REFINE_TOL 1e-13     // the cold path's own ||H L G - D||_F / ||L||_F reaches 6.5e-14 on the quadrotor fixtures
#endif
constexpr double BDF_REFINE_TOL = CPDP_BDF_REFINE_TOL;
CPDP_D_NOINLINE bool bdf_eig_refine() {
    BDF_SM();
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool own = lane < n;
    const int j = own ? lane : 0;
    double* G = sm + bo::QT;                                           // G[i][k] = G[k * QS + i]: k-major operand of G x
    double* LT = sm + bo::PV;                                          // L[i][k] = LT[k * QS + i]
    double* XA = sm + bo::XA; double* XB = sm + bo::XB;
    const double* part = sm + bo::ROT + 3 * n;
    BDF_SYNC();
    const int pj = (int)part[j];
    const double sj = (pj > j) ? 1.0 : ((pj < j) ? -1.0 : 0.0);
    double nl = 0.0, s2 = 0.0;
    if (own) {
        CPDP_LOOP for (int i = 0; i < n; ++i) {
            const double v = sm[bo::LM + i * n + j], g = G[j * QS + i], gp = G[pj * QS + i];
            LT[j * QS + i] = v;
            nl += v * v;
            s2 += (pj != j) ? g * g + gp * gp : g * g;
        }
    }
    nl = bdf_reduce(nl, false);
    BDF_SYNC();
    if (own) {
        int e;
        (void)frexp(s2, &e);
        CPDP_LOOP for (int i = 0; i < n; ++i) G[j * QS + i] = ldexp(G[j * QS + i], -(e >> 1));
    }
    int hc, hi0;
    const bool hact = bdf_half(lane, hc, hi0);
    for (int it = 0;; ++it) {
        if (own) { BDF_UNROLL for (int i = 0; i < n; ++i) XA[i * NCS + j] = G[j * QS + i]; }
        if (!bdf_gauss_jordan(sm + bo::Q)) return false;            // Q[k][i] = H[i][k]
        if (hact) bdf_lmul_to(LT, QS, G + hc * QS, 1, XA + hc, NCS, hi0);              // (L G)[:, c]
        BDF_SYNC();
        if (hact) bdf_lmul_to(sm + bo::Q, QS, XA + hc, NCS, XB + hc, NCS, hi0);        // M[:, c] = H (L G)[:, c]
        BDF_SYNC();
        double a = 0.0, b = 0.0, res = 0.0, ng = 0.0, nh = 0.0;
        if (own) {
            if (pj == j) a = XB[j * NCS + j];
            else {
                const int f = (pj > j) ? j : pj, s = (pj > j) ? pj : j;
                a = 0.5 * (XB[f * NCS + f] + XB[s * NCS + s]);
                b = 0.5 * (XB[f * NCS + s] - XB[s * NCS + f]);
            }
            BDF_UNROLL for (int i = 0; i < n; ++i) {
                const double d = (i == j) ? a : ((i == pj) ? -sj * b : 0.0);
                const double r = XB[i * NCS + j] - d, g = G[j * QS + i], h = sm[bo::Q + j * QS + i];
                res += r * r; ng += g * g; nh += h * h;
            }
            BDF_ST2(sm + bo::TD + 2 * j, a, b);
        }
        res = bdf_reduce(res, false); ng = bdf_reduce(ng, false); nh = bdf_reduce(nh, false);
        if (bdf_ballot(sm, own && pj != j && !(b > 0.0))) return false;
        if (res <= (BDF_REFINE_TOL * BDF_REFINE_TOL) * nl) return ng * nh <= BDF_EIG_KAPPA * BDF_EIG_KAPPA;
        if (it == BDF_REFINE_STEPS) return false;
        BDF_SYNC();
        bool bad = false;
        if (own) {                                                     // column j of F -> XA
            const auto lj = BDF_LD2(sm + bo::TD + 2 * j);
            CPDP_LOOP for (int i = 0; i < n; ++i) {
                const auto li = BDF_LD2(sm + bo::TD + 2 * i);
                const int pi = (int)part[i];
                const double si = (pi > i) ? 1.0 : ((pi < i) ? -1.0 : 0.0);
                const bool blk = (i == j) || (i == pj);
                const double dr = li.x - lj.x, dp = li.y - lj.y, dm = li.y + lj.y;
                const double ip = blk ? 0.0 : 1.0 / (dr * dr + dp * dp);
                const double im = (i == j && pj == j) ? 0.0 : 1.0 / (dr * dr + dm * dm);
                const double ur = dr * ip, ui = -dp * ip, wr = dr * im, wi = -dm * im;     // w+ = ur + i ui, w- = wr + i wi
                const double k1 = 0.5 * (ur + wr), k2 = si * (0.5 * (ui + wi)), k3 = sj * (0.5 * (wi - ui)), k4 = (si * sj) * (0.5 * (ur - wr));
                const double f = -(((k1 * XB[i * NCS + j] + k2 * XB[pi * NCS + j]) + k3 * XB[i * NCS + pj]) + k4 * XB[pi * NCS + pj]);
                if (!(fabs(f) <= BDF_REFINE_FMAX)) bad = true;
                XA[i * NCS + j] = f;
            }
        }
        if (bdf_ballot(sm, bad)) return false;
        BDF_SYNC();
        if (hact) bdf_lmul_to(G, QS, XA + hc, NCS, XB + hc, NCS, hi0);                 // (G F)[:, c]
        BDF_SYNC();
        if (own) { BDF_UNROLL for (int i = 0; i < n; ++i) G[j * QS + i] += XB[i * NCS + j]; }
        BDF_SYNC();
    }
}

// A new Jacobian's decomposition: the warm refinement when the previous Jacobian took the eigen path, else (and when the
// refinement is rejected) the Schur form.  0: the QR iteration did not converge; 1: Schur form; 2: refinement accepted;
// 3: refinement rejected, then the Schur form.
#if CPDP_BDF_EIG_WARM
CPDP_D_NOINLINE int bdf_decompose() {
    BDF_SM();
    if (BDF_EIG_KAPPA > 0.0 && ((const int*)(sm + bo::FLAG))[3]) {
        BDF_TS0();
        const bool warm = bdf_eig_refine();
        BDF_TS(6);
        if (warm) return 2;
        return bdf_schur() ? 3 : 0;
    }
    return bdf_schur() ? 1 : 0;
}
#else
CPDP_D int bdf_decompose() { return bdf_schur() ? 1 : 0; }      // (the call sites of the Schur form as without the refinement)
#endif

// Lyapunov sweep  (1/2 + cT) Y + Y (1/2 + cT)^H = C  along anti-diagonals i + j = d, four lanes per entry.  C in Y2 (upper
// triangle), Y overwrites it, both triangles are kept (Y is Hermitian), so both sums of an entry have one form:
//   Y_ij / pivot_ij = C_ij - c ( S(i, j) + conj S(j, i) ),     S(r, s) = sum_{k > r} T_rk Y_ks .
// T is stored skewed (T2S[r][t] = T[r][r+1+t], zero beyond the matrix): every lane runs the same SWQ unconditional complex
// multiply-adds per sum at constant offsets from two base addresses; terms past the matrix multiply a stored zero (the Y
// operand of such a term may lie past Y2, inside T2S: finite).
CPDP_D void bdf_sweep(double* sm, const double c) {
    constexpr int n = NX;
    const int tid = threadIdx.x;
    const double* T2 = sm + bo::T2S; double* Y = sm + bo::Y2; const double* PVm = sm + bo::PV;
    const int e = tid >> 2, sub = tid & 3;
    // Lanes without an entry on the current anti-diagonal run on whatever their (i, j) addresses (all inside the kernel's
    // shared memory, see the asserts below) and store to a scratch slot, so the operand offsets of every lane move by
    // constants from one anti-diagonal to the next (above the main anti-diagonal the row index of an entry drops, below it
    // the column index does): they are carried in registers and stepped -- no address arithmetic behind the barrier.
    static_assert(bo::Y2 - 2 * 7 * NX >= 0 && bo::T2S - 2 * 8 * TW >= 0, "sweep: idle-lane operands below the arrays");
    static_assert(bo::Y2 + 2 * ((NX + 7 + 4 * SWQ) * NX + NX) <= bo::END && bo::T2S + 2 * ((NX + 7) * TW + 4 * SWQ) <= bo::END,
                  "sweep: idle-lane operands beyond the arrays");
    int d = 2 * (n - 1);
    int i = (n - 1) + e, j = d - i;                              // entry e of the first anti-diagonal (only e = 0 exists there)
#ifdef __CUDACC__
    int oti = 2 * (i * TW + sub), otj = 2 * (j * TW + sub);      // T rows i and j (my quarter of the terms)
    int oij = 2 * (i * n + j), oji = 2 * (j * n + i);            // entries (i, j) and (j, i)
    const int ysub = 2 * (1 + sub) * n;
#endif
    CPDP_LOOP for (; d >= 0; --d) {
        const bool valid = (i <= j) && (i >= 0);
#ifdef __CUDACC__
        // (idle lanes take their Y operands from the read-only arrays behind Y2 -- T2S, TD, PV: finite values, no store of this
        //  sweep lands there -- so no lane reads an entry another lane writes on the same anti-diagonal)
#ifdef CPDP_BDF_SWEEP_UNCLAMPED      // (developer A/B switch: idle lanes read wherever their stepped offsets point)
        const double* ta = T2 + oti; const double* ya = Y + oij + ysub;
        const double* tb = T2 + otj; const double* yb = Y + oji + ysub;
        const double* cvp = Y + oij; const double* pvp = PVm + oij;
#else
        const int rij = valid ? oij : 2 * n * n, rji = valid ? oji : 2 * n * n;
        const double* ta = T2 + (valid ? oti : 0); const double* ya = Y + rij + ysub;
        const double* tb = T2 + (valid ? otj : 0); const double* yb = Y + rji + ysub;
        const double* cvp = Y + ((valid && sub == 0) ? oij : 2 * n * n);      // (the right-hand side entry: read by the lane that stores)
        const double* pvp = PVm + oij;
#endif
#else
        const int ic = valid ? i : 0, jc = valid ? j : 0;        // (host emulation: idle lanes read entry (0, 0) -- no stray reads)
        const double* ta = T2 + 2 * (ic * TW + sub); const double* ya = Y + 2 * ((ic + 1 + sub) * n + jc);
        const double* tb = T2 + 2 * (jc * TW + sub); const double* yb = Y + 2 * ((jc + 1 + sub) * n + ic);
        const double* cvp = Y + 2 * (ic * n + jc); const double* pvp = PVm + 2 * (ic * n + jc);
#endif
        double pr[2 * SWQ], pi_[2 * SWQ];
        BDF_UNROLL for (int m = 0; m < SWQ; ++m) {
            const auto t1 = BDF_LD2(ta + 8 * m), y1 = BDF_LD2(ya + 8 * m * n);
            const auto t2 = BDF_LD2(tb + 8 * m), y2 = BDF_LD2(yb + 8 * m * n);
            pr[m] = t1.x * y1.x - t1.y * y1.y; pi_[m] = t1.x * y1.y + t1.y * y1.x;
            pr[SWQ + m] = t2.x * y2.x - t2.y * y2.y; pi_[SWQ + m] = -(t2.x * y2.y + t2.y * y2.x);      // conj S(j, i)
        }
        const auto cv = BDF_LD2(cvp), pv = BDF_LD2(pvp);
        // pairwise tree over the 2 SWQ products
        BDF_UNROLL for (int w = 1; w < 2 * SWQ; w *= 2) {
            BDF_UNROLL for (int m = 0; m + w < 2 * SWQ; m += 2 * w) { pr[m] += pr[m + w]; pi_[m] += pi_[m + w]; }
        }
        double ar = pr[0], ai = pi_[0];
#ifdef __CUDACC__
        ar += __shfl_xor_sync(0xffffffffu, ar, 1); ai += __shfl_xor_sync(0xffffffffu, ai, 1);
        ar += __shfl_xor_sync(0xffffffffu, ar, 2); ai += __shfl_xor_sync(0xffffffffu, ai, 2);
#else
        double* red = sm + bo::RED;
        __syncthreads();
        red[tid] = ar; red[32 + tid] = ai;
        __syncthreads();
        if (sub == 0) {
            ar = (red[tid] + red[tid + 1]) + (red[tid + 2] + red[tid + 3]);
            ai = (red[32 + tid] + red[32 + tid + 1]) + (red[32 + tid + 2] + red[32 + tid + 3]);
        }
#endif
        {   // branch-free: every lane forms the entry; lanes without one (and the mirror of a diagonal entry) store to a scratch slot
            const double rr = cv.x - c * ar, ri = cv.y - c * ai;
            const double yr = rr * pv.x - ri * pv.y, yi = rr * pv.y + ri * pv.x;
            const bool st = valid && (sub == 0);
            double* dump = sm + bo::RU + 2 * tid;                 // (change_D's scratch: free during a Newton solve)
#ifdef __CUDACC__
            double* p1 = st ? Y + oij : dump;
            double* p2 = (st && i != j) ? Y + oji : dump + 64;
#else
            double* p1 = st ? Y + 2 * (i * n + j) : dump;
            double* p2 = (st && i != j) ? Y + 2 * (j * n + i) : dump + 64;
#endif
            BDF_ST2(p1, yr, (i == j) ? 0.0 : yi);
            BDF_ST2(p2, yr, -yi);
        }
        // next anti-diagonal: d > n-1: the first row of the diagonal drops by one (i - 1, same j); else the column does
        const bool up = d > n - 1;
        if (up) --i; else --j;
#ifdef __CUDACC__
        oti -= up ? 2 * TW : 0; otj -= up ? 0 : 2 * TW;
        oij -= up ? 2 * n : 2; oji -= up ? 2 : 2 * n;
#endif
        BDF_SYNC();
    }
}

// r <- (I - cJ)^{-1} r   (r: my register column; right-hand side on entry, Newton correction on exit).  Between the stages
// the columns travel through the exchange buffers, so every product reads its operand vector from shared memory.
CPDP_D void bdf_solve_cols(double* sm, const double c, double (&r)[NX] BDF_TP_PARAM) {
    constexpr int n = NX;
    const int lane = threadIdx.x;
    const bool isP = lane < n, isW = (lane >= n) && (lane < NC);
    const int j = isP ? lane : 0;
    const double* rot = sm + bo::ROT;
    double* XA = sm + bo::XA; double* XB = sm + bo::XB;
    int hc, hi0;
    const bool hact = bdf_half(lane, hc, hi0);                   // products: lanes c and 16 + c share column c
    const bool eig = BDF_EIG_KAPPA > 0.0 && ((const int*)(sm + bo::FLAG))[3];     // (uniform)
    double* ZB = sm + bo::T2S;                                   // eigen path: Z, row stride QS
    BDF_T(10, {
    if (isP) bdf_put(XA, j, r);
    BDF_SYNC();
    if (hact) bdf_lmul_to(sm + bo::Q, QS, XA + hc, NCS, XB + hc, NCS, hi0);        // (Q'B)[:, c]
    BDF_SYNC();
    if (hact) bdf_lmul_to(sm + bo::Q, QS, XB + hc * NCS, 1, XA + hc, NCS, hi0);    // Q'(row c of Q'B)' = row c (= column c) of E = Q'BQ
    BDF_SYNC();
    });
    if (eig) {
    BDF_T(9, {
    if (isP) {                                                   // Z = block-diagonal solve of E = H B' H' (bdf_factor_eig), my column
        const double* part = rot + 3 * n;
        const int pj = (int)part[j];
        CPDP_LOOP for (int i = 0; i < n; ++i) {
            const int pi = (int)part[i];
            const auto k12 = BDF_LD2(sm + bo::PV + 2 * (i * n + j)), k34 = BDF_LD2(sm + bo::Y2 + 2 * (i * n + j));
            ZB[i * QS + j] = ((k12.x * XA[i * NCS + j] + k12.y * XA[pi * NCS + j]) + k34.x * XA[i * NCS + pj]) + k34.y * XA[pi * NCS + pj];
        }
    }
    BDF_SYNC();
    });
    } else {
    BDF_T(11, {
    if (isP) {                                                   // C = G E G^H, upper triangle of my column -> sweep array
        BDF_PRAGMA_UNROLL(CPDP_BDF_STENCIL_UNROLL) for (int i = 0; i <= j; ++i) {
            double cr, ci;
            bdf_stencil_GEGh(rot, XA, NCS, i, j, cr, ci);
            BDF_ST2(sm + bo::Y2 + 2 * (i * n + j), cr, ci);
        }
    }
    BDF_SYNC();
    });
    BDF_T(12, { bdf_sweep(sm, c); BDF_SYNC(); });
    BDF_T(13, {
    if (isP) {                                                   // Yr = Re(G^H Y G), my column -> XA
        BDF_PRAGMA_UNROLL(CPDP_BDF_STENCIL_UNROLL) for (int i = 0; i < n; ++i) XA[i * NCS + j] = bdf_stencil_GhYG(rot, sm + bo::Y2, i, j);
    }
    BDF_SYNC();
    });
    }
    BDF_T(14, {
    if (hact) bdf_lmul_to(sm + bo::QT, QS, (eig ? ZB : XA) + hc, eig ? QS : NCS, XB + hc, NCS, hi0);     // (Q Yr)[:, c] | (G Z)[:, c]
    BDF_SYNC();
    if (hact) bdf_lmul_to(sm + bo::QT, QS, XB + hc * NCS, 1, XA + hc, NCS, hi0);   // row c of X = Q Yr Q':  XA[i][c] = X[c][i]
    BDF_SYNC();
    });
    BDF_T(15, {
    double xs_[NX];
    if (isP) { BDF_UNROLL for (int i = 0; i < n; ++i) xs_[i] = 0.5 * (XA[i * NCS + j] + XA[j * NCS + i]); }   // X <- (X + X') / 2
    BDF_SYNC();
    if (isP) {
        BDF_UNROLL for (int i = 0; i < n; ++i) r[i] = xs_[i];
        bdf_put(XA, j, r);                                       // XA = X, bitwise symmetric
    }
    BDF_SYNC();
    // dW = (I + cL)^{-1} (B_W + c X C), two lanes per W column.  (X C)[:, k] = X C[:, k]: X is symmetric, so X itself (XA,
    // row stride NCS) is the k-major operand of the product
    const int wc = lane & 15, wi0 = (lane >> 4) ? NX - NH : 0;
    if (wc < NP) bdf_lmul_to(XA, NCS, sm + bo::CM + wc, NP, XB + n + wc, NCS, wi0);
    BDF_SYNC();
    if (isW) { BDF_UNROLL for (int i = 0; i < n; ++i) XB[i * NCS + lane] = r[i] + c * XB[i * NCS + lane]; }
    BDF_SYNC();
    if (wc < NP) bdf_lmul_to(sm + bo::WT, QS, XB + n + wc, NCS, XA + n + wc, NCS, wi0);
    BDF_SYNC();
    if (isW) { BDF_UNROLL for (int i = 0; i < n; ++i) r[i] = XA[i * NCS + lane]; }
    BDF_SYNC();
    });
}

// change_D (bdf.py:18-33): D[:order+1] <- (R U)' D[:order+1]   (D in the global workspace, [row][i][lane])
CPDP_D_NOINLINE void bdf_change_D(double* D, const int order, const double factor) {
    BDF_SM();
    const int lane = threadIdx.x;
    double* RU = sm + bo::RU; double* R = RU + 36; double* U = RU + 72;         // 6 x 6 scratch
    BDF_SYNC();
    if (lane <= order) {                                    // column lane of R and U: cumprod down the rows (compute_R)
        const int j = lane;
        R[j] = 1.0; U[j] = 1.0;
        CPDP_LOOP for (int i = 1; i <= order; ++i) {
            R[i * 6 + j] = (j == 0) ? 0.0 : R[(i - 1) * 6 + j] * (((double)(i - 1) - factor * j) / i);
            U[i * 6 + j] = (j == 0) ? 0.0 : U[(i - 1) * 6 + j] * (((double)(i - 1) - (double)j) / i);
        }
    }
    BDF_SYNC();
    CPDP_LOOP for (int e = lane; e < 36; e += BDF_THREADS) {
        const int i = e / 6, j = e % 6;
        if (i <= order && j <= order) {
            double acc = 0.0;
            CPDP_LOOP for (int k = 0; k <= order; ++k) acc += R[i * 6 + k] * U[k * 6 + j];
            RU[i * 6 + j] = acc;
        }
    }
    BDF_SYNC();
    if (lane < NC) {
        CPDP_LOOP for (int q = 0; q < NX; ++q) {
            double* Dq = D + (size_t)q * NC + lane;
            double v[BDF_MAX_ORDER + 1];
            BDF_UNROLL for (int i = 0; i <= BDF_MAX_ORDER; ++i) v[i] = (i <= order) ? Dq[(size_t)i * NX * NC] : 0.0;
            BDF_UNROLL for (int i = 0; i <= BDF_MAX_ORDER; ++i) {
                if (i <= order) {
                    double acc = 0.0;
                    BDF_UNROLL for (int jj = 0; jj <= BDF_MAX_ORDER; ++jj) if (jj <= order) acc += RU[jj * 6 + i] * v[jj];
                    Dq[(size_t)i * NX * NC] = acc;
                }
            }
        }
    }
    BDF_SYNC();
}

// RMS norm over the FULL (n^2 + n r) state of mul * v * isc (isc = 1 / scale)
CPDP_D double bdf_norm_cols(const double (&v)[NX], const double (&isc)[NX], const double mul, const bool act) {
    double a = 0.0;
    if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) { const double x = mul * v[i] * isc[i]; a += x * x; } }
    return sqrt(bdf_reduce(a, false) / (double)NFULL_R);
}
// the same for a row of the differences array (global memory)
CPDP_D_NOINLINE double bdf_norm_row(const double* Drow, const double* iscm, const double mul) {
    const int lane = threadIdx.x;
    double a = 0.0;
    if (lane < NC) { BDF_UNROLL for (int i = 0; i < NX; ++i) { const double x = mul * Drow[(size_t)i * NC + lane] * iscm[i * NCS + lane]; a += x * x; } }
    return sqrt(bdf_reduce(a, false) / (double)NFULL_R);
}

// The one out-of-line instance of the right-hand side: state columns in through XB, derivative columns out through XB.
// sym: bitwise symmetric P block (start-up of an interval, where the value seeds the differences array).
CPDP_D_NOINLINE void bdf_rhs_smem(const bool sym) {
    BDF_SM();
    const int c = threadIdx.x < NC ? threadIdx.x : 0;
    double y[NX], f[NX];
    bdf_get_col(sm + bo::XB, c, y);
    BDF_SYNC();
    bdf_rhs_cols(sm, y, f, sym);
    if (threadIdx.x < NC) bdf_put(sm + bo::XB, c, f);
    BDF_SYNC();
}

// One grid interval [t0, t1] with scipy's BDF.  y: state columns in registers (in/out).  Returns 0 ok, 1 step too small,
// 2 non-finite, 4 singular Newton matrix.  cnt: [rhs evaluations, steps (accepted), LU factorisations, Jacobians]
CPDP_D int bdf_interval(double* sm, double* D, const AuxProblem& p, const double t0, const double t1,
                        const double rtol, const double atol, double (&y)[NX], int* cnt BDF_TP_PARAM) {
    const int lane = threadIdx.x;
    const bool act = lane < NC;
    const int lc = act ? lane : 0;
    const double dir = (t1 >= t0) ? 1.0 : -1.0;
    const double EPS = 2.220446049250313e-16;
#define D_(row, i) D[((size_t)(row) * NX + (i)) * NC + lc]
    bdf_stage_nodes(sm, p, t0);
    // ---- __init__ (bdf.py:200-257)
    { bool okp__; BDF_TB(0, okp__, bdf_prepare(p, t0)); if (!okp__) return 2; }
    double f0[NX];
    if (act) bdf_put(sm + bo::XA, lc, y);
    BDF_SYNC();
    BDF_T(2, bdf_jacobian()); ++cnt[3];                                  // reads the state columns from XA
    if (act) bdf_put(sm + bo::XB, lc, y);
    BDF_SYNC();
    BDF_T(1, bdf_rhs_smem(true)); ++cnt[0];
    bdf_get_col(sm + bo::XB, lc, f0);
    BDF_SYNC();
    { int dk__; BDF_TB(3, dk__, bdf_decompose()); if (!dk__) return 4; BDF_WARM(dk__); }
    BDF_PATH(sm, 2);
    double h_abs;
    {
        const double interval_length = fabs(t1 - t0);
        double a0 = 0.0, a1 = 0.0;
        double isc0[NX];
        BDF_UNROLL for (int i = 0; i < NX; ++i) isc0[i] = bdf_rcp(atol + fabs(y[i]) * rtol);
        if (act) {
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                a0 += (y[i] * isc0[i]) * (y[i] * isc0[i]);
                a1 += (f0[i] * isc0[i]) * (f0[i] * isc0[i]);
            }
        }
        const double d0 = sqrt(bdf_reduce(a0, false) / (double)NFULL_R);
        const double d1 = sqrt(bdf_reduce(a1, false) / (double)NFULL_R);
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, interval_length);
        double f1[NX];
        if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) f1[i] = y[i] + h0 * dir * f0[i]; bdf_put(sm + bo::XB, lc, f1); }
        { bool okp__; BDF_TB(0, okp__, bdf_prepare(p, t0 + h0 * dir)); if (!okp__) return 2; }
        BDF_T(1, bdf_rhs_smem(true)); ++cnt[0];
        bdf_get_col(sm + bo::XB, lc, f1);
        BDF_SYNC();
        double a2 = 0.0;
        if (act) {
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                const double v = (f1[i] - f0[i]) * isc0[i];
                a2 += v * v;
            }
        }
        const double d2 = sqrt(bdf_reduce(a2, false) / (double)NFULL_R) / h0;
        double h1;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
        else h1 = bdf_pow(0.01 / fmax(d1, d2), 1.0 / 2.0);       // order 1
        h_abs = fmin(fmin(100 * h0, h1), interval_length);
    }
    const double newton_tol = fmax(10 * EPS / rtol, fmin(0.03, sqrt(rtol)));
    if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) { D_(0, i) = y[i]; D_(1, i) = f0[i] * h_abs * dir; } }
    BDF_SYNC();
    int order = 1, n_equal_steps = 0;
    bool lu_valid = false;
    double c_lu = 0.0;                 // the c the current LU was built with (scipy keeps a stale LU after an error rejection)
    double t = t0;
    double d[NX], psi[NX], isc[NX];
    BDF_UNROLL for (int i = 0; i < NX; ++i) { d[i] = 0.0; psi[i] = 0.0; isc[i] = 0.0; }

    while (dir * (t - t1) < 0) {
        // ---- _step_impl (bdf.py:314-453)
        const double min_step = 10 * fabs(nextafter(t, dir * INFINITY) - t);
        if (h_abs < min_step) {
            BDF_T(7, bdf_change_D(D, order, min_step / h_abs));
            h_abs = min_step;
            n_equal_steps = 0;
        }
        bool current_jac = false;
        double t_new = t, error_norm = 0.0, safety = 0.0;
        int n_iter = 0;
        while (true) {
            if (h_abs < min_step) return 1;
            double h = h_abs * dir;
            t_new = t + h;
            if (dir * (t_new - t1) > 0) {
                t_new = t1;
                BDF_T(7, bdf_change_D(D, order, fabs(t_new - t) / h_abs));
                n_equal_steps = 0;
                lu_valid = false;
            }
            h = t_new - t;
            h_abs = fabs(h);
            const double al = bdf_alpha(order), ial = 1.0 / al;
            if (act) {
                double dk[NX];
                BDF_UNROLL for (int i = 0; i < NX; ++i) { y[i] = 0.0; psi[i] = 0.0; }
                CPDP_LOOP for (int k = 0; k <= order; ++k) {
                    const double gk = bdf_gamma(k);                          // gamma_0 = 0: psi += 0 * D[0] adds an exact zero
                    BDF_UNROLL for (int i = 0; i < NX; ++i) dk[i] = D_(k, i);
                    BDF_UNROLL for (int i = 0; i < NX; ++i) { y[i] += dk[i]; psi[i] += dk[i] * gk; }
                }
                BDF_UNROLL for (int i = 0; i < NX; ++i) {                // y = y_predict: the Newton iteration starts from it
                    isc[i] = bdf_rcp(atol + rtol * fabs(y[i]));
                    psi[i] = psi[i] * ial;
                }
            }
            { bool okp__; BDF_TB(0, okp__, bdf_prepare(p, t_new)); if (!okp__) return 2; }      // PMP matrices at t_new (every Newton iterate shares them)
            const double c = h / al;
            bool converged = false;
            while (!converged) {
                if (!lu_valid) {
                    { bool okf__; BDF_TB(4, okf__, bdf_factor(c)); if (!okf__) return 4; }
                    lu_valid = true; c_lu = c; ++cnt[2];
                }
                // ---- solve_bdf_system (bdf.py:36-75)
                BDF_UNROLL for (int i = 0; i < NX; ++i) d[i] = 0.0;
                double dy_norm_old = -1.0;
                int k = 0;
                CPDP_LOOP for (k = 0; k < BDF_NEWTON_MAXITER; ++k) {
                    double r[NX];
                    if (act) bdf_put(sm + bo::XB, lc, y);
                    BDF_SYNC();
                    BDF_T(1, bdf_rhs_smem(false)); ++cnt[0];
                    bdf_get_col(sm + bo::XB, lc, r);
                    bool fin = false;
                    BDF_UNROLL for (int i = 0; i < NX; ++i) {
                        if (act && !(fabs(r[i]) < 1e300)) fin = true;
                        r[i] = c * r[i] - psi[i] - d[i];
                    }
                    if (bdf_ballot(sm, fin)) break;
                    BDF_T(5, bdf_solve_cols(sm, c_lu, r BDF_TP_ARG));
                    BDF_PATH(sm, 0);
                    double dy_norm; BDF_TB(6, dy_norm, bdf_norm_cols(r, isc, 1.0, act));
                    const bool have_rate = dy_norm_old >= 0.0;
                    const double rate = have_rate ? dy_norm / dy_norm_old : 0.0;
                    double rpow = rate;                                  // rate ** (NEWTON_MAXITER - k), exponent 3, 2 or 1
                    if (BDF_NEWTON_MAXITER - k >= 2) rpow *= rate;
                    if (BDF_NEWTON_MAXITER - k >= 3) rpow *= rate;
                    static_assert(BDF_NEWTON_MAXITER == 4, "rate power above is written for exponents <= 3");
                    if (have_rate && (rate >= 1 || rpow / (1 - rate) * dy_norm > newton_tol)) break;
                    BDF_UNROLL for (int i = 0; i < NX; ++i) { y[i] += r[i]; d[i] += r[i]; }
                    if (dy_norm == 0 || (have_rate && rate / (1 - rate) * dy_norm < newton_tol)) { converged = true; break; }
                    dy_norm_old = dy_norm;
                }
                n_iter = (k < BDF_NEWTON_MAXITER) ? k + 1 : BDF_NEWTON_MAXITER;
                if (!converged) {
                    if (current_jac) break;
                    // back to y_predict (same sum, same order => same bits as above), Jacobian there (bdf.py:372)
                    if (act) {
                        BDF_UNROLL for (int i = 0; i < NX; ++i) y[i] = 0.0;
                        CPDP_LOOP for (int kk = 0; kk <= order; ++kk) { BDF_UNROLL for (int i = 0; i < NX; ++i) y[i] += D_(kk, i); }
                        bdf_put(sm + bo::XA, lc, y);
                    }
                    BDF_SYNC();
                    BDF_T(2, bdf_jacobian()); ++cnt[3];
                    { int dk__; BDF_TB(3, dk__, bdf_decompose()); if (!dk__) return 4; BDF_WARM(dk__); }
                    BDF_PATH(sm, 2);
                    lu_valid = false;
                    current_jac = true;
                }
            }
            if (!converged) {
                h_abs *= 0.5;
                BDF_T(7, bdf_change_D(D, order, 0.5));
                n_equal_steps = 0;
                lu_valid = false;
                continue;
            }
            safety = 0.9 * (2 * BDF_NEWTON_MAXITER + 1) / (double)(2 * BDF_NEWTON_MAXITER + n_iter);
            BDF_UNROLL for (int i = 0; i < NX; ++i) isc[i] = bdf_rcp(atol + rtol * fabs(y[i]));
            BDF_TB(6, error_norm, bdf_norm_cols(d, isc, bdf_error_const(order), act));
            if (!(error_norm == error_norm)) return 2;
            if (error_norm > 1) {
                const double factor = fmax(0.2, safety * bdf_pow(error_norm, -1.0 / (order + 1)));
                h_abs *= factor;
                BDF_T(7, bdf_change_D(D, order, factor));
                n_equal_steps = 0;
                // LU deliberately kept (bdf.py:404-405)
            } else {
                break;
            }
        }
        ++n_equal_steps;
        ++cnt[1];
        t = t_new;
        // ---- update the differences (bdf.py:417-421)
        const bool sel_order = !(n_equal_steps < order + 1);
        if (act) {
            double up[NX];
            BDF_UNROLL for (int i = 0; i < NX; ++i) up[i] = D_(order + 1, i);
            BDF_UNROLL for (int i = 0; i < NX; ++i) { D_(order + 2, i) = d[i] - up[i]; D_(order + 1, i) = d[i]; up[i] = d[i]; }
            CPDP_LOOP for (int k = order; k >= 0; --k) {
                double cur[NX];
                BDF_UNROLL for (int i = 0; i < NX; ++i) cur[i] = D_(k, i);
                BDF_UNROLL for (int i = 0; i < NX; ++i) { up[i] += cur[i]; D_(k, i) = up[i]; }
            }
            if (sel_order) { BDF_UNROLL for (int i = 0; i < NX; ++i) sm[bo::XB + i * NCS + lc] = isc[i]; }
        }
        BDF_SYNC();
        if (!sel_order) continue;
        double error_m_norm = INFINITY, error_p_norm = INFINITY;
        if (order > 1) BDF_TB(6, error_m_norm, bdf_norm_row(D + (size_t)order * NX * NC, sm + bo::XB, bdf_error_const(order - 1)));
        if (order < BDF_MAX_ORDER) BDF_TB(6, error_p_norm, bdf_norm_row(D + (size_t)(order + 2) * NX * NC, sm + bo::XB, bdf_error_const(order + 1)));
        const double fm = bdf_pow(error_m_norm, -1.0 / order);
        const double f0_ = bdf_pow(error_norm, -1.0 / (order + 1));
        const double fp = bdf_pow(error_p_norm, -1.0 / (order + 2));
        int delta_order = -1; double fmaxv = fm;          // np.argmax: first maximum
        if (f0_ > fmaxv) { fmaxv = f0_; delta_order = 0; }
        if (fp > fmaxv) { fmaxv = fp; delta_order = 1; }
        order += delta_order;
        const double factor = fmin(10.0, safety * fmaxv);
        h_abs *= factor;
        BDF_T(7, bdf_change_D(D, order, factor));
        n_equal_steps = 0;
        lu_valid = false;
    }
    // solve_ivp(t_eval=[t1]) returns the dense output at the step end = D[0] (bdf.py:462-484)
    if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) y[i] = D_(0, i); }
    BDF_SYNC();
#undef D_
    return 0;
}

// k_riccati_bdf: backward sweep of COCSys.auxSysSolver as shipped (CPDP.py:327-338).
CPDP_GLOBAL void __launch_bounds__(BDF_THREADS, CPDP_BDF_MINB) k_riccati_bdf(AuxArgs a) {
    const int b = blockIdx.x, lane = threadIdx.x;
    if (a.solve_status && (a.solve_status[b] == ST_NUMERIC || a.solve_status[b] == ST_RUNNING ||
                           (HAS_BOUNDS && a.solve_status[b] == ST_INFEASIBLE))) {
        if (lane == 0) a.aux_status[b] = 3;
        return;
    }
    BDF_SM();
    const bool act = lane < NC, isP = lane < NX;
    const int lc = act ? lane : 0;
    CPDP_LOOP for (int q = lane; q < MSZ; q += BDF_THREADS) sm[bo::M + q] = 0.0;        // structural zeros of the PMP matrices
    double* D = a.Dws + (size_t)b * BDF_WS_DOUBLES;
    const int N = a.N;
    AuxProblem p;
    p.X = a.X + (size_t)b * (N + 1) * NX; p.U = a.U + (size_t)b * (N + 1) * NU; p.Lam = a.Lam + (size_t)b * (N + 1) * NX;
    p.th = a.theta + (size_t)b * a.theta_stride; p.pd = a.pdata + (size_t)b * NQ; p.PW = nullptr; p.dt = a.T / N; p.N = N;
    double* PW = a.PW + (size_t)b * (N + 1) * NYR;
    double* s_hxx = sm + bo::PV; double* s_hxe = sm + bo::XA;     // terminal condition staged in scratch (NX*NX and NX*NP doubles)
    if (lane == 0) {
        const double tN = p.dt * N;
        double xT[NX];
        const int lo = interp_lo(tN, p.dt, N);
        CPDP_LOOP for (int i = 0; i < NX; ++i) xT[i] = interp_val(p.X[(size_t)lo * NX + i], p.X[(size_t)(lo + 1) * NX + i], p.dt * lo, p.dt * (lo + 1), tN);
        PdBuf pdb;
        Model::term2(xT, p.th, pd_at(p.pd, tN, pdb), s_hxx, s_hxe);
    }
    BDF_SYNC();
    double y[NX];
    BDF_UNROLL for (int i = 0; i < NX; ++i) {
        // packed node table [upper-tri(P) | W] for the forward sweep; full, bitwise symmetric columns here
        y[i] = isP ? 0.5 * (s_hxx[i * NX + lc] + s_hxx[lc * NX + i]) : s_hxe[i * NP + (act ? lc - NX : 0)];
    }
    BDF_SYNC();
#define BDF_STORE_NODE(k_)                                                                              \
    if (act) {                                                                                          \
        BDF_UNROLL for (int i = 0; i < NX; ++i) {                                                       \
            if (isP) { if (i <= lc) PW[(size_t)(k_) * NYR + tri(i, lc)] = y[i]; }                       \
            else PW[(size_t)(k_) * NYR + NT + i * NP + (lc - NX)] = y[i];                               \
        }                                                                                               \
    }
    BDF_STORE_NODE(N)
    int cnt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};                   // (4..9: CPDP_BDF_PATH_COUNTS)
    if (lane == 0) ((int*)(sm + bo::FLAG))[3] = 0;                  // no eigenbasis to warm-start the first Jacobian from
    int st = 0;
#ifdef CPDP_BDF_TIMING
    long long tp[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (lane < 8) sm[bo::TS + lane] = 0.0;
    const long long tstart__ = clock64();
#endif
    CPDP_LOOP for (int k = N; k >= 1 && st == 0; --k) {
        st = bdf_interval(sm, D, p, p.dt * k, p.dt * (k - 1), a.rtol_b, a.atol_b, y, cnt BDF_TP_ARG);
        BDF_STORE_NODE(k - 1)
        BDF_SYNC();
    }
#undef BDF_STORE_NODE
#ifdef CPDP_BDF_TIMING
    if (lane == 0) {
        tp[8] = clock64() - tstart__;
        double* dst = a.Ua + (size_t)b * (N + 1) * NU * NP;
        for (int i = 0; i < 16; ++i) dst[i] = (double)tp[i];
        for (int i = 0; i < 8; ++i) dst[16 + i] = sm[bo::TS + i];
    }
#endif
#ifdef CPDP_BDF_PATH_COUNTS
    if (lane == 0) { for (int i = 0; i < 6; ++i) a.Ua[(size_t)b * (N + 1) * NU * NP + 24 + i] = (double)cnt[4 + i]; }
#endif
    if (lane == 0) {
        a.aux_status[b] = st;
        a.counters[b * NCOUNTERS + 0] = cnt[0]; a.counters[b * NCOUNTERS + 1] = cnt[1];
        a.counters[b * NCOUNTERS + 4] = cnt[2]; a.counters[b * NCOUNTERS + 5] = cnt[3];
    }
}


// ------------------------------------------------------------------------------------------------
// k_riccati_rk45: the backward sweep with scipy's RK45 (mode 0: `oracle_tight`, COCSys_TimeVarying as shipped, CPDP.py:740) in the
// shape of k_riccati_bdf -- one warp per problem, lane c owns column c of S = [P | W] in registers, the right-hand side is
// bdf_prepare + bdf_rhs_smem (bitwise symmetric P block), the seven stage derivatives of Dormand-Prince live in shared memory
// (over the arrays only the Newton solve of the BDF sweep uses, when they fit).  Control logic: rk.py:14-16, 111-170 and
// common.py:63-134, statement for statement as rk45_interval of cpdp_aux.cuh (the first version, 64-thread CTAs on a packed
// state in shared memory); the norms run over the full n x (n + r) state, as scipy's do.
// ------------------------------------------------------------------------------------------------
constexpr int RKW_K_DOUBLES = 7 * NX * NC;
constexpr bool RKW_K_OVERLAID = RKW_K_DOUBLES <= bo::XA - bo::Q;
constexpr int RKW_K = RKW_K_OVERLAID ? bo::Q : ((bo::END + 1) & ~1);
constexpr int RKW_SMEM_DOUBLES = RKW_K_OVERLAID ? bo::END : RKW_K + RKW_K_DOUBLES;
constexpr size_t RKW_SMEM_BYTES = (size_t)RKW_SMEM_DOUBLES * sizeof(double);

// K[stage] = f(t, yin); with_prepare = false reuses the PMP matrices of the previous call (same time)
CPDP_D bool rkw_rhs(double* sm, const AuxProblem& p, const double t, const bool with_prepare, const double (&yin)[NX], const int stage,
                    const bool act, const int lc) {
    if (with_prepare && !bdf_prepare(p, t)) return false;
    if (act) bdf_put(sm + bo::XB, lc, yin);
    BDF_SYNC();
    bdf_rhs_smem(true);
    if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) sm[RKW_K + (stage * NX + i) * NC + lc] = sm[bo::XB + i * NCS + lc]; }
    BDF_SYNC();
    return true;
}

CPDP_D int rkw_interval(double* sm, const AuxProblem& p, const double t0, const double t1, const double rtol, const double atol,
                        double (&y)[NX], int& nrhs, int& nsteps) {
    const int lane = threadIdx.x;
    const bool act = lane < NC;
    const int lc = act ? lane : 0;
    const double dir = (t1 >= t0) ? 1.0 : -1.0;
    const double NF = (double)NFULL_R;
#define K_(s_, i_) sm[RKW_K + ((s_) * NX + (i_)) * NC + lc]
    bdf_stage_nodes(sm, p, t0);
    if (!rkw_rhs(sm, p, t0, true, y, 0, act, lc)) return 2;
    ++nrhs;
    double h_abs;
    {   // select_initial_step (common.py:68-134), order = 4
        const double interval_length = fabs(t1 - t0);
        double a0 = 0.0, a1 = 0.0;
        if (act) {
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                const double sc = atol + fabs(y[i]) * rtol;
                const double f = K_(0, i);
                a0 += (y[i] / sc) * (y[i] / sc);
                a1 += (f / sc) * (f / sc);
            }
        }
        const double d0 = sqrt(bdf_reduce(a0, false) / NF);
        const double d1 = sqrt(bdf_reduce(a1, false) / NF);
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, interval_length);
        double ys[NX];
        BDF_UNROLL for (int i = 0; i < NX; ++i) ys[i] = act ? y[i] + h0 * dir * K_(0, i) : 0.0;
        if (!rkw_rhs(sm, p, t0 + h0 * dir, true, ys, 1, act, lc)) return 2;          // f1 parked in K[1]
        ++nrhs;
        double a2 = 0.0;
        if (act) {
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                const double sc = atol + fabs(y[i]) * rtol;
                const double v = (K_(1, i) - K_(0, i)) / sc;
                a2 += v * v;
            }
        }
        const double d2 = sqrt(bdf_reduce(a2, false) / NF) / h0;
        double h1;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
        else h1 = bdf_pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
        h_abs = fmin(fmin(100 * h0, h1), interval_length);
    }
    double t = t0;
    while (dir * (t - t1) < 0) {
        const double min_step = 10 * fabs(nextafter(t, dir * (double)INFINITY) - t);
        if (h_abs < min_step) h_abs = min_step;
        bool rejected = false;
        double t_new = t;
        double yn[NX];
        while (true) {
            if (h_abs < min_step) return 1;
            double h = h_abs * dir;
            t_new = t + h;
            if (dir * (t_new - t1) > 0) t_new = t1;
            h = t_new - t;
            h_abs = fabs(h);
            BDF_UNROLL for (int st = 1; st < 6; ++st) {
                double ys[NX];
                BDF_UNROLL for (int i = 0; i < NX; ++i) {
                    double acc = 0.0;
                    BDF_UNROLL for (int j = 0; j < st; ++j) acc += (act ? K_(j, i) : 0.0) * dp_A(st, j);
                    ys[i] = y[i] + acc * h;
                }
                if (!rkw_rhs(sm, p, t + dp_C(st) * h, true, ys, st, act, lc)) return 2;
                ++nrhs;
            }
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                double acc = 0.0;
                BDF_UNROLL for (int j = 0; j < 6; ++j) acc += (act ? K_(j, i) : 0.0) * dp_B(j);
                yn[i] = y[i] + h * acc;
            }
            if (!rkw_rhs(sm, p, t + dp_C(5) * h, false, yn, 6, act, lc)) return 2;     // (the time of stage 5: its PMP matrices are in place)
            ++nrhs;
            double ae = 0.0;
            bool fin = false;
            if (act) {
                BDF_UNROLL for (int i = 0; i < NX; ++i) {
                    double acc = 0.0;
                    BDF_UNROLL for (int j = 0; j < 7; ++j) acc += K_(j, i) * dp_E(j);
                    const double sc = atol + fmax(fabs(y[i]), fabs(yn[i])) * rtol;
                    const double v = acc * h / sc;
                    ae += v * v;
                    if (!(fabs(yn[i]) < 1e300)) fin = true;
                }
            }
            const double error_norm = sqrt(bdf_reduce(ae, false) / NF);
            if (bdf_ballot(sm, fin) || !(error_norm == error_norm)) return 2;
            ++nsteps;
            if (error_norm < 1) {
                double factor = (error_norm == 0) ? 10.0 : fmin(10.0, 0.9 * bdf_pow(error_norm, -0.2));
                if (rejected) factor = fmin(1.0, factor);
                h_abs *= factor;
                break;
            }
            h_abs *= fmax(0.2, 0.9 * bdf_pow(error_norm, -0.2));
            rejected = true;
        }
        t = t_new;
        BDF_UNROLL for (int i = 0; i < NX; ++i) y[i] = yn[i];
        if (act) { BDF_UNROLL for (int i = 0; i < NX; ++i) K_(0, i) = K_(6, i); }
        BDF_SYNC();
    }
#undef K_
    return 0;
}

CPDP_GLOBAL void __launch_bounds__(BDF_THREADS, CPDP_BDF_MINB) k_riccati_rk45(AuxArgs a) {
    const int b = blockIdx.x, lane = threadIdx.x;
    if (a.solve_status && (a.solve_status[b] == ST_NUMERIC || a.solve_status[b] == ST_RUNNING ||
                           (HAS_BOUNDS && a.solve_status[b] == ST_INFEASIBLE))) {
        if (lane == 0) a.aux_status[b] = 3;
        return;
    }
    BDF_SM();
    const bool act = lane < NC, isP = lane < NX;
    const int lc = act ? lane : 0;
    CPDP_LOOP for (int q = lane; q < MSZ; q += BDF_THREADS) sm[bo::M + q] = 0.0;        // structural zeros of the PMP matrices
    const int N = a.N;
    AuxProblem p;
    p.X = a.X + (size_t)b * (N + 1) * NX; p.U = a.U + (size_t)b * (N + 1) * NU; p.Lam = a.Lam + (size_t)b * (N + 1) * NX;
    p.th = a.theta + (size_t)b * a.theta_stride; p.pd = a.pdata + (size_t)b * NQ; p.PW = nullptr; p.dt = a.T / N; p.N = N;
    double* PW = a.PW + (size_t)b * (N + 1) * NYR;
    double* s_hxx = sm + bo::PV; double* s_hxe = sm + bo::XA;     // terminal condition (CPDP.py:327-331) staged in scratch
    if (lane == 0) {
        const double tN = p.dt * N;
        double xT[NX];
        const int lo = interp_lo(tN, p.dt, N);
        CPDP_LOOP for (int i = 0; i < NX; ++i) xT[i] = interp_val(p.X[(size_t)lo * NX + i], p.X[(size_t)(lo + 1) * NX + i], p.dt * lo, p.dt * (lo + 1), tN);
        PdBuf pdb;
        Model::term2(xT, p.th, pd_at(p.pd, tN, pdb), s_hxx, s_hxe);
    }
    BDF_SYNC();
    double y[NX];
    BDF_UNROLL for (int i = 0; i < NX; ++i) y[i] = isP ? 0.5 * (s_hxx[i * NX + lc] + s_hxx[lc * NX + i]) : s_hxe[i * NP + (act ? lc - NX : 0)];
    BDF_SYNC();
    int nrhs = 0, nsteps = 0, st = 0;
    CPDP_LOOP for (int k = N; k >= 0; --k) {
        if (act) {                                                  // packed node table [upper-tri(P) | W] for the forward sweep
            BDF_UNROLL for (int i = 0; i < NX; ++i) {
                if (isP) { if (i <= lc) PW[(size_t)k * NYR + tri(i, lc)] = y[i]; }
                else PW[(size_t)k * NYR + NT + i * NP + (lc - NX)] = y[i];
            }
        }
        if (k == 0) break;
        st = rkw_interval(sm, p, p.dt * k, p.dt * (k - 1), a.rtol_b, a.atol_b, y, nrhs, nsteps);
        BDF_SYNC();
        if (st != 0) break;
    }
    if (lane == 0) { a.aux_status[b] = st; a.counters[b * NCOUNTERS + 0] = nrhs; a.counters[b * NCOUNTERS + 1] = nsteps; }
}

}  // namespace CPDP_NS
