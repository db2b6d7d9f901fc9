// Probe of the Newton solve's warp linear algebra in csrc/cpdp_bdf.cuh (TEST INFRASTRUCTURE ONLY: the product never builds it).
// k_bdf_probe runs one warp per case over the UNMODIFIED device functions of the kernel, in the order bdf_interval calls them:
// a case is S steps, and each step writes L and C, decomposes L (bdf_decompose: warm refinement when the previous step left
// the eigen path, else the Schur form), factorises for c (bdf_factor) and solves the Newton system for the right-hand side
// [B_P | B_W] (bdf_solve_cols, lane c holding column c).  FLAG[3] is 0 before the first step and carried from step to step,
// as in k_riccati_bdf.  k_bdf_probe_gj inverts a matrix with bdf_gauss_jordan.  Included by tests/emu/emu_bdf_probe.cpp
// (thread emulation, g++) and tests/bdf_probe/bdf_probe.cu (nvcc, sm_100a) after the model header and cpdp_bdf.cuh.
#pragma once

namespace CPDP_NS {
namespace probe {
// one step of a case on input: L (NX x NX, row-major) | C (NX x NP) | c | B (NX x NC, column c = lane c's right-hand side)
constexpr int IN_L = 0;
constexpr int IN_C = IN_L + NX * NX;
constexpr int IN_CC = IN_C + NX * NP;
constexpr int IN_B = IN_CC + 1;
constexpr int IN_STEP = IN_B + NX * NC;
// one step on output: dk | FLAG[1] | FLAG[3] | factor's return value, then the decomposition as bdf_decompose leaves it
// (shared-memory slots copied verbatim: Q and QT [k][i] without the row padding, TD, ROT's four rows, T2S, and the Schur
// iteration's work arrays Tr | Ti in PV: the real quasi-triangular T on the eigen path, the complex triangular T on the sweep),
// WT [k][i], and the solved columns X | dW (NX x NC, column c from lane c)
constexpr int OUT_HDR = 0;
constexpr int OUT_Q = 4;
constexpr int OUT_QT = OUT_Q + NX * NX;
constexpr int OUT_TD = OUT_QT + NX * NX;
constexpr int OUT_ROT = OUT_TD + 2 * NX;
constexpr int OUT_T2S = OUT_ROT + 4 * NX;
constexpr int OUT_PV = OUT_T2S + 2 * NX * TW;
constexpr int OUT_WT = OUT_PV + 2 * NX * NX;
constexpr int OUT_R = OUT_WT + NX * NX;
constexpr int OUT_STEP = OUT_R + NX * NC;
}  // namespace probe

CPDP_GLOBAL void __launch_bounds__(BDF_THREADS) k_bdf_probe(const double* __restrict__ in, double* __restrict__ out, const int S) {
    BDF_SM();
    const int lane = threadIdx.x;
    const double* cin = in + (size_t)blockIdx.x * S * probe::IN_STEP;
    double* cout = out + (size_t)blockIdx.x * S * probe::OUT_STEP;
    int* flag = (int*)(sm + bo::FLAG);
    CPDP_LOOP for (int q = lane; q < BDF_SMEM_DOUBLES; q += BDF_THREADS) sm[q] = 0.0;
    BDF_SYNC();
    if (lane == 0) flag[3] = 0;
    for (int s = 0; s < S; ++s) {
        const double* x = cin + (size_t)s * probe::IN_STEP;
        double* o = cout + (size_t)s * probe::OUT_STEP;
        BDF_SYNC();
        CPDP_LOOP for (int q = lane; q < NX * NX; q += BDF_THREADS) sm[bo::LM + q] = x[probe::IN_L + q];
        CPDP_LOOP for (int q = lane; q < NX * NP; q += BDF_THREADS) sm[bo::CM + q] = x[probe::IN_C + q];
        BDF_SYNC();
        const int dk = bdf_decompose();
        BDF_SYNC();
        CPDP_LOOP for (int q = lane; q < NX * NX; q += BDF_THREADS) {
            const int k = q / NX, i = q % NX;
            o[probe::OUT_Q + q] = sm[bo::Q + k * QS + i];
            o[probe::OUT_QT + q] = sm[bo::QT + k * QS + i];
        }
        CPDP_LOOP for (int q = lane; q < 2 * NX; q += BDF_THREADS) o[probe::OUT_TD + q] = sm[bo::TD + q];
        CPDP_LOOP for (int q = lane; q < 4 * NX; q += BDF_THREADS) o[probe::OUT_ROT + q] = sm[bo::ROT + q];
        CPDP_LOOP for (int q = lane; q < 2 * NX * TW; q += BDF_THREADS) o[probe::OUT_T2S + q] = sm[bo::T2S + q];
        CPDP_LOOP for (int q = lane; q < 2 * NX * NX; q += BDF_THREADS) o[probe::OUT_PV + q] = sm[bo::PV + q];
        const double c = x[probe::IN_CC];
        BDF_SYNC();
        const bool fok = dk != 0 && bdf_factor(c);
        BDF_SYNC();
        double r[NX];
        BDF_UNROLL for (int i = 0; i < NX; ++i) r[i] = lane < NC ? x[probe::IN_B + i * NC + lane] : 0.0;
        if (fok) bdf_solve_cols(sm, c, r);
        BDF_SYNC();
        if (lane < NC) { BDF_UNROLL for (int i = 0; i < NX; ++i) o[probe::OUT_R + i * NC + lane] = fok ? r[i] : 0.0; }
        CPDP_LOOP for (int q = lane; q < NX * NX; q += BDF_THREADS) {
            const int k = q / NX, i = q % NX;
            o[probe::OUT_WT + q] = sm[bo::WT + k * QS + i];
        }
        if (lane == 0) { o[0] = dk; o[1] = flag[1]; o[2] = flag[3]; o[3] = fok ? 1.0 : 0.0; }
        BDF_SYNC();
    }
}

// A^{-1} by bdf_gauss_jordan, one warp per NX x NX matrix (row-major in a); out: ok | A^{-1} row-major (zeros when not ok)
CPDP_GLOBAL void __launch_bounds__(BDF_THREADS) k_bdf_probe_gj(const double* __restrict__ a, double* __restrict__ out) {
    BDF_SM();
    const int lane = threadIdx.x;
    const double* A = a + (size_t)blockIdx.x * NX * NX;
    double* o = out + (size_t)blockIdx.x * (1 + NX * NX);
    CPDP_LOOP for (int q = lane; q < BDF_SMEM_DOUBLES; q += BDF_THREADS) sm[q] = 0.0;
    BDF_SYNC();
    if (lane < NX) { BDF_UNROLL for (int i = 0; i < NX; ++i) sm[bo::XA + i * NCS + lane] = A[i * NX + lane]; }
    BDF_SYNC();
    const bool ok = bdf_gauss_jordan(sm + bo::WT);
    BDF_SYNC();
    CPDP_LOOP for (int q = lane; q < NX * NX; q += BDF_THREADS) {
        const int i = q / NX, k = q % NX;
        o[1 + q] = ok ? sm[bo::WT + k * QS + i] : 0.0;
    }
    if (lane == 0) o[0] = ok ? 1.0 : 0.0;
}
}  // namespace CPDP_NS
