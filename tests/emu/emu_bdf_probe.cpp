// Host emulation of tests/bdf_probe/bdf_probe.cuh (TEST INFRASTRUCTURE ONLY): the probe kernels over the device functions of
// cpdp_bdf.cuh, one std::thread per lane, std::barrier for the warp barriers, as in emu_lib.cpp.  Only the BDF sweep's headers
// are compiled, so that one build per state dimension stays cheap.
#include <barrier>
#include <thread>
#include <vector>

#include CPDP_MODEL_HEADER_PORT
#include CPDP_MODEL_HEADER
#include "cpdp_bdf.cuh"
#include "bdf_probe.cuh"

thread_local cpdp_emu_dim3 threadIdx;
cpdp_emu_dim3 blockIdx, blockDim, gridDim;
double* cpdp_emu_dyn_smem = nullptr;
static std::barrier<>* g_bar = nullptr;
void cpdp_emu_syncthreads() { g_bar->arrive_and_wait(); }

template <class F, class... Args>
static void emu_launch(F kernel, int grid, Args... args) {
    std::vector<double> dyn(CPDP_NS::BDF_SMEM_DOUBLES + 16);
    cpdp_emu_dyn_smem = dyn.data();
    gridDim = {grid, 1, 1};
    blockDim = {CPDP_NS::BDF_THREADS, 1, 1};
    for (int b = 0; b < grid; ++b) {
        blockIdx = {b, 0, 0};
        std::barrier<> bar(CPDP_NS::BDF_THREADS);
        g_bar = &bar;
        std::vector<std::thread> th;
        for (int t = 0; t < CPDP_NS::BDF_THREADS; ++t)
            th.emplace_back([=] {
                threadIdx = {t, 0, 0};
                kernel(args...);
                g_bar->arrive_and_drop();
            });
        for (auto& x : th) x.join();
    }
}

#include "bdf_probe_api.inl"
extern "C" CPDP_API int bdf_probe_run(const double* in, double* out, int cases, int S, void*) {
    emu_launch(CPDP_NS::k_bdf_probe, cases, in, out, S);
    return 0;
}
extern "C" CPDP_API int bdf_probe_gj(const double* a, double* out, int cases, void*) {
    emu_launch(CPDP_NS::k_bdf_probe_gj, cases, a, out);
    return 0;
}
