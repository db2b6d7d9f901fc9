// Shipped library translation unit: one shared object per model, built with
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC -DCPDP_MODEL_HEADER=...
// Exposes the C ABI of include/cpdp.h (plain pointers and sizes, no torch types).
#include <cuda_runtime.h>
#include <cstdio>

#include "cpdp_port.h"
#include CPDP_MODEL_HEADER
#include "cpdp_kernels.cuh"
#include "cpdp_aux.cuh"
#include "cpdp_bdf.cuh"
#include "cpdp_fwd.cuh"
#include "cpdp_disc.cuh"
#include "cpdp_optim.cuh"

// The only host-side state of the library: the first launch error of the call in progress.  Thread-local, cleared by every
// entry point before it returns, so host threads driving different streams (or devices) never see each other's errors.
static thread_local int g_last_error = 0;

static int cpdp_num_sms() {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    return sms;
}

static int cpdp_take_error() {
    cudaError_t e = cudaGetLastError();
    int r = g_last_error ? g_last_error : (int)e;
    g_last_error = 0;
    return r;
}

template <class K>
static void cpdp_prepare_smem(K kernel, size_t bytes) {
    // always opt in: static + dynamic shared memory may exceed 48 KB even when the dynamic part alone does not
    if (bytes > 32 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess && !g_last_error) g_last_error = (int)e;
    }
}

#define CPDP_LAUNCH(kernel, grid, block, smem, stream, ...)                         \
    do {                                                                            \
        CPDP_NS::kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);           \
        cudaError_t e__ = cudaPeekAtLastError();                                    \
        if (e__ != cudaSuccess && !g_last_error) g_last_error = (int)e__;           \
    } while (0)
#define CPDP_READ_INT(dst, src, stream)                                             \
    do {                                                                            \
        cudaError_t e__ = cudaMemcpyAsync(&(dst), (src), sizeof(int), cudaMemcpyDeviceToHost, (stream)); \
        if (e__ == cudaSuccess) e__ = cudaStreamSynchronize(stream);                \
        if (e__ != cudaSuccess) { if (!g_last_error) g_last_error = (int)e__; (dst) = 0; } \
    } while (0)
#define CPDP_NUM_SMS() cpdp_num_sms()
#define CPDP_PREPARE_SMEM(kernel, bytes) cpdp_prepare_smem(CPDP_NS::kernel, bytes)
#define CPDP_LAST_ERROR() cpdp_take_error()
#include "cpdp_api.inl"

// Digest of (generated model header, kernel sources, compiler flags) this library was built from; lfsd_b200._capi looks
// for the marker in the file to decide whether a prebuilt library is up to date.
#ifndef CPDP_BUILD_DIGEST
#define CPDP_BUILD_DIGEST "CPDP_BUILD_DIGEST=unknown"
#endif
extern "C" CPDP_API const char* cpdp_build_digest(void) { return CPDP_BUILD_DIGEST; }

extern "C" CPDP_API const char* cpdp_error_string(int code) {
    if (code < 0) {
        switch (code) {
            case -1: return "null pointer or non-positive size";
            case -2: return "theta_stride must be 0 (shared) or r";
            case -3: return "workspace too small (see cpdp_workspace_bytes)";
            case -4: return "bad waypoint arguments";
            case -5: return "taus_stride must be 0 (shared) or W";
            case -6: return "observed state index out of range";
            case -7: return "unknown integrator mode";
            case -8: return "model has per-problem constants but pdata is null";
            case -9: return "phases must be 1, 2 or 3";
            case -10: return "max_iter must be in [0, 255]";
            case -11: return "the model has no finite bound";
            case -12: return "shift must be 0 or 1";
            case -13: return "mu_init must be > 0 on a bounded model";
            case -14: return "the model has no per-problem constants (pdata)";
            case -15: return "the library was built without the pdata derivatives (or n + m + r + q > 32)";
            default: return "invalid argument";
        }
    }
    return cudaGetErrorString((cudaError_t)code);
}
