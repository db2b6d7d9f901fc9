// Device build of tests/bdf_probe/bdf_probe.cuh for sm_100a (TEST INFRASTRUCTURE ONLY): extern "C" launchers on device
// pointers, one warp per case with BDF_SMEM_BYTES of dynamic shared memory, opted in as cpdp_lib.cu's cpdp_prepare_smem does.
#include <cuda_runtime.h>

#include "cpdp_port.h"
#include CPDP_MODEL_HEADER
#include "cpdp_bdf.cuh"
#include "bdf_probe.cuh"
#include "bdf_probe_api.inl"

template <class K>
static int prepare_smem(K kernel) {
    if (CPDP_NS::BDF_SMEM_BYTES > 32 * 1024)
        return (int)cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CPDP_NS::BDF_SMEM_BYTES);
    return 0;
}

extern "C" CPDP_API int bdf_probe_run(const double* in, double* out, int cases, int S, void* stream) {
    if (int e = prepare_smem(CPDP_NS::k_bdf_probe)) return e;
    CPDP_NS::k_bdf_probe<<<cases, CPDP_NS::BDF_THREADS, CPDP_NS::BDF_SMEM_BYTES, (cudaStream_t)stream>>>(in, out, S);
    return (int)cudaPeekAtLastError();
}
extern "C" CPDP_API int bdf_probe_gj(const double* a, double* out, int cases, void* stream) {
    if (int e = prepare_smem(CPDP_NS::k_bdf_probe_gj)) return e;
    CPDP_NS::k_bdf_probe_gj<<<cases, CPDP_NS::BDF_THREADS, CPDP_NS::BDF_SMEM_BYTES, (cudaStream_t)stream>>>(a, out);
    return (int)cudaPeekAtLastError();
}
