// Error plumbing and device queries for libdet_b200.so.
#include "common.cuh"
#include <stdarg.h>
#include <stdio.h>

namespace det {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error in %s: %s (%d)", what, cudaGetErrorString(e), (int)e);
    return DET_ERR_CUDA;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

}  // namespace det

extern "C" {

int det_abi_version(void) { return DET_ABI_VERSION; }

const char* det_last_error(void) { return det::g_err; }

int det_sm_count(void) {
    int dev = 0, n = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return det::cuda_fail(e, "cudaGetDevice");
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return det::cuda_fail(e, "cudaDeviceGetAttribute");
    return n;
}

}  // extern "C"
