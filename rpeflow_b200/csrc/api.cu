// api.cu — library identification and the thread-local error channel of the C-ABI (include/b200flow.h).
#include <stdarg.h>
#include <stdio.h>

#include "common.cuh"

#define B200_STR_(x) #x
#define B200_STR(x) B200_STR_(x)

namespace b200 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error in %s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return B200_ECUDA;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached_dev = dev;
        cached = n;
    }
    return cached;
}

}  // namespace b200

extern "C" {

int b200_abi_version(void) { return 8; }

const char* b200_build_info(void) {
    return "libb200flow sm_100a; nvcc " B200_STR(__CUDACC_VER_MAJOR__) "." B200_STR(__CUDACC_VER_MINOR__)
           "; built " __DATE__;
}

const char* b200_last_error(void) { return b200::g_err; }

}  // extern "C"
