// libsng.so: error plumbing and device queries shared by every entry point of include/sng.h.
#include "sng_common.cuh"
#include <stdarg.h>

namespace sng {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();  // clear the sticky launch error so the next call reports its own
        set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
        return SNG_ERR_CUDA;
    }
    return SNG_OK;
}

// Without a device every launch fails anyway; the host-side plans (sng_simknn_plan, the workspace sizes) then report what
// they would be on a B200.
int sm_count() {
    constexpr int kNoDevice = 148;
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return kNoDevice; }
    if (cached[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { cudaGetLastError(); return kNoDevice; }
        cached[dev] = v;
    }
    return cached[dev];
}

}  // namespace sng

extern "C" int sng_version(void) { return 100; }

extern "C" const char* sng_last_error(void) { return sng::g_err; }

extern "C" int sng_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        sng::set_error("sng_device_info: no CUDA device (%s)", cudaGetErrorString(e));
        return SNG_ERR_CUDA;
    }
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        sng::set_error("sng_device_info: %s", cudaGetErrorString(e));
        return SNG_ERR_CUDA;
    }
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return SNG_OK;
}
