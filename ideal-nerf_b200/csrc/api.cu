// Library-level entry points: version, error string, device check.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace inerf {
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace inerf

extern "C" int inerf_version(void) { return INERF_VERSION; }

extern "C" const char* inerf_last_error(void) { return inerf::g_err; }

extern "C" size_t inerf_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(InerfNetDims);
        case 1: return sizeof(InerfRenderNet);
        case 2: return sizeof(InerfRenderArgs);
        case 4: return sizeof(InerfPixelSampleArgs);
        default: return 0;
    }
}

extern "C" int inerf_device_check(void) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        inerf::set_error("cudaGetDevice: %s", cudaGetErrorString(e));
        return (int)e;
    }
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (major != 10) {
        inerf::set_error("device %d has compute capability %d.x; this library is built for sm_100a only", dev, major);
        return INERF_E_DEVICE;
    }
    return INERF_OK;
}
