// Error reporting + version/device queries of the C ABI (include/b200pose.h).
#include "common.cuh"
#include <string.h>

namespace b200pose {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace b200pose

extern "C" __attribute__((visibility("default"))) const char* b200pose_last_error(void) { return b200pose::g_err; }
extern "C" __attribute__((visibility("default"))) int b200pose_version(void) { return 200; }
extern "C" __attribute__((visibility("default"))) int b200pose_device_cc(void) {
    int dev = 0, major = 0, minor = 0;
    B2_CHECK_CUDA(cudaGetDevice(&dev));
    B2_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    B2_CHECK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    return major * 10 + minor;
}
