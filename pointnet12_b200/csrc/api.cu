// api.cu -- library identification, error reporting and the device check of the C ABI.
#include <stdarg.h>

#include "common.cuh"

namespace pn {

static thread_local char g_err[512] = "no error";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace pn

PN_EXPORT int pn_version(void) { return 402; /* 0.4.2: function-level gradients: pn_square_distance_bwd_f32, pn_chamfer_argmin_f32, pn_chamfer_bwd_f32; 0.4.1: sampling on clusters of three and 48 points per thread; 3-NN block workspace in pairs (opaque, size changed); 0.4.0: per-call pn_launch_opts replace the process-wide setters; dynamic tile scheduling */ }

PN_EXPORT const char* pn_last_error_string(void) { return pn::g_err; }

PN_EXPORT int pn_device_check(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pn::set_error("pn_device_check: %s", cudaGetErrorString(e));
        return (int)e;
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    PN_REQUIRE(prop.major == 10, PN_ERR_DEVICE, "pn_device_check: kernels are built for sm_100a only; device is sm_%d%d",
               prop.major, prop.minor);
    return PN_OK;
}
