// Library-level entry points: version, last error, device check.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>

static thread_local char g_last_error[512] = "";

void spnet_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
}

int spnet_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        spnet_set_error("%s: %s", what, cudaGetErrorString(e));
        return SPNET_ERR_CUDA;
    }
    return SPNET_OK;
}

extern "C" {

int spnet_version(void) { return 100; }

const char* spnet_last_error(void) { return g_last_error; }

// Returns 0 when the current device is compute capability 10.x (the only
// architecture this library carries code for), SPNET_ERR_ARCH otherwise.
int spnet_check_device(void) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        spnet_set_error("cudaGetDevice: %s", cudaGetErrorString(e));
        return SPNET_ERR_CUDA;
    }
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) {
        spnet_set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e));
        return SPNET_ERR_CUDA;
    }
    if (p.major != 10) {
        spnet_set_error("spnet_b200 is built for sm_100a only; device is sm_%d%d", p.major, p.minor);
        return SPNET_ERR_ARCH;
    }
    return SPNET_OK;
}

}  // extern "C"
