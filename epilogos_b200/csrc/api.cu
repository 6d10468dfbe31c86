// Library-level plumbing of the C ABI: error strings, device checks, driver entry points.
#include <stdarg.h>

#include "common.cuh"

namespace epi {

static thread_local char g_error[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

static int g_sm_count = 0;

int check_device() {
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        set_error("no CUDA device available (%s); epilogos_b200 has no CPU fallback", cudaGetErrorString(e));
        cudaGetLastError();
        return 3;
    }
    int major = 0, minor = 0, sms = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (major != 10) {
        set_error("device %d has compute capability %d.%d; this library contains sm_100a code only", dev, major, minor);
        return 3;
    }
    g_sm_count = sms;
    return 0;
}

int sm_count() {
    if (g_sm_count == 0) check_device();
    return g_sm_count > 0 ? g_sm_count : 148;
}

unsigned grid_for(long long n, int per_block, int per_sm) {
    long long blocks = (n + per_block - 1) / per_block;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}

tensor_map_encode_fn get_tensor_map_encode() {
    static tensor_map_encode_fn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<tensor_map_encode_fn>(p);
    }
    return fn;
}

}  // namespace epi

extern "C" int epi_abi_version(void) { return EPI_ABI_VERSION; }

extern "C" const char* epi_last_error(void) { return epi::g_error; }

extern "C" int epi_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    if (epi::check_device()) {
        // still report what we can for diagnostics
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess) {
            cudaGetLastError();
            return 3;
        }
        if (cc_major) cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev);
        if (cc_minor) cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev);
        return 3;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    if (sm_count) cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (cc_major) cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev);
    if (cc_minor) cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev);
    return 0;
}
