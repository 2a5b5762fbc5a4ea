// The C ABI's version, error string, launch counter and device check.
#include "common.cuh"

extern "C" int rajni_abi_version(void) { return RAJNI_ABI_VERSION; }

extern "C" const char* rajni_last_error(void) { return rajni::error_text(); }

extern "C" uint64_t rajni_launch_count(void) { return rajni::launches(); }

extern "C" int rajni_device_check(void) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        rajni::set_error("rajni_device_check: no CUDA device: %s", cudaGetErrorString(e));
        return RAJNI_ECUDA;
    }
    int major = 0, minor = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (major != 10) {
        rajni::set_error("rajni_device_check: device %d is sm_%d%d; this library is sm_100a only", dev, major, minor);
        return RAJNI_EARCH;
    }
    return RAJNI_OK;
}
