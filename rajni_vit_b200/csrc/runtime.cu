// Error string and launch counter shared by librajni_b200.so and librajni_jpeg.so (each library links its own copy).
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace rajni {

static thread_local char g_error[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}

const char* error_text() { return g_error; }

uint64_t launches() { return g_launches.load(std::memory_order_relaxed); }

void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
        return RAJNI_ECUDA;
    }
    return RAJNI_OK;
}

}  // namespace rajni
