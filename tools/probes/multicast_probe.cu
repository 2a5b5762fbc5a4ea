// How do TMA multicast loads signal mbarriers in a cluster of 4 CTAs (two cta_group::2 pairs)?  Groundwork for sharing the B
// operand between two CTA pairs in the GEMM (DESIGN.md, "TMA multicast across two CTA pairs").
//   test 0: plain  .multicast::cluster  from CTA s to mask m, mbarrier = own CTA-relative address
//   test 1: .cta_group::2 .multicast::cluster from CTA s to mask m, mbarrier = address of the SAME barrier in the pair leader (rank & ~1)
// Every CTA arms bar with expect_tx(8 KB) and polls it for a bounded time; the host prints which CTAs saw their barrier complete
// and what value landed at the start of their buffer (source row r holds the value r, the box starts at row 64*s).
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../rajni_vit_b200/csrc multicast_probe.cu -o multicast_probe -lcuda
#include <cstdio>
#include <cuda.h>
#include "common.cuh"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return 0; } int current_device() { return 0; } }
using namespace rajni;

struct Result { int done[4]; float first[4]; };

template <int TEST>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(64) probe_kernel(const __grid_constant__ CUtensorMap tmap, int src_cta, int mask, Result* res) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* buf = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bar = reinterpret_cast<uint64_t*>(buf + 8192);
    const uint32_t rank = cluster_ctarank();
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2048; ++i) reinterpret_cast<float*>(buf)[i] = -1.f;
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    cluster_sync_all();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, 8192);                       // every CTA arms its own barrier (arrive + expect)
    }
    cluster_sync_all();
    if (threadIdx.x == 0 && (int)rank == src_cta) {
        const uint16_t m16 = (uint16_t)mask;
        if (TEST == 0) {
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                :: "r"(smem_u32(buf)), "l"(&tmap), "r"(smem_u32(bar)), "r"(0), "r"(64 * src_cta), "h"(m16) : "memory");
        } else {
            const uint32_t lead_bar = mapa_u32(smem_u32(bar), rank & ~1u);
            asm volatile(
                "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                :: "r"(smem_u32(buf)), "l"(&tmap), "r"(lead_bar), "r"(0), "r"(64 * src_cta), "h"(m16) : "memory");
        }
    }
    if (threadIdx.x == 0) {
        int done = 0;
        for (int i = 0; i < 200000 && !done; ++i) done = mbar_test(bar, 0);
        res->done[rank] = done;
        res->first[rank] = __bfloat162float(*reinterpret_cast<__nv_bfloat16*>(buf));
    }
    __syncthreads();
    cluster_sync_all();
}

int main() {
    const int rows = 256, cols = 64;
    __nv_bfloat16* h = new __nv_bfloat16[rows * cols];
    for (int r = 0; r < rows; ++r) for (int c = 0; c < cols; ++c) h[r * cols + c] = __float2bfloat16((float)r);
    __nv_bfloat16* d; cudaMalloc(&d, rows * cols * 2); cudaMemcpy(d, h, rows * cols * 2, cudaMemcpyHostToDevice);
    CUtensorMap map;
    void* fn = nullptr; cudaDriverEntryPointQueryResult q;
    cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    auto enc = reinterpret_cast<CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                             const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill)>(fn);
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows}; cuuint64_t strides[1] = {cols * 2}; cuuint32_t box[2] = {64, 64}; cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { printf("encode failed %d\n", (int)r); return 1; }
    Result* res; cudaMallocManaged(&res, sizeof(Result));
    const int smem = 8192 + 64 + 1024;
    struct Case { int test, src, mask; } cases[] = {{0, 0, 0x5}, {0, 1, 0xA}, {0, 2, 0x5}, {0, 0, 0xF}, {1, 0, 0x5}, {1, 1, 0xA}, {1, 2, 0x5}, {1, 3, 0xA}, {1, 1, 0x2}};
    for (auto c : cases) {
        for (int i = 0; i < 4; ++i) { res->done[i] = -1; res->first[i] = -2.f; }
        if (c.test == 0) probe_kernel<0><<<4, 64, smem>>>(map, c.src, c.mask, res);
        else probe_kernel<1><<<4, 64, smem>>>(map, c.src, c.mask, res);
        cudaError_t e = cudaDeviceSynchronize();
        printf("%s multicast from CTA %d mask 0x%x: %s | barrier completed in CTA", c.test ? "cta_group::2" : "plain       ", c.src, c.mask,
               e == cudaSuccess ? "ok" : cudaGetErrorString(e));
        for (int i = 0; i < 4; ++i) if (res->done[i] == 1) printf(" %d", i);
        printf(" | first value per CTA:");
        for (int i = 0; i < 4; ++i) printf(" %g", res->first[i]);
        printf("\n");
        if (e != cudaSuccess) return 1;
    }
    return 0;
}
