// Issue/complete rate of tcgen05.mma.cta_group::2 (M=256 across a CTA pair, N=256/128, K=16, SS operands, bf16):
// the ceiling of the GEMM main loop.   build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../rajni_vit_b200/csrc mma2_probe.cu -o mma2_probe
#include <cstdio>
#include "common.cuh"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return 0; } }
using namespace rajni;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128) mma2_kernel(int N, int reps, int nacc, long long* out) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    if (warp == 0) { tmem_alloc_cg2(&slot, 512); if (lane == 0) { mbar_init(&bar, 1); mbar_fence_init(); } }
    for (int i = threadIdx.x; i < 96 * 1024 / 4; i += 128) reinterpret_cast<uint32_t*>(smem_raw)[i] = 0x3c003c00u;
    fence_async_smem();
    tc_fence_before(); cluster_sync_all(); tc_fence_after();
    const uint32_t tm = slot;
    if (threadIdx.x == 0 && rank == 0) {
        const uint32_t idesc = umma_idesc_bf16(256, N, 0, 0);
        const uint32_t sa = base, sb = base + 32768;
        uint64_t ad[4], bd[4];
        for (int k = 0; k < 4; ++k) { ad[k] = umma_desc_sw128(sa + k * 32, 16, 1024); bd[k] = umma_desc_sw128(sb + k * 32, 16, 1024); }
        long long t0 = clock64();
        for (int r = 0; r < reps; r += 4) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_cg2(tm + ((r / 4) % nacc) * N, ad[k], bd[k], idesc, r >= 4 * nacc);
        }
        long long t1 = clock64();
        umma_commit_cg2(&bar, 0x3);
        mbar_wait(&bar, 0);
        long long t2 = clock64();
        out[0] = t1 - t0;
        out[1] = t2 - t0;
    } else if (threadIdx.x == 0) {
        mbar_wait(&bar, 0);
    }
    tc_fence_before(); cluster_sync_all();
    if (warp == 0) { tc_fence_after(); tmem_dealloc_cg2(tm, 512); }
}

int main() {
    long long* out;
    cudaMallocManaged(&out, 64);
    cudaFuncSetAttribute(mma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    const int reps = 512;
    for (int N : {64, 128, 192, 256})
        for (int nacc : {1, 2}) {
            if (N * nacc > 512) continue;
            for (int it = 0; it < 2; ++it) {
                mma2_kernel<<<2, 128, 100 * 1024>>>(N, reps, nacc, out);
                cudaError_t e = cudaDeviceSynchronize();
                if (e != cudaSuccess) { printf("N=%d: %s\n", N, cudaGetErrorString(e)); return 1; }
            }
            printf("cta_group::2 SS M=256 N=%3d K=16, %d accumulator(s): issue %.1f cyc/mma, complete %.1f cyc/mma (ideal %d) -> %.0f%% of the 8192 flop/clk/SM peak\n",
                   N, nacc, (double)out[0] / reps, (double)out[1] / reps, N / 2, 100.0 * (N / 2) / ((double)out[1] / reps));
        }
    return 0;
}
