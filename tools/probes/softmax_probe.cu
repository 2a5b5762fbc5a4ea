// Where does the exp pass of the attention softmax spend its time?  One CTA, S tiles pre-filled in TMEM, variants of the
// pass (read fp32 S from TMEM -> exp2 -> row sum -> bf16 P back into TMEM) timed with clock64 over `tiles` tiles at once.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../rajni_vit_b200/csrc softmax_probe.cu -o softmax_probe
#include <cstdio>
#include "common.cuh"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return 0; } }
using namespace rajni;

__device__ __forceinline__ float ex2a(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// mode 0: full pass, 32x32b.x32 loads, next chunk prefetched (what attention_tc does)      [4 warps per tile]
// mode 1: same, but no exp (TMEM traffic only: load, pack raw, store)
// mode 2: same, but no TMEM (exp / sum / pack on register data only)
// mode 3: full pass, 16-lane shapes, 16x256b.x4 loads                                      [8 warps per tile]
// mode 4: full pass, 16-lane shapes, 16x256b.x8 loads                                      [8 warps per tile]
// mode 5: mode 0 with four partial sums and the FFMAs of the whole chunk issued before its MUFUs
template <int mode>
__global__ void __launch_bounds__(512) softmax_kernel(int ncols, int tiles, int reps, long long* out, float* sink) {
    __shared__ uint32_t slot;
    __shared__ long long t_end[16];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&slot, 512);
    tc_fence_before(); __syncthreads(); tc_fence_after();
    const uint32_t tm = slot;
    const int wpt = (mode == 3 || mode == 4) ? 8 : 4;           // warps per tile
    const int t = warp / wpt, wi = warp % wpt;
    const bool active = t < tiles;
    // fill S: value depends on (row, col) a little so that nothing is constant-folded
    if (active && wi < 4) {
        for (int c0 = 0; c0 < 256; c0 += 32) {
            uint32_t v[32];
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(-0.01f * (float)((c0 + j + lane) & 63));
            tmem_st32(tm + t * 256 + ((uint32_t)((warp & 3) * 32) << 16) + c0, v);
        }
        tmem_st_wait();
    }
    tc_fence_before(); __syncthreads(); tc_fence_after();
    const float sl2 = 0.18f, mb = 0.05f;
    float sum = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    long long t0 = clock64();
    if (active) {
        for (int r = 0; r < reps; ++r) {
            if (mode <= 2 || mode == 5) {
                const uint32_t trow = tm + t * 256 + ((uint32_t)((warp & 3) * 32) << 16);
                uint32_t va[32], vb[32];
                if (mode != 2) tmem_ld32(trow, va);
                else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) { va[j] = __float_as_uint(-0.01f * (j + lane + r)); vb[j] = va[j] ^ 0x100u; }
                }
                auto step = [&](uint32_t (&cur)[32], uint32_t (&nxt)[32], int c0) {
                    if (mode != 2) {
                        tmem_ld_wait();
                        if (c0 + 32 < ncols) tmem_ld32(trow + c0 + 32, nxt);
                    }
                    uint32_t pk[16];
                    if (mode == 1) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) pk[j >> 1] = cur[j] ^ cur[j + 1];
                    } else if (mode == 5) {
                        float x[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) x[j] = fmaf(__uint_as_float(cur[j]), sl2, -mb);
#pragma unroll
                        for (int j = 0; j < 32; ++j) x[j] = ex2a(x[j]);
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            sum += x[j] + x[j + 1]; s1 += x[j + 2] + x[j + 3]; s2 += x[j + 4] + x[j + 5]; s3 += x[j + 6] + x[j + 7];
                        }
#pragma unroll
                        for (int j = 0; j < 32; j += 2) pk[j >> 1] = float2_to_bf16x2(x[j], x[j + 1]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float e0 = ex2a(fmaf(__uint_as_float(cur[j]), sl2, -mb));
                            const float e1 = ex2a(fmaf(__uint_as_float(cur[j + 1]), sl2, -mb));
                            sum += e0 + e1;
                            pk[j >> 1] = float2_to_bf16x2(e0, e1);
                        }
                    }
                    if (mode != 2) tmem_st16(trow + (c0 >> 1), pk);
                    else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) s1 += __uint_as_float(pk[j]);
                    }
                };
                for (int c0 = 0; c0 < ncols; c0 += 64) {
                    step(va, vb, c0);
                    if (c0 + 32 < ncols) step(vb, va, c0 + 32);
                }
                if (mode != 2) tmem_st_wait();
            } else {
                const int rbase = (wi & 3) * 32 + ((wi >> 2) & 1) * 16;
                const uint32_t twin = tm + t * 256 + ((uint32_t)rbase << 16);
                auto grp = [&](uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t& p0, uint32_t& p1) {
                    const float e00 = ex2a(fmaf(__uint_as_float(a), sl2, -mb)), e01 = ex2a(fmaf(__uint_as_float(b), sl2, -mb));
                    const float e10 = ex2a(fmaf(__uint_as_float(c), sl2, -mb)), e11 = ex2a(fmaf(__uint_as_float(d), sl2, -mb));
                    sum += e00 + e01; s1 += e10 + e11;
                    p0 = float2_to_bf16x2(e00, e01); p1 = float2_to_bf16x2(e10, e11);
                };
                if (mode == 3) {
                    uint32_t xa[16], xb[16];
                    tmem_ld16x256_x4(twin, xa);
                    auto step4 = [&](uint32_t (&cur)[16], uint32_t (&nxt)[16], int c0) {
                        tmem_ld_wait();
                        if (c0 + 32 < ncols) tmem_ld16x256_x4(twin + c0 + 32, nxt);
                        uint32_t pk[8];
#pragma unroll
                        for (int g = 0; g < 4; ++g) grp(cur[4 * g], cur[4 * g + 1], cur[4 * g + 2], cur[4 * g + 3], pk[2 * g], pk[2 * g + 1]);
                        tmem_st16x128_x4(twin + (c0 >> 1), pk);
                    };
                    for (int c0 = 0; c0 < ncols; c0 += 64) {
                        step4(xa, xb, c0);
                        if (c0 + 32 < ncols) step4(xb, xa, c0 + 32);
                    }
                } else {
                    uint32_t xa[32], xb[32];
                    tmem_ld16x256_x8(twin, xa);
                    auto step8 = [&](uint32_t (&cur)[32], uint32_t (&nxt)[32], int c0) {
                        tmem_ld_wait();
                        if (c0 + 64 < ncols) tmem_ld16x256_x8(twin + c0 + 64, nxt);
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            uint32_t pk[8];
#pragma unroll
                            for (int g = 0; g < 4; ++g)
                                grp(cur[16 * hh + 4 * g], cur[16 * hh + 4 * g + 1], cur[16 * hh + 4 * g + 2], cur[16 * hh + 4 * g + 3], pk[2 * g], pk[2 * g + 1]);
                            tmem_st16x128_x4(twin + ((c0 + 32 * hh) >> 1), pk);
                        }
                    };
                    for (int c0 = 0; c0 < ncols; c0 += 128) {
                        step8(xa, xb, c0);
                        if (c0 + 64 < ncols) step8(xb, xa, c0 + 64);
                    }
                }
                tmem_st_wait();
            }
        }
    }
    long long t1 = clock64();
    if (lane == 0) t_end[warp] = active ? t1 - t0 : 0;
    tc_fence_before(); __syncthreads();
    if (tid == 0) { long long m = 0; for (int w = 0; w < 16; ++w) m = t_end[w] > m ? t_end[w] : m; out[0] = m; }
    sink[tid] = sum + s1 + s2 + s3;
    if (warp == 0) { tc_fence_after(); tmem_dealloc(tm, 512); }
}

int main() {
    long long* out; float* sink;
    cudaMallocManaged(&out, 64); cudaMallocManaged(&sink, 4096);
    const char* names[] = {"x32 loads, 4 warps/tile (attention_tc)", "  same, TMEM traffic only", "  same, exp/sum/pack only (no TMEM)",
                           "16-lane x4 loads, 8 warps/tile", "16-lane x8 loads, 8 warps/tile", "x32 loads, FFMAs before MUFUs, 4 sums"};
    const int reps = 64, ncols = 208;
    for (int tiles : {1, 2})
        for (int mode : {0, 5, 1, 2, 3, 4}) {
            const int wpt = (mode == 3 || mode == 4) ? 8 : 4;
            for (int it = 0; it < 2; ++it) {
                const int th = tiles * wpt * 32;
                switch (mode) {
                    case 0: softmax_kernel<0><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                    case 1: softmax_kernel<1><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                    case 2: softmax_kernel<2><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                    case 3: softmax_kernel<3><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                    case 4: softmax_kernel<4><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                    default: softmax_kernel<5><<<1, th>>>(ncols, tiles, reps, out, sink); break;
                }
                cudaError_t e = cudaDeviceSynchronize();
                if (e != cudaSuccess) { printf("mode %d: %s\n", mode, cudaGetErrorString(e)); return 1; }
            }
            printf("%d tile(s) at once, %-42s: %7.0f cycles per 128x%d tile pass (MUFU floor %d)\n", tiles, names[mode],
                   (double)out[0] / reps, ncols, 128 * ncols / 16 * tiles);
        }
    return 0;
}
