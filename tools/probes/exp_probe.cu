// What bounds the exp pass of the attention kernels?  8 warps (2 per scheduler), registers only: per 16 "scores" a warp runs
//   variant 0: 16 MUFU.EX2                          variant 1: + 16 FFMA (scale, subtract max)
//   variant 2: + 16 FADD (row sum, two chains)       variant 3: + 8 F2FP.BF16.PACK_AB (cvt.rn.bf16x2.f32)
//   variant 4: as 2, packing by integer ops instead (round-half-up: IADD 0x8000 x2, PRMT)     variant 5: as 2, PRMT truncation only
//   variant 6: as 3 with packed FFMA2 / FADD2 (half the issue slots for the fp32 math)
//   variant 7: F2FP only (8 per 16 scores)           variant 8: FFMA+FADD only (no MUFU, no pack)
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../rajni_vit_b200/csrc exp_probe.cu -o exp_probe
#include <cstdio>
#include "common.cuh"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return 0; } int current_device() { return 0; } }
using namespace rajni;
__device__ __forceinline__ float ex2f(float x) { float y; asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { uint32_t d; asm volatile("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel)); return d; }
__device__ __forceinline__ uint32_t cvt2(float lo, float hi) { uint32_t d; asm volatile("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo)); return d; }

template <int V>
__global__ void __launch_bounds__(512, 1) exp_kernel(int reps, long long* out, float* sink, const float* src) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float s[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) s[j] = src[(threadIdx.x * 16 + j) & 1023];
    const float sl2 = src[5], mb = src[7];
    float sum0 = 0.f, sum1 = 0.f;
    uint64_t sum2 = 0;
    uint32_t acc = 0;
    __syncthreads();
    const long long t0 = clock64();
    for (int r = 0; r < reps; ++r) {
        float e[16];
        if (V == 6) {
            const uint64_t sl22 = f2pack(sl2, sl2), mb2 = f2pack(-mb, -mb);
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                float x0, x1;
                f2unpack(fma2(f2pack(s[j], s[j + 1]), sl22, mb2), x0, x1);
                e[j] = ex2f(x0); e[j + 1] = ex2f(x1);
                sum2 = add2(sum2, f2pack(e[j], e[j + 1]));
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float x = s[j];
                if (V >= 1 && V != 7) x = fmaf(x, sl2, -mb);
                e[j] = (V == 7 || V == 8) ? x : ex2f(x);
                if (V >= 2 && V != 7) { if (j & 1) sum1 += e[j]; else sum0 += e[j]; }
            }
        }
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
            uint32_t pk;
            if (V == 3 || V == 6 || V == 7) pk = cvt2(e[j], e[j + 1]);
            else if (V == 4) pk = prmt(__float_as_uint(e[j]) + 0x8000u, __float_as_uint(e[j + 1]) + 0x8000u, 0x7632);
            else if (V == 5) pk = prmt(__float_as_uint(e[j]), __float_as_uint(e[j + 1]), 0x7632);
            else pk = __float_as_uint(e[j]) ^ __float_as_uint(e[j + 1]);
            acc ^= pk;
            s[j] = __uint_as_float((__float_as_uint(s[j]) & 0xfffffffeu) | (pk & 1u));     // keep the chain data-dependent, values stable
        }
    }
    const long long t1 = clock64();
    if (lane == 0) out[warp] = t1 - t0;
    float a, b; f2unpack(sum2, a, b);
    sink[threadIdx.x] = sum0 + sum1 + a + b + __uint_as_float(acc);
}

template <int V> void run(const char* name, long long* out, float* sink, float* src) {
    for (int warps : {4, 8, 12}) {
        const int reps = 2048;
        for (int it = 0; it < 2; ++it) { exp_kernel<V><<<1, warps * 32>>>(reps, out, sink, src); cudaDeviceSynchronize(); }
        long long mx = 0;
        for (int w = 0; w < warps; ++w) mx = out[w] > mx ? out[w] : mx;
        printf("%-58s %2d warps: %6.2f cycles per 16 scores per warp, %5.2f scores/clk/SM\n", name, warps, (double)mx / reps, 16.0 * 32 * warps * reps / mx);
    }
}

int main() {
    long long* out; float* sink; float* src;
    cudaMallocManaged(&out, 4096); cudaMallocManaged(&sink, 1 << 16); cudaMallocManaged(&src, 4096);
    for (int i = 0; i < 1024; ++i) src[i] = -((i * 37) % 200) / 40.f;
    src[5] = 0.18f; src[7] = 0.5f;
    run<0>("0: MUFU.EX2 only", out, sink, src);
    run<1>("1: FFMA + MUFU", out, sink, src);
    run<2>("2: FFMA + MUFU + FADD", out, sink, src);
    run<3>("3: FFMA + MUFU + FADD + F2FP.BF16 pack", out, sink, src);
    run<4>("4: FFMA + MUFU + FADD + integer round-half-up pack", out, sink, src);
    run<5>("5: FFMA + MUFU + FADD + PRMT truncation pack", out, sink, src);
    run<6>("6: FFMA2 + MUFU + FADD2 + F2FP.BF16 pack", out, sink, src);
    run<7>("7: F2FP.BF16 pack only (8 per 16 scores)", out, sink, src);
    run<8>("8: FFMA + FADD only", out, sink, src);
    return 0;
}
