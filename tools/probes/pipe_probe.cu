// Resource-contention probe for attention_pipe.cu: the three roles of the kernel (exp warps, max/epilogue helper warps, the MMA
// issuer) run their per-tile instruction streams on one SM WITHOUT any barrier between them, alone and together.  If a role
// slows down when another runs beside it, the two share a resource (TMEM port, issue slots, MUFU ...), whatever the
// dependency chain of the real kernel looks like.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../rajni_vit_b200/csrc pipe_probe.cu -o pipe_probe
#include <cstdio>
#include "common.cuh"
namespace rajni { void set_error(const char*, ...) {} void count_launch(int) {} int check_launch(const char*) { return 0; } int current_device() { return 0; } }
using namespace rajni;

__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fmax3f(float a, float b, float c) { float d; asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c)); return d; }

// roles bitmask: 1 = exp warps (0-7), 2 = helper warps (8-11), 4 = MMA issuer (warp 12)
// exp_mode: 0 = full (ld16 + ffma/ex2/add + pack + st8), 1 = no MUFU (ffma only), 2 = no TMEM (registers only), 3 = x32 chunks
// help_mode: 0 = max pass (208 cols, x32 loads, 2 in flight) + O read (64 cols), 1 = max pass only, 2 = O read only
// mma_mode: 0 = per tile 4 SS N=208 + 13 TS N=64, 1 = 13 TS only, 2 = 4 SS only
template <int exp_mode>
__global__ void __launch_bounds__(512, 1) pipe_kernel(int roles, int help_mode, int mma_mode, int tiles, long long* out, float* sink) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t slot;
    __shared__ float pm[512];
    __shared__ __align__(8) uint64_t pbar[2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 12) { tmem_alloc(&slot, 512); if (lane == 0) { mbar_init(&bar, 1); mbar_init(&pbar[0], 8); mbar_init(&pbar[1], 8); mbar_fence_init(); } }
    for (int i = threadIdx.x; i < 150 * 1024 / 4; i += 512) reinterpret_cast<uint32_t*>(smem_raw + (base - smem_u32(smem_raw)))[i] = 0x3c003c00u;
    fence_async_smem();
    tc_fence_before(); __syncthreads(); tc_fence_after();
    const uint32_t tm = slot;
    const uint32_t lane_base = tm + ((uint32_t)((warp & 3) * 32) << 16);
    float acc = 0.f;
    long long t0 = clock64(), t1 = t0;
    if (warp < 8) {
      if (exp_mode >= 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");      // the register split of attention_pipe.cu
      if (roles & 1) {
        const int half = warp >> 2;
        const int cb = half ? 112 : 0, ce = half ? 208 : 112;
        const float sl2 = 0.18f, mb = 3.f;
        long long ph[4] = {0, 0, 0, 0}, tl = clock64();
        for (int t = 0; t < tiles; ++t) {
            const uint32_t sb = lane_base + (t & 1) * 224;
            float sum0 = 0.f, sum1 = 0.f;
            if (exp_mode == 4 || exp_mode == 5) {
                // attention_pipe.cu's flow: the whole half row in one go, max from registers (+ pair barrier), exp, in-place pack, <= 3 stores
                const int ncol = ce - cb, n32 = ncol >> 5;
                const bool has16 = (ncol & 16) != 0;
                uint32_t s[112];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    if (i < n32) tmem_ld32(sb + cb + 32 * i, *reinterpret_cast<uint32_t(*)[32]>(&s[32 * i]));
                if (has16) tmem_ld16(sb + cb + n32 * 32, *reinterpret_cast<uint32_t(*)[16]>(&s[96]));
                tmem_ld_wait();
                const long long ta = clock64();
                float m4[4] = {-1e30f, -1e30f, -1e30f, -1e30f};
#pragma unroll
                for (int ch = 0; ch < 7; ++ch) {
                    const bool present = ch < 6 ? (ch >> 1) < n32 : has16;
                    if (!present) continue;
#pragma unroll
                    for (int j = 0; j < 16; j += 2)
                        m4[(j >> 1) & 3] = fmax3f(m4[(j >> 1) & 3], __uint_as_float(s[16 * ch + j]), __uint_as_float(s[16 * ch + j + 1]));
                }
                float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                if (exp_mode == 4) {
                    pm[(t & 1) * 256 + half * 128 + (warp & 3) * 32 + lane] = mx;
                    asm volatile("bar.sync %0, 64;" :: "r"(1 + (warp & 3)) : "memory");
                    mx = fmaxf(mx, pm[(t & 1) * 256 + (half ^ 1) * 128 + (warp & 3) * 32 + lane]);
                }
                const float mb2 = mx * sl2 * 0.f + mb;
                const long long tb = clock64();
#pragma unroll
                for (int ch = 0; ch < 7; ++ch) {
                    const bool present = ch < 6 ? (ch >> 1) < n32 : has16;
                    if (!present) continue;
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        const float e0 = ex2f(fmaf(__uint_as_float(s[16 * ch + j]), sl2, -mb2));
                        const float e1 = ex2f(fmaf(__uint_as_float(s[16 * ch + j + 1]), sl2, -mb2));
                        sum0 += e0; sum1 += e1;
                        s[8 * ch + (j >> 1)] = float2_to_bf16x2(e0, e1);
                    }
                }
                const long long tc = clock64();
                if (n32 >= 2) tmem_st32(sb + cb, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
                else if (n32 == 1) tmem_st16(sb + cb, *reinterpret_cast<uint32_t(*)[16]>(&s[0]));
                if (n32 == 3) tmem_st16(sb + cb + 32, *reinterpret_cast<uint32_t(*)[16]>(&s[32]));
                if (has16) tmem_st8(sb + cb + n32 * 16, *reinterpret_cast<uint32_t(*)[8]>(&s[48]));
                tmem_st_wait();
                if (help_mode == 7) { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(&pbar[t & 1]); }
                const long long td = clock64();
                ph[0] += ta - tl; ph[1] += tb - ta; ph[2] += tc - tb; ph[3] += td - tc;
                tl = td;
            } else if (exp_mode == 3) {
                uint32_t va[32];
                for (int c0 = cb; c0 < ce; c0 += 32) {
                    tmem_ld32(sb + c0, va);
                    tmem_ld_wait();
                    uint32_t pk[16];
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        const float e0 = ex2f(fmaf(__uint_as_float(va[j]), sl2, -mb));
                        const float e1 = ex2f(fmaf(__uint_as_float(va[j + 1]), sl2, -mb));
                        sum0 += e0; sum1 += e1;
                        pk[j >> 1] = float2_to_bf16x2(e0, e1);
                    }
                    tmem_st16(sb + cb + ((c0 - cb) >> 1), pk);
                }
            } else {
                uint32_t va[16], vb[16];
                auto exp16 = [&](const uint32_t (&cur)[16], uint32_t (&nxt)[16], int c0) {
                    if (exp_mode != 2) {
                        tmem_ld_wait();
                        if (c0 + 16 < ce) tmem_ld16(sb + c0 + 16, nxt);
                    }
                    uint32_t pk[8];
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        float e0 = fmaf(__uint_as_float(cur[j]), sl2, -mb), e1 = fmaf(__uint_as_float(cur[j + 1]), sl2, -mb);
                        if (exp_mode != 1) { e0 = ex2f(e0); e1 = ex2f(e1); }
                        sum0 += e0; sum1 += e1;
                        pk[j >> 1] = float2_to_bf16x2(e0, e1);
                    }
                    if (exp_mode != 2) tmem_st8(sb + cb + ((c0 - cb) >> 1), pk);
                    else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) nxt[j] = pk[j] + nxt[j + 8];
                    }
                };
                if (exp_mode != 2) tmem_ld16(sb + cb, va);
                else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) { va[j] = lane + j; vb[j] = lane * j; }
                }
                for (int c0 = cb; c0 < ce; c0 += 32) {
                    exp16(va, vb, c0);
                    if (c0 + 16 < ce) exp16(vb, va, c0 + 16);
                }
                if (exp_mode == 2) acc += __uint_as_float(va[3]) + __uint_as_float(vb[5]);
            }
            acc += sum0 + sum1;
            if (exp_mode != 2 && exp_mode < 4) tmem_st_wait();
        }
        t1 = clock64();
        if (lane == 0 && exp_mode >= 4) for (int i = 0; i < 4; ++i) out[32 + warp * 4 + i] = ph[i];
      }
    } else if (warp < 12) {
      if (exp_mode >= 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
      if (roles & 2) {
        for (int t = 0; t < tiles; ++t) {
            const uint32_t sb = lane_base + ((t + 1) & 1) * 224;
            if (help_mode != 2) {
                uint32_t va[32], vb[32];
                float mx = -1e30f;
                for (int c0 = 0; c0 < 197; c0 += 64) {
                    tmem_ld32(sb + c0, va);
                    tmem_ld32(sb + c0 + 32, vb);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j += 2) mx = fmax3f(mx, __uint_as_float(va[j]), __uint_as_float(va[j + 1]));
#pragma unroll
                    for (int j = 0; j < 32; j += 2) mx = fmax3f(mx, __uint_as_float(vb[j]), __uint_as_float(vb[j + 1]));
                }
                acc += mx;
            }
            if (help_mode != 1) {
                uint32_t o0[32], o1[32];
                tmem_ld32(lane_base + 448, o0);
                tmem_ld32(lane_base + 480, o1);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) acc += __uint_as_float(o0[j]) * 0.5f + __uint_as_float(o1[j]);
            }
        }
        t1 = clock64();
      }
    } else {
      if (exp_mode >= 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
      if (warp == 12 && lane == 0 && (roles & 4)) {
        const uint32_t idesc_s = umma_idesc_bf16(128, 208, 0, 0), idesc_o = umma_idesc_bf16(128, 64, 0, 1);
        const uint64_t qd = umma_desc_sw128(base, 16, 1024), kd = umma_desc_sw128(base + 32768, 16, 1024), vd = umma_desc_sw128(base + 65536, 16, 1024);
        long long iss = 0;
        for (int t = 0; t < tiles; ++t) {
            const uint32_t sbuf = tm + (t & 1) * 224;
            if (help_mode == 7) { mbar_wait(&pbar[t & 1], (t >> 1) & 1); tc_fence_after(); }
            const long long i0 = clock64();
            if (mma_mode != 1)
                for (int k = 0; k < 4; ++k) umma_bf16(sbuf, qd + k * 2, kd + k * 2, idesc_s, k != 0);
            if (mma_mode != 2)
                for (int k = 0; k < 13; ++k) umma_bf16_ts(tm + 448, tm + ((t + 1) & 1) * 224 + (k < 7 ? k * 8 : 112 + (k - 7) * 8), vd + (uint64_t)(k * 128), idesc_o, k != 0);
            iss += clock64() - i0;
        }
        out[20] = iss;
        umma_commit(&bar);
        mbar_wait(&bar, 0);
        t1 = clock64();
      }
    }
    if (lane == 0) out[warp] = t1 - t0;
    sink[threadIdx.x] = acc;
    tc_fence_before(); __syncthreads();
    if (warp == 12) { tc_fence_after(); tmem_dealloc(tm, 512); }
}

int main() {
    long long* out; float* sink;
    cudaMallocManaged(&out, 4096); cudaMallocManaged(&sink, 1 << 16);
    cudaFuncSetAttribute(pipe_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaFuncSetAttribute(pipe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaFuncSetAttribute(pipe_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaFuncSetAttribute(pipe_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaFuncSetAttribute(pipe_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    cudaFuncSetAttribute(pipe_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    const int tiles = 64;
    struct Cfg { int roles, exp_mode, help_mode, mma_mode; const char* name; };
    const Cfg cfgs[] = {
        {1, 4, 0, 0, "exp: whole half row in registers (v4 flow)"},
        {1, 5, 0, 0, "exp: v4 flow without the pair barrier"},
        {5, 4, 0, 0, "exp v4 + MMA"},
        {5, 4, 7, 0, "exp v4 + MMA issued per tile after the exp warps' barrier"},
        {5, 4, 7, 1, "exp v4 + MMA (TS only) issued after the barrier"},
        {7, 4, 2, 0, "exp v4 + helpers (O read only) + MMA"},
        {1, 0, 0, 0, "exp warps alone (ld16 / ffma+ex2+add / pack / st8)"},
        {1, 3, 0, 0, "exp warps alone, x32 chunks, no prefetch"},
        {1, 1, 0, 0, "exp warps alone, no MUFU"},
        {1, 2, 0, 0, "exp warps alone, no TMEM (registers only)"},
        {2, 0, 0, 0, "helpers alone (max pass + O read)"},
        {2, 0, 1, 0, "helpers alone (max pass only)"},
        {4, 0, 0, 0, "MMA alone (4 SS N=208 + 13 TS N=64 per tile)"},
        {4, 0, 0, 1, "MMA alone (13 TS only)"},
        {4, 0, 0, 2, "MMA alone (4 SS only)"},
        {3, 0, 0, 0, "exp + helpers"},
        {5, 0, 0, 0, "exp + MMA"},
        {5, 0, 0, 1, "exp + MMA (TS only)"},
        {5, 0, 0, 2, "exp + MMA (SS only)"},
        {5, 2, 0, 0, "exp (no TMEM) + MMA"},
        {5, 1, 0, 0, "exp (no MUFU) + MMA"},
        {6, 0, 0, 0, "helpers + MMA"},
        {7, 0, 0, 0, "exp + helpers + MMA"},
        {7, 0, 2, 0, "exp + helpers (O read only) + MMA"},
        {7, 2, 0, 0, "exp (no TMEM) + helpers + MMA"},
    };
    for (const Cfg& c : cfgs) {
        for (int it = 0; it < 2; ++it) {
            switch (c.exp_mode) {
                case 0: pipe_kernel<0><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
                case 1: pipe_kernel<1><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
                case 2: pipe_kernel<2><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
                case 3: pipe_kernel<3><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
                case 4: pipe_kernel<4><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
                default: pipe_kernel<5><<<1, 512, 160 * 1024>>>(c.roles, c.help_mode, c.mma_mode, tiles, out, sink); break;
            }
            cudaError_t e = cudaDeviceSynchronize();
            if (e != cudaSuccess) { printf("%s: %s\n", c.name, cudaGetErrorString(e)); return 1; }
        }
        long long ex = 0, hp = 0;
        for (int w = 0; w < 8; ++w) ex = out[w] > ex ? out[w] : ex;
        for (int w = 8; w < 12; ++w) hp = out[w] > hp ? out[w] : hp;
        printf("%-52s cycles per 128x208 tile:  exp %6.0f   helpers %6.0f   mma %6.0f", c.name,
               (c.roles & 1) ? (double)ex / tiles : 0.0, (c.roles & 2) ? (double)hp / tiles : 0.0, (c.roles & 4) ? (double)out[12] / tiles : 0.0);
        if (c.roles & 4) printf("  issue %5.0f", (double)out[20] / tiles);
        if (c.exp_mode >= 4) printf("   warp0 load %4.0f max %4.0f math %4.0f store %4.0f | warp4 load %4.0f max %4.0f math %4.0f store %4.0f",
                                    (double)out[32] / tiles, (double)out[33] / tiles, (double)out[34] / tiles, (double)out[35] / tiles,
                                    (double)out[48] / tiles, (double)out[49] / tiles, (double)out[50] / tiles, (double)out[51] / tiles);
        printf("\n");
    }
    return 0;
}
