// Persistent warp-specialised bf16 GEMM for sm_100a: TMA -> smem ring -> tcgen05.mma -> TMEM
// -> fused epilogue (bias, exact-erf GELU, gathered residual, row-remapped store).
//
//   D[orow(m), n] = epi( sum_k A[m,k] * W[n,k] )         A [M,K], W [N,K] (nn.Linear layout)
//
// Serves every dense contraction on the path: qkv (attention.py:22), proj (attention.py:55)
// with the kept-token residual gather folded into the epilogue (model.py:55-58), fc1+GELU,
// fc2+residual (model.py:59), patch-embed as a GEMM over im2col'd patches (+pos_embed as the
// "residual", model.py:34-37) and the classifier head (model.py:66).
//
// CTA = 352 threads, one CTA per SM, tiles 128 x BN x 64:
//   warps 0-7: epilogue; warp w reads TMEM lanes 32*(w%4).. and column half w/4
//   warp 8   : TMA producer (one lane)         warp 9 : tcgen05.mma issuer (one lane)
//   warp 10  : TMEM allocator
// (the single-lane producer and issuer sit on the HIGHEST warp ids: the issue arbiter favours them over
//  the epilogue warps they share a scheduler with, so a busy epilogue never delays an MMA or a TMA.)
// Pipelines: smem full/empty ring (TMA <-> MMA), TMEM full/empty double buffer (MMA <-> epilogue).
//
// Epilogue (hot modes): thread = output row (= TMEM lane).  Each warp pulls 32-column chunks of its
// rows straight from TMEM into registers (next chunk in flight while the current one is processed),
// applies the fused element-wise work with packed fp32x2 arithmetic (FFMA2), and writes 32-byte
// pieces of its own row (STG.256) - every thread fills whole sectors, no shared-memory transpose.
// The accumulator is handed back to the MMA issuer as soon as the last chunk is in registers.
//
// LayerNorm folding (model.py:51,59): LN(x) W^T = rstd*(x (W.gamma)^T - mean * wsum) + W beta, so the
// normalised activations are never materialised: the GEMM that PRODUCES x (proj / fc2 / patch-embed
// epilogue) also emits per-row partial (sum, sum of squares) of the bf16 values it stores, one slot
// per 32-column chunk; the GEMM that CONSUMES LN(x) (qkv / fc1) runs on x itself with
// gamma-scaled weights and applies  acc*rstd + (-mean*rstd)*wsum[n] + bias'[n]  in its epilogue.
#include <cuda.h>
#include <cstdlib>

#include "common.cuh"

namespace rajni {

constexpr int BM = 128;
constexpr int BK = 64;                 // 64 bf16 = one 128-byte swizzle row
constexpr int kGemmThreads = 352;
constexpr int kTmaWarp = 8, kMmaWarp = 9, kAllocWarp = 10;
constexpr int kEpiWarps = 8;
constexpr int kEpiStageBytes = 32 * 128;   // per-warp staging: 32 rows x 32 fp32

// CG = CTAs per MMA (tcgen05 cta_group): 1, or 2 = a CTA pair computing a 256 x BN tile together.
// In pair mode each CTA stages its own 128 A rows and BN/2 of the B rows, so a CTA pulls
// (128 + BN/2) x 64 bf16 from L2 per k-block instead of (128 + BN) x 64: the 1-CTA 128x256 tile is
// L2-bandwidth bound on B200 (measured 11.7 TB/s of operand traffic at ~1000 TFLOP/s).
template <int BN, int CG> struct GemmCfg {
    static constexpr int kBRows = BN / CG;                  // B rows staged by each CTA
    static constexpr int kABytes = BM * BK * 2;
    static constexpr int kBBytes = kBRows * BK * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kStages = (192 * 1024) / kStageBytes;
    static constexpr int kTmemCols = 2 * BN <= 64 ? 64 : 2 * BN <= 128 ? 128 : 2 * BN <= 256 ? 256 : 512;   // double-buffered accumulator, power of 2
    static constexpr int kSmemBytes = kStages * kStageBytes + kEpiWarps * kEpiStageBytes + 256 /*barriers*/ + 1024 /*align*/;
};

struct GemmParams {
    const float* bias;
    void* D;
    const __nv_bfloat16* residual;
    const int32_t* res_row_map;
    const int32_t* out_row_map;
    long long ldd, ldres;
    int M, N, K, flags;
    int tiles_m, tiles_n, k_blocks;
    int reverse_m;              // walk the M tiles from the last to the first (L2 reuse hint, results identical)
    // LayerNorm folding
    const float2* ln_stats;     // [ln_slots][ln_stats_ld] partial (sum, sumsq) of the rows of A
    const float* ln_wsum;       // [N] sum_k W'[n,k]
    long long ln_stats_ld;
    int ln_slots;
    float ln_inv_k, ln_eps;
    float2* row_stats;          // [N >> stat_shift][row_stats_ld] partial (sum, sumsq) of the rows of D per 32- or 64-column slot, or null
    long long row_stats_ld;
    int stat_shift;             // 5 or 6: log2 of the slot width (rajni_gemm_row_stats_slots)
    // stream-K tail (see "Stream-K" below): the first sk_tiles tiles are split along K over sk_pairs CTA pairs
    int sk_tiles, sk_pairs, sk_units;   // sk_units = sk_tiles * k_blocks
    float* sk_ws;               // fp32 partial accumulators: [pair][piece 0/1][cta rank][128][BN]
    int* sk_flags;              // [2][2 * sk_tiles]: partials arrived / finishing warps done, per (tile, cta rank); zero between launches
};

// ---------------------------------------------------------------------------------------------------------------------
// Stream-K tail.  tiles_m * tiles_n is rarely a multiple of the 74 CTA pairs: the last, partial wave costs a whole tile time
// (173 x 3 tiles = 7.01 waves -> 8).  For long K the R = tiles % pairs leftover tiles are therefore taken FIRST and split along
// K: their R * k_blocks k-blocks are dealt out evenly to sk_pairs CTA pairs (a contiguous range each, so a pair gets pieces of
// at most two tiles), every pair then runs its whole tiles as before.  A piece's fp32 accumulator goes to a scratch slot
// (thread = row, 128-byte runs) and a counter per (tile, CTA rank) is bumped; after its last whole tile each of the first
// min(pieces, BN/64) contributors of a tile adds up ALL the pieces of its own 64-column slices (fixed order: deterministic)
// and runs the usual fused epilogue on them - the fix-up is spread over the contributors, and by then the partials have
// been in L2 for the length of the kernel, so nobody waits.  Every piece is written before any pair starts waiting: no
// deadlock.  The last finisher zeroes the counters for the next launch (launches sharing a workspace are stream-ordered).
struct SkPlan { int n, tile0, k00, k10, tile1, k11; };      // piece 0 = (tile0, [k00, k10)), piece 1 = (tile1, [0, k11))
__device__ __forceinline__ int sk_bound(const GemmParams& p, int j) { return (int)(((long long)j * p.sk_units) / p.sk_pairs); }
// the pair whose range holds k-block unit u: the largest j with sk_bound(j) <= u
__device__ __forceinline__ int sk_pair_of(const GemmParams& p, int u) {
    return (int)(((long long)(u + 1) * p.sk_pairs + p.sk_units - 1) / p.sk_units) - 1;
}
template <bool SK>
__device__ __forceinline__ SkPlan sk_plan(const GemmParams& p, int pair) {
    SkPlan s{0, 0, 0, 0, 0, 0};
    if (SK && pair < p.sk_pairs) {
        const int b0 = sk_bound(p, pair), b1 = sk_bound(p, pair + 1);
        if (b1 > b0) {
            const int t0 = b0 / p.k_blocks, t1 = (b1 - 1) / p.k_blocks;
            s.tile0 = t0; s.k00 = b0 - t0 * p.k_blocks; s.k10 = min(b1 - t0 * p.k_blocks, p.k_blocks);
            s.n = 1;
            if (t1 > t0) { s.tile1 = t1; s.k11 = b1 - t1 * p.k_blocks; s.n = 2; }
        }
    }
    return s;
}
// item `it` of a pair's sequence of accumulator-producing work: its stream-K pieces first, then whole tiles
template <bool SK>
__device__ __forceinline__ bool sk_item(const GemmParams& p, const SkPlan& plan, int pair, int stride, int num_tiles, int it,
                                        int& tile, int& k0, int& k1) {
    if (SK && it < plan.n) {
        tile = it == 0 ? plan.tile0 : plan.tile1;
        k0 = it == 0 ? plan.k00 : 0;
        k1 = it == 0 ? plan.k10 : plan.k11;
        return true;
    }
    tile = (SK ? p.sk_tiles : 0) + pair + (it - (SK ? plan.n : 0)) * stride;
    k0 = 0; k1 = p.k_blocks;
    return tile < num_tiles;
}
__device__ __forceinline__ int ld_acquire_gpu(const int* ptr) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
    return v;
}

// Exact-erf GELU (timm nn.GELU) evaluated as x*Phi(x) with
//   Phi(-a) = 0.5 * 2^(-a*P(a)),  a = min(|x|, 6),  P = degree-4 fit of -log2(erfc(a/sqrt2))/a, weighted so that the error of
//   gelu relative to max(|gelu|, 1e-3) is equalised: 4.3e-5 at most (absolute 7e-6), i.e. ~50x below bf16 rounding.
// 9 FP32 instructions + one MUFU.EX2 instead of erff's ~30 (the fc1 epilogue is otherwise CUDA-core bound and, under the
// power cap, every FMA it saves is clock for the tensor pipe).  tools/gelu_fit.py derives the coefficients.
__device__ __forceinline__ float gelu_erf(float x) {
    const float a = fminf(fabsf(x), 6.0f);
    float p = 3.838799e-04f;
    p = fmaf(p, a, -6.4209225e-03f);
    p = fmaf(p, a, 5.0176125e-02f);
    p = fmaf(p, a, 0.4615304f);
    p = fmaf(p, a, 1.1504223f);
    const float s = x * (0.5f * ex2_approx(-a * p));
    return x >= 0.f ? x - s : s;
}

// Two GELUs per call on packed fp32x2.  Same fit, rearranged so that every step is an FFMA2:
//   na = -min(|x|, 6),  t = 2^(na*Q(na) - 1) = Phi(-|x|)  (Q = P with odd coefficients negated),
//   gelu(x) = relu(x) + na * t.      6 FFMA2 + 4 FMNMX + 2 MUFU.EX2 per pair.
__device__ __forceinline__ uint64_t gelu_erf2(uint64_t x2) {
    float x0, x1;
    f2unpack(x2, x0, x1);
    const uint64_t na = f2pack(fmaxf(-fabsf(x0), -6.0f), fmaxf(-fabsf(x1), -6.0f));
    uint64_t q = fma2(f2pack(3.838799e-04f, 3.838799e-04f), na, f2pack(6.4209225e-03f, 6.4209225e-03f));
    q = fma2(q, na, f2pack(5.0176125e-02f, 5.0176125e-02f));
    q = fma2(q, na, f2pack(-0.4615304f, -0.4615304f));
    q = fma2(q, na, f2pack(1.1504223f, 1.1504223f));
    const uint64_t arg = fma2(na, q, f2pack(-1.0f, -1.0f));
    float a0, a1;
    f2unpack(arg, a0, a1);
    return fma2(na, f2pack(ex2_approx(a0), ex2_approx(a1)), f2pack(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f)));
}

// explicit shared-state-space load (a generic pointer into dynamic smem compiles to LD.E)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// Epilogue modes: the three hot ones are compiled without any per-element flag or column-tail
// logic (they require N % BN == 0); MODE_GENERIC reads the runtime flags and handles every edge.
enum { MODE_GENERIC = 0, MODE_BIAS = 1, MODE_BIAS_GELU = 2, MODE_BIAS_RES = 3 };

// One 32-column chunk of one output row in the hot epilogues: cur = the fp32 accumulators (from TMEM, or summed stream-K
// partials), r = the residual's 32 bf16.  Bias / LayerNorm fold / GELU / residual in packed fp32x2, bf16 row stores, and the
// row statistics of the values as stored (MODE_BIAS_RES with row_stats).
template <int MODE, bool LN>
__device__ __forceinline__ void epi_chunk(const uint32_t (&cur)[32], const uint32_t (&r)[16], int ch, uint32_t sb, uint32_t sg,
                                          uint64_t rstd2, uint64_t mr2, uint64_t& sum2, uint64_t& sq2, bool wide_slots,
                                          bool valid, __nv_bfloat16* dptr, long long orow, int ncol0, const GemmParams& p) {
    constexpr bool kGelu = MODE == MODE_BIAS_GELU;
    constexpr bool kRes = MODE == MODE_BIAS_RES;
    uint32_t o[16];
    if (!wide_slots || !(ch & 1)) { sum2 = 0; sq2 = 0; }       // (0.f, 0.f): a new statistics slot starts here
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        const float4 bv = lds128(sb + (ch * 32 + j) * 4);
        uint64_t x01 = f2pack(__uint_as_float(cur[j]), __uint_as_float(cur[j + 1]));
        uint64_t x23 = f2pack(__uint_as_float(cur[j + 2]), __uint_as_float(cur[j + 3]));
        if (LN) {
            const float4 gv = lds128(sg + (ch * 32 + j) * 4);
            x01 = fma2(x01, rstd2, fma2(mr2, f2pack(gv.x, gv.y), f2pack(bv.x, bv.y)));
            x23 = fma2(x23, rstd2, fma2(mr2, f2pack(gv.z, gv.w), f2pack(bv.z, bv.w)));
        } else {
            x01 = add2(x01, f2pack(bv.x, bv.y));
            x23 = add2(x23, f2pack(bv.z, bv.w));
        }
        if (kGelu) {
            x01 = gelu_erf2(x01);
            x23 = gelu_erf2(x23);
        }
        if (kRes) {
            const float2 r0 = bf16x2_to_float2(r[j >> 1]), r1 = bf16x2_to_float2(r[(j >> 1) + 1]);
            x01 = add2(x01, f2pack(r0.x, r0.y));
            x23 = add2(x23, f2pack(r1.x, r1.y));
        }
        float e0, e1, e2, e3;
        f2unpack(x01, e0, e1);
        f2unpack(x23, e2, e3);
        o[j >> 1] = float2_to_bf16x2(e0, e1);
        o[(j >> 1) + 1] = float2_to_bf16x2(e2, e3);
        if (kRes) {
            // statistics of the values as stored (bf16-rounded), for the LayerNorm that follows
            const float2 q0 = bf16x2_to_float2(o[j >> 1]), q1 = bf16x2_to_float2(o[(j >> 1) + 1]);
            const uint64_t y01 = f2pack(q0.x, q0.y), y23 = f2pack(q1.x, q1.y);
            sum2 = add2(sum2, add2(y01, y23));
            sq2 = fma2(y01, y01, sq2);
            sq2 = fma2(y23, y23, sq2);
        }
    }
    if (valid) {
        stg256(dptr + ch * 32, *reinterpret_cast<uint32_t(*)[8]>(&o[0]));
        stg256(dptr + ch * 32 + 16, *reinterpret_cast<uint32_t(*)[8]>(&o[8]));
        if (kRes && p.row_stats != nullptr && (!wide_slots || (ch & 1))) {
            // one slot per 32 (or 64) columns of the row, whatever the tile width: the partition (and so the
            // rounding of the LayerNorm statistics) does not depend on the batch size
            float a0, a1, b0, b1;
            f2unpack(sum2, a0, a1);
            f2unpack(sq2, b0, b1);
            p.row_stats[(long long)((ncol0 + ch * 32) >> p.stat_shift) * p.row_stats_ld + orow] = make_float2(a0 + a1, b0 + b1);
        }
    }
}


template <int BN, int CG, int MODE, bool LN, bool SK>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const GemmParams p) {
    using Cfg = GemmCfg<BN, CG>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* s_a = smem;                                        // [stages][128][64] bf16, SW128
    uint8_t* s_b = smem + Cfg::kStages * Cfg::kABytes;          // [stages][BN/CG][64] bf16, SW128
    uint8_t* s_epi = smem + Cfg::kStages * Cfg::kStageBytes;    // [8 warps][32][32] fp32
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_epi + kEpiWarps * kEpiStageBytes);
    uint64_t* full_bar = bars;                                  // [stages]  (pair mode: the leader's is used)
    uint64_t* empty_bar = bars + Cfg::kStages;                  // [stages]
    uint64_t* tmem_full = bars + 2 * Cfg::kStages;              // [2]
    uint64_t* tmem_empty = tmem_full + 2;                       // [2]       (pair mode: the leader's is used)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_tiles = p.tiles_m * p.tiles_n;
    const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
    const int first_tile = blockIdx.x / CG, tile_stride = gridDim.x / CG;

    if (warp == kTmaWarp && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
    }
    if (warp == kMmaWarp && lane == 0) {
        for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(&full_bar[s], CG); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], kEpiWarps * CG); }
        mbar_fence_init();
    }
    if (warp == kAllocWarp) {
        if (CG == 2) tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);
        else tmem_alloc(tmem_slot, Cfg::kTmemCols);
    }
    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch();
    griddep_wait();          // everything above overlapped the previous kernel's tail; global memory from here on

    if (warp == kTmaWarp) {
        // ================= TMA producer (one lane per CTA) =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const SkPlan plan = sk_plan<SK>(p, first_tile);
            int tile, k0, k1;
            for (int it = 0; sk_item<SK>(p, plan, first_tile, tile_stride, num_tiles, it, tile, k0, k1); ++it) {
                const int m_lin = tile / p.tiles_n, n_blk = tile % p.tiles_n;
                const int m_blk = p.reverse_m ? p.tiles_m - 1 - m_lin : m_lin;
                const int row_a = m_blk * (BM * CG) + (int)cta_rank * BM;
                const int row_b = n_blk * BN + (int)cta_rank * Cfg::kBRows;
                for (int kb = k0; kb < k1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (CG == 2) {
                        const uint32_t lead_bar = mapa_u32(smem_u32(&full_bar[stage]), 0);
                        mbar_expect_tx_cluster(lead_bar, Cfg::kStageBytes);
                        tma_load_2d_cg2(s_a + stage * Cfg::kABytes, &tmap_a, lead_bar, kb * BK, row_a);
                        tma_load_2d_cg2(s_b + stage * Cfg::kBBytes, &tmap_b, lead_bar, kb * BK, row_b);
                    } else {
                        mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                        tma_load_2d(s_a + stage * Cfg::kABytes, &tmap_a, &full_bar[stage], kb * BK, row_a);
                        tma_load_2d(s_b + stage * Cfg::kBBytes, &tmap_b, &full_bar[stage], kb * BK, row_b);
                    }
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ================= MMA issuer (one lane of the leader CTA) =================
        if (lane == 0 && cta_rank == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BM * CG, BN, 0, 0);
            int stage = 0;
            uint32_t phase = 0;
            const SkPlan plan = sk_plan<SK>(p, first_tile);
            int tile, k0, k1;
            for (int local = 0; sk_item<SK>(p, plan, first_tile, tile_stride, num_tiles, local, tile, k0, k1); ++local) {
                const int acc = local & 1;
                const uint32_t acc_phase = (local >> 1) & 1;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);          // epilogues have drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = k0; kb < k1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(s_a + stage * Cfg::kABytes);
                    const uint32_t b_addr = smem_u32(s_b + stage * Cfg::kBBytes);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        // advancing 16 bf16 along K = +32 bytes inside the 128-byte swizzle row
                        const uint64_t a_desc = umma_desc_sw128(a_addr + k * 32, 16, 1024);
                        const uint64_t b_desc = umma_desc_sw128(b_addr + k * 32, 16, 1024);
                        if (CG == 2) umma_bf16_cg2(d_tmem, a_desc, b_desc, idesc, (uint32_t)(kb != k0 || k != 0));
                        else umma_bf16(d_tmem, a_desc, b_desc, idesc, (uint32_t)(kb != k0 || k != 0));
                    }
                    // frees the smem slot (in both CTAs of a pair) when these MMAs finish
                    if (CG == 2) umma_commit_cg2(&empty_bar[stage], 0x3); else umma_commit(&empty_bar[stage]);
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
                // accumulator ready for the epilogue warps (of both CTAs)
                if (CG == 2) umma_commit_cg2(&tmem_full[acc], 0x3); else umma_commit(&tmem_full[acc]);
            }
        }
    } else if (warp < kEpiWarps) {
        // ================= epilogue =================
        const int ew = warp;
        const int sub = warp & 3;                   // TMEM sub-partition = warp id % 4
        const int half = ew >> 2;                   // which half of the BN columns
        const uint32_t stg = smem_u32(s_epi + ew * kEpiStageBytes);
        if (MODE != MODE_GENERIC) {
            // ---------- hot modes: thread = row, straight from TMEM, packed fp32x2 math, 32-byte row stores ----------
            constexpr int HALF = BN / 2;                // columns per epilogue warp
            constexpr int NCH = HALF / 32;              // 32-column chunks per warp and tile
            constexpr bool kGelu = MODE == MODE_BIAS_GELU;
            constexpr bool kRes = MODE == MODE_BIAS_RES;
            const uint32_t sb = stg, sg = stg + HALF * 4;   // this warp's bias / weight-row-sum vectors
            __nv_bfloat16* const Dp = static_cast<__nv_bfloat16*>(p.D);
            const bool wide_slots = kRes && p.stat_shift == 6;   // 64-column statistics slots: two chunks each (NCH is even then)
            const int pair = first_tile;
            // ---- state of the tile being finished (set by `setup`)
            int ncol0 = 0;
            bool valid = false;
            long long orow = 0;
            __nv_bfloat16* dptr = nullptr;
            uint32_t rr[kRes ? NCH : 1][16];
            uint64_t rstd2 = 0, mr2 = 0;
            // everything of a tile's epilogue that does not need the accumulator; `chunks`: bit c = this warp will process chunk c
            auto setup = [&](int tile, uint32_t chunks) {
                const int m_lin = tile / p.tiles_n, n_blk = tile % p.tiles_n;
                const int m_blk = p.reverse_m ? p.tiles_m - 1 - m_lin : m_lin;
                const int m = m_blk * (BM * CG) + (int)cta_rank * BM + sub * 32 + lane;
                valid = m < p.M;
                ncol0 = n_blk * BN + half * HALF;
                // column vectors of this tile -> the warp's shared slice (read back as broadcasts)
                __syncwarp();
                if (lane < HALF / 4) {
                    const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + ncol0) + lane);
                    sts128(sb + lane * 16, __float_as_uint(bv.x), __float_as_uint(bv.y), __float_as_uint(bv.z), __float_as_uint(bv.w));
                    if (LN) {
                        const float4 gv = __ldg(reinterpret_cast<const float4*>(p.ln_wsum + ncol0) + lane);
                        sts128(sg + lane * 16, __float_as_uint(gv.x), __float_as_uint(gv.y), __float_as_uint(gv.z), __float_as_uint(gv.w));
                    }
                }
                __syncwarp();
                orow = 0;
                if (valid) orow = p.out_row_map ? (long long)__ldg(p.out_row_map + m) : (long long)m;
                dptr = Dp + orow * p.ldd + ncol0;
                // the whole residual slab of this thread's row (HALF bf16) is requested before the wait for the
                // accumulator, so its DRAM latency hides behind the MMAs of this tile
                if (kRes) {
                    if (valid) {
                        const __nv_bfloat16* rptr = p.residual + (p.res_row_map ? (long long)__ldg(p.res_row_map + m) : (long long)m) * p.ldres + ncol0;
#pragma unroll
                        for (int c = 0; c < NCH; ++c) {
                            if (!((chunks >> c) & 1u)) continue;
                            ldg256(rptr + c * 32, *reinterpret_cast<uint32_t(*)[8]>(&rr[kRes ? c : 0][0]));      // (coherent: the residual may alias D)
                            ldg256(rptr + c * 32 + 16, *reinterpret_cast<uint32_t(*)[8]>(&rr[kRes ? c : 0][8]));
                        }
                    }
                }
                if (LN) {
                    // row statistics of A from the producer's partial sums (model.py:51,59: LayerNorm, biased variance)
                    float s1 = 0.f, s2 = 0.f;
                    if (valid) {
                        for (int sl = 0; sl < p.ln_slots; ++sl) {
                            const float2 t = __ldg(p.ln_stats + (long long)sl * p.ln_stats_ld + m);
                            s1 += t.x;
                            s2 += t.y;
                        }
                    }
                    const float mean = s1 * p.ln_inv_k;
                    const float rstd = rsqrtf(fmaxf(s2 * p.ln_inv_k - mean * mean, 0.f) + p.ln_eps);
                    rstd2 = f2pack(rstd, rstd);
                    mr2 = f2pack(-mean * rstd, -mean * rstd);
                }
            };
            uint32_t va[32], vb[32];
            uint64_t sum2 = 0, sq2 = 0;                      // row statistics of the current slot (kRes)
            int local = 0;
            if (SK) {
                // ---- this pair's stream-K pieces come first: the fp32 partial goes to the pair's scratch slot, the tile is
                //      finished after the whole tiles (below).  (A piece is never a whole tile: sk_decide.)
                const int n_pieces = sk_plan<SK>(p, pair).n;
                for (; local < n_pieces; ++local) {
                    const SkPlan plan = sk_plan<SK>(p, pair);
                    const int tile = local == 0 ? plan.tile0 : plan.tile1;
                    const int acc = local & 1;
                    const uint32_t taddr = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * BN + half * HALF);
                    // slot layout: [warp (sub, half)][chunk][4-column group][lane][4 fp32] - every warp store / load is 512 contiguous bytes
                    float* slot = p.sk_ws + (size_t)((pair * 2 + local) * 2 + (int)cta_rank) * (BM * BN) + (size_t)(sub * 2 + half) * (32 * HALF) + lane * 4;
                    mbar_wait(&tmem_full[acc], 0);
                    tc_fence_after();
                    tmem_ld32(taddr, va);
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch) {
                        uint32_t (&cur)[32] = (ch & 1) ? vb : va;
                        uint32_t (&nxt)[32] = (ch & 1) ? va : vb;
                        tmem_ld_wait();
                        if (ch + 1 < NCH) {
                            tmem_ld32(taddr + (ch + 1) * 32, nxt);
                        } else {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) {
                                if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty[acc]), 0));
                                else mbar_arrive(&tmem_empty[acc]);
                            }
                        }
#pragma unroll
                        for (int g = 0; g < 8; ++g)
                            st_stream16(slot + (ch * 8 + g) * 128, make_uint4(cur[4 * g], cur[4 * g + 1], cur[4 * g + 2], cur[4 * g + 3]));
                    }
                    __syncwarp();
                    if (lane == 0) {
                        __threadfence();                     // the warp's stores (ordered before this by the __syncwarp) are visible first
                        atomicAdd(p.sk_flags + tile * 2 + (int)cta_rank, 1);
                    }
                }
            }
            const int local0 = local;
            for (int tile = (SK ? p.sk_tiles : 0) + pair; tile < num_tiles; tile += tile_stride, ++local) {
                const int acc = local & 1;
                const uint32_t acc_phase = (local >> 1) & 1;
                const uint32_t taddr = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * BN + half * HALF);
                setup(tile, 0xffffffffu);
                mbar_wait(&tmem_full[acc], acc_phase);
                tc_fence_after();
                tmem_ld32(taddr, va);
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    uint32_t (&cur)[32] = (ch & 1) ? vb : va;
                    uint32_t (&nxt)[32] = (ch & 1) ? va : vb;
                    tmem_ld_wait();
                    if (ch + 1 < NCH) {
                        tmem_ld32(taddr + (ch + 1) * 32, nxt);
                    } else {
                        // every chunk of this warp's rows is in registers: give the accumulator back
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty[acc]), 0));
                            else mbar_arrive(&tmem_empty[acc]);
                        }
                    }
                    epi_chunk<MODE, LN>(cur, rr[kRes ? ch : 0], ch, sb, sg, rstd2, mr2, sum2, sq2, wide_slots, valid, dptr, orow, ncol0, p);
                }
            }
            // ---- stream-K: finish this pair's share of the split tiles it contributed to
            for (int q = 0; SK && q < local0; ++q) {
                int pair_o = pair;
                asm volatile("" : "+r"(pair_o));                            // (recomputed here rather than kept live across the tile loop)
                const SkPlan plan = sk_plan<SK>(p, pair_o);
                const int t = q == 0 ? plan.tile0 : plan.tile1, u0 = t * p.k_blocks;
                const int jf = sk_pair_of(p, u0), jl = sk_pair_of(p, u0 + p.k_blocks - 1);
                const int pieces = jl - jf + 1, me = pair - jf;
                constexpr int UNITS = BN / 64;                               // 64-column slices of a tile (= statistics slots)
                const int nfin = pieces < UNITS ? pieces : UNITS;
                if (me >= nfin) continue;
                uint32_t mine = 0;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) if ((((half * HALF + ch * 32) >> 6) % nfin) == me) mine |= 1u << ch;
                int* const arrived = p.sk_flags + t * 2 + (int)cta_rank;
                int* const done = arrived + 2 * p.sk_tiles;
                setup(t, 0u);                                               // (the residual is fetched per chunk below)
                if (mine != 0) {
                    if (lane == 0) {
                        // pieces * 8 epilogue warps of this CTA rank arrive; all of them were written before anybody waits here
                        unsigned spins = 0;
                        while (ld_acquire_gpu(arrived) < pieces * kEpiWarps) {
                            __nanosleep(200);
                            if (++spins > (1u << 24)) asm volatile("trap;");  // (seconds: a lost contributor must not hang the GPU)
                        }
                    }
                    __syncwarp();
                    // slot of contributor i: its first piece unless the pair's range began in the previous tile
                    const int q0 = sk_bound(p, jf) == u0 ? 0 : 1;
                    const size_t slot_floats = (size_t)2 * BM * BN;          // both CTA ranks of one piece
                    const float* const base0 = p.sk_ws + ((size_t)(jf * 2 + q0) * 2 + (int)cta_rank) * (BM * BN) + (size_t)(sub * 2 + half) * (32 * HALF) + lane * 4;
                    const float* const base1 = p.sk_ws + ((size_t)(jf * 2 + 2) * 2 + (int)cta_rank) * (BM * BN) + (size_t)(sub * 2 + half) * (32 * HALF) + lane * 4;
                    const __nv_bfloat16* rptr = nullptr;
                    if (kRes && valid) {
                        const int m_lin = t / p.tiles_n;
                        const int m = (p.reverse_m ? p.tiles_m - 1 - m_lin : m_lin) * (BM * CG) + (int)cta_rank * BM + sub * 32 + lane;
                        rptr = p.residual + (p.res_row_map ? (long long)__ldg(p.res_row_map + m) : (long long)m) * p.ldres + ncol0;
                    }
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch) {
                        if (!((mine >> ch) & 1u)) continue;
                        uint32_t r1[16];
                        if (kRes && valid) {
                            ldg256(rptr + ch * 32, *reinterpret_cast<uint32_t(*)[8]>(&r1[0]));
                            ldg256(rptr + ch * 32 + 16, *reinterpret_cast<uint32_t(*)[8]>(&r1[8]));
                        }
                        // sum of the pieces in contributor order (deterministic); two pieces' loads in flight at a time
                        float a32[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) a32[j] = 0.f;
                        for (int i = 0; i < pieces; i += 2) {
                            const float* s0 = (i == 0 ? base0 : base1 + (size_t)(i - 1) * 2 * slot_floats) + ch * 1024;
                            const bool two = i + 1 < pieces;
                            const float* s1 = base1 + (size_t)i * 2 * slot_floats + ch * 1024;
                            float4 x[8], y[8];
#pragma unroll
                            for (int g = 0; g < 8; ++g) x[g] = __ldcg(reinterpret_cast<const float4*>(s0 + g * 128));
#pragma unroll
                            for (int g = 0; g < 8; ++g) y[g] = two ? __ldcg(reinterpret_cast<const float4*>(s1 + g * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                            for (int g = 0; g < 8; ++g) { a32[4 * g] += x[g].x; a32[4 * g + 1] += x[g].y; a32[4 * g + 2] += x[g].z; a32[4 * g + 3] += x[g].w; }
#pragma unroll
                            for (int g = 0; g < 8; ++g) { a32[4 * g] += y[g].x; a32[4 * g + 1] += y[g].y; a32[4 * g + 2] += y[g].z; a32[4 * g + 3] += y[g].w; }
                        }
#pragma unroll
                        for (int j = 0; j < 32; ++j) va[j] = __float_as_uint(a32[j]);
                        epi_chunk<MODE, LN>(va, r1, ch, sb, sg, rstd2, mr2, sum2, sq2, wide_slots, valid, dptr, orow, ncol0, p);
                    }
                }
                __syncwarp();
                if (lane == 0) {
                    // the last of the nfin * 8 finishing warps re-arms the counters for the next launch
                    if (atomicAdd(done, 1) == nfin * kEpiWarps - 1) {
                        *arrived = 0;
                        *done = 0;
                    }
                }
            }
        } else {
        // ---------- generic mode: runtime flags, column tails, fp32 output, staged through shared memory ----------
        const bool has_bias = (p.flags & RAJNI_EPI_BIAS) != 0;
        const bool do_gelu = (p.flags & RAJNI_EPI_GELU) != 0;
        const bool has_res = (p.flags & RAJNI_EPI_RESIDUAL) != 0;
        const bool out_f32 = (p.flags & RAJNI_EPI_OUT_F32) != 0;
        const int r_in = lane >> 3;                 // row within a group of 4 (phase 2)
        const int c4 = lane & 7;                    // 4-column group within the 32-column chunk
        // phase-1 / phase-2 staging addresses (XOR swizzle on 16-byte slots; both conflict-free)
        uint32_t st_addr[8], ld_addr[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) st_addr[c] = stg + lane * 128 + ((c ^ (lane & 7)) << 4);
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int r = it * 4 + r_in;
            ld_addr[it] = stg + r * 128 + ((c4 ^ (r & 7)) << 4);
        }
        int local = 0;
        for (int tile = first_tile; tile < num_tiles; tile += tile_stride, ++local) {
            const int m_lin = tile / p.tiles_n, n_blk = tile % p.tiles_n;
            const int m_blk = p.reverse_m ? p.tiles_m - 1 - m_lin : m_lin;
            const int acc = local & 1;
            const uint32_t acc_phase = (local >> 1) & 1;
            const int row0 = m_blk * (BM * CG) + (int)cta_rank * BM + sub * 32;
            const int ncol0 = n_blk * BN + half * (BN / 2) + c4 * 4;     // this lane's first column
            // rows this lane handles in phase 2: row0 + it*4 + r_in
            uint32_t valid = 0;
            long long ooff[8], roff[8];
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int m = row0 + it * 4 + r_in;
                ooff[it] = 0;
                roff[it] = 0;
                if (m < p.M) {
                    valid |= 1u << it;
                    ooff[it] = (p.out_row_map ? (long long)__ldg(p.out_row_map + m) : (long long)m) * p.ldd + ncol0;
                    if (has_res)
                        roff[it] = (p.res_row_map ? (long long)__ldg(p.res_row_map + m) : (long long)m) * p.ldres + ncol0;
                }
            }
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
#pragma unroll 1
            for (int ch = 0; ch < BN / 64; ++ch) {
                const int n = ncol0 + ch * 32;
                const uint32_t taddr = tmem_base + ((uint32_t)(sub * 32) << 16) + (uint32_t)(acc * BN + half * (BN / 2) + ch * 32);
                // ---------- generic path: runtime flags, column tails, fp32 output ----------
                const bool full4 = (n + 4 <= p.N);
                uint32_t v[32];
                tmem_ld32(taddr, v);
                tmem_ld_wait();
#pragma unroll
                for (int c = 0; c < 8; ++c) sts128(st_addr[c], v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                __syncwarp();
                float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_bias && n < p.N) {
                    if (full4) bv = __ldg(reinterpret_cast<const float4*>(p.bias + n));
                    else {
                        bv.x = __ldg(p.bias + n);
                        if (n + 1 < p.N) bv.y = __ldg(p.bias + n + 1);
                        if (n + 2 < p.N) bv.z = __ldg(p.bias + n + 2);
                    }
                }
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    float4 a = lds128(ld_addr[it]);
                    if (!((valid >> it) & 1) || n >= p.N) continue;
                    a.x += bv.x; a.y += bv.y; a.z += bv.z; a.w += bv.w;
                    if (do_gelu) { a.x = gelu_erf(a.x); a.y = gelu_erf(a.y); a.z = gelu_erf(a.z); a.w = gelu_erf(a.w); }
                    if (has_res) {
                        const __nv_bfloat16* rp = p.residual + roff[it] + ch * 32;
                        if (full4) {
                            const uint2 rr = __ldg(reinterpret_cast<const uint2*>(rp));
                            const float2 r0 = bf16x2_to_float2(rr.x), r1 = bf16x2_to_float2(rr.y);
                            a.x += r0.x; a.y += r0.y; a.z += r1.x; a.w += r1.y;
                        } else {
                            a.x += __bfloat162float(rp[0]);
                            if (n + 1 < p.N) a.y += __bfloat162float(rp[1]);
                            if (n + 2 < p.N) a.z += __bfloat162float(rp[2]);
                        }
                    }
                    if (out_f32) {
                        float* dp = static_cast<float*>(p.D) + ooff[it] + ch * 32;
                        if (full4) *reinterpret_cast<float4*>(dp) = a;
                        else {
                            dp[0] = a.x;
                            if (n + 1 < p.N) dp[1] = a.y;
                            if (n + 2 < p.N) dp[2] = a.z;
                        }
                    } else {
                        __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(p.D) + ooff[it] + ch * 32;
                        if (full4) *reinterpret_cast<uint2*>(dp) = make_uint2(float2_to_bf16x2(a.x, a.y), float2_to_bf16x2(a.z, a.w));
                        else {
                            dp[0] = __float2bfloat16(a.x);
                            if (n + 1 < p.N) dp[1] = __float2bfloat16(a.y);
                            if (n + 2 < p.N) dp[2] = __float2bfloat16(a.z);
                        }
                    }
                }
                __syncwarp();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty[acc]), 0));
                else mbar_arrive(&tmem_empty[acc]);
            }
        }
        }
    }

    tc_fence_before();
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == kAllocWarp) {
        tc_fence_after();
        if (CG == 2) tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols);
        else tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
    return fn;
}

// One cuTensorMapEncodeTiled call on a bf16 tensor of `rank` <= 3 dimensions (dims and box innermost first, strides in
// bytes for dims 1..rank-1): unit element strides, 128-byte swizzle, zero OOB fill.  Sets `r` to the driver's result and
// returns 0, or RAJNI_ECUDA when the driver lacks the entry point.
static int encode_tmap_bf16(CUtensorMap* map, const void* base, cuuint32_t rank, const cuuint64_t* dims, const cuuint64_t* strides,
                            const cuuint32_t* box, CUtensorMapL2promotion l2, CUresult& r) {
    EncodeTiledFn fn = get_encode_fn();
    RAJNI_REQUIRE(fn != nullptr, RAJNI_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), dims, strides, box, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return 0;
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems, int box_rows) {
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld_elems * 2};
    const cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
    CUresult r;
    if (int rc = encode_tmap_bf16(map, base, 2, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, r)) return rc;
    RAJNI_REQUIRE(r == CUDA_SUCCESS, RAJNI_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld box=%dx%d",
                  (int)r, rows, cols, ld_elems, box_rows, 64);
    return 0;
}
// [batch][rows][cols], densely packed: the two 3-D views differ only in L2 promotion
int make_tmap_bf16_3d_box(CUtensorMap* map, const void* base, long long batch, long long rows, long long cols, int box_rows) {
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows * (cuuint64_t)cols * 2};
    const cuuint32_t box[3] = {64u, (cuuint32_t)box_rows, 1u};
    CUresult r;
    if (int rc = encode_tmap_bf16(map, base, 3, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE, r)) return rc;
    RAJNI_REQUIRE(r == CUDA_SUCCESS, RAJNI_ECUDA, "cuTensorMapEncodeTiled (3d) failed (%d) batch=%lld rows=%lld cols=%lld",
                  (int)r, batch, rows, cols);
    return 0;
}
int make_tmap_bf16_3d_ld(CUtensorMap* map, const void* base, long long batch, long long rows, long long cols, int box_rows) {
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows * (cuuint64_t)cols * 2};
    const cuuint32_t box[3] = {64u, (cuuint32_t)box_rows, 1u};
    CUresult r;
    if (int rc = encode_tmap_bf16(map, base, 3, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, r)) return rc;
    RAJNI_REQUIRE(r == CUDA_SUCCESS, RAJNI_ECUDA, "cuTensorMapEncodeTiled (3d load) failed (%d) batch=%lld rows=%lld cols=%lld box_rows=%d",
                  (int)r, batch, rows, cols, box_rows);
    return 0;
}

// Stream-K scratch: a 4 KB header of counters, then one fp32 slot per (pair, piece, CTA rank) of 128 x 256 accumulators.
constexpr size_t kSkHeaderBytes = 4096;
constexpr int kSkMinKBlocks = 16;          // shorter K: a tile is too cheap for a fix-up to pay
constexpr int kSkMinPiece = 8;             // k-blocks per pair at least (bounds the pieces per tile at k_blocks / 8 + 1)
static size_t sk_workspace_bytes() { return kSkHeaderBytes + (size_t)(num_sms() / 2) * 2 * 2 * BM * 256 * sizeof(float); }

// Decide whether the leftover tiles of the last wave are split along K (see "Stream-K" above).  Time is counted in k-blocks
// of one pair: without the split the R leftover tiles cost a whole extra tile time (k_blocks); with it every sharing pair
// gets ceil(R * k_blocks / pairs) k-blocks plus the fix-up - writing the fp32 partials (256 KB per pair and piece) and
// reading them back costs ~`fix` k-block times, measured (profiles/r2_gemm_stream_k.md: 6-10 us with few pieces, 17-27 us
// when every pair holds two).  The split must save at least 15 % of the whole call: that admits the short calls of small
// shards (M = 6304, K = 3072: 41.0 -> 33.4 us) and rejects the long ones, where under the power cap an idle tail costs
// little anyway (M = 44288: 153.9 vs 156.1 us).  Returns R (0: no split) and the number of pairs that share the pieces.
static int sk_decide(int tiles, int pairs, int k_blocks, bool force, int* sk_pairs) {
    static const char* env = getenv("RAJNI_GEMM_SK");                       // "0" disables, "1" forces wherever it is legal
    static const int fix = getenv("RAJNI_GEMM_SK_FIX") ? atoi(getenv("RAJNI_GEMM_SK_FIX")) : 20;
    if (env && env[0] == '0') return 0;
    const int R = tiles % pairs, full = tiles / pairs;
    if (R == 0 || k_blocks < kSkMinKBlocks) return 0;
    long long units = (long long)R * k_blocks;
    int sp = (int)(units / kSkMinPiece);
    if (sp > pairs) sp = pairs;
    if (sp < R) sp = R;                                                      // a pair's range never spans three tiles
    const int per_pair = (int)((units + sp - 1) / sp);
    if (per_pair >= k_blocks) return 0;                                      // nothing is split (and a piece is never a whole tile)
    const bool forced = force || (env && env[0] == '1');
    if (!forced && (long long)(k_blocks - per_pair - fix) * 100 < 15LL * (full + 1) * k_blocks) return 0;
    *sk_pairs = sp;
    return R;
}

template <int BN, int CG, int MODE, bool LN>
static int launch_gemm_mode(const void* A, const void* W, GemmParams& p, void* ws, size_t ws_bytes, cudaStream_t stream) {
    using Cfg = GemmCfg<BN, CG>;
    CUtensorMap ta, tb;
    if (int rc = make_tmap_bf16_2d(&ta, A, p.M, p.K, p.K, BM)) return rc;
    if (int rc = make_tmap_bf16_2d(&tb, W, p.N, p.K, p.K, Cfg::kBRows)) return rc;
    p.tiles_m = (p.M + BM * CG - 1) / (BM * CG);
    p.tiles_n = (p.N + BN - 1) / BN;
    p.k_blocks = (p.K + BK - 1) / BK;
    int max_grid = (num_sms() / CG) * CG;
    static const int cta_cap = getenv("RAJNI_GEMM_MAX_CTAS") ? atoi(getenv("RAJNI_GEMM_MAX_CTAS")) : 0;     // experiments: leave SMs free
    if (cta_cap > 0 && cta_cap < max_grid) max_grid = (cta_cap / CG) * CG;
    int grid = p.tiles_m * p.tiles_n * CG;
    if (grid > max_grid) grid = max_grid;
    constexpr bool kSkCapable = BN == 256 && CG == 2 && MODE != MODE_GENERIC;
    bool sk = false;
    if (kSkCapable && ws != nullptr && ws_bytes >= sk_workspace_bytes() && (reinterpret_cast<uintptr_t>(ws) & 127u) == 0) {
        int sp = 0;
        const int R = sk_decide(p.tiles_m * p.tiles_n, max_grid / CG, p.k_blocks, (p.flags & RAJNI_HINT_STREAM_K) != 0, &sp);
        if (R > 0) {
            sk = true;
            p.sk_tiles = R; p.sk_pairs = sp; p.sk_units = R * p.k_blocks;
            p.sk_flags = static_cast<int*>(ws);
            p.sk_ws = reinterpret_cast<float*>(static_cast<char*>(ws) + kSkHeaderBytes);
            if (grid < sp * CG) grid = sp * CG;          // fewer tiles than pairs: the pieces still go to sk_pairs pairs
        }
    }
    auto kern = gemm_bf16_kernel<BN, CG, MODE, LN, false>;
    if constexpr (kSkCapable) { if (sk) kern = gemm_bf16_kernel<BN, CG, MODE, LN, true>; }
    static int smem_granted[2][kMaxDevices] = {};
    if (int rc = raise_smem_limit("gemm", kern, Cfg::kSmemBytes, smem_granted[sk ? 1 : 0])) return rc;
    return launch_checked("gemm_bf16", kern, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, stream, CG, ta, tb, p);
}

static bool aligned32(const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 31u) == 0; }

// Pick the compile-time epilogue.  The hot modes need: no column tail, 32-byte-aligned rows of D (and of
// the residual), bf16 output, and one of the flag combinations below; everything else runs MODE_GENERIC.
template <int BN, int CG>
static int launch_gemm(const void* A, const void* W, GemmParams& p, void* ws, size_t ws_bytes, cudaStream_t stream) {
    const int ln = p.flags & RAJNI_EPI_LN_FOLD, stats = p.flags & RAJNI_EPI_ROW_STATS;
    const int core = p.flags & ~(RAJNI_EPI_LN_FOLD | RAJNI_EPI_ROW_STATS | RAJNI_HINT_REVERSE_M | RAJNI_HINT_STREAM_K);
    bool hot = p.N % BN == 0 && p.ldd % 16 == 0 && aligned32(p.D);
    if (core & RAJNI_EPI_RESIDUAL) hot = hot && p.ldres % 16 == 0 && aligned32(p.residual);
    if (hot) {
        if (core == RAJNI_EPI_BIAS && !stats)
            return ln ? launch_gemm_mode<BN, CG, MODE_BIAS, true>(A, W, p, ws, ws_bytes, stream) : launch_gemm_mode<BN, CG, MODE_BIAS, false>(A, W, p, ws, ws_bytes, stream);
        if (core == (RAJNI_EPI_BIAS | RAJNI_EPI_GELU) && !stats)
            return ln ? launch_gemm_mode<BN, CG, MODE_BIAS_GELU, true>(A, W, p, ws, ws_bytes, stream) : launch_gemm_mode<BN, CG, MODE_BIAS_GELU, false>(A, W, p, ws, ws_bytes, stream);
        if (core == (RAJNI_EPI_BIAS | RAJNI_EPI_RESIDUAL) && !ln)
            return launch_gemm_mode<BN, CG, MODE_BIAS_RES, false>(A, W, p, ws, ws_bytes, stream);
    }
    RAJNI_REQUIRE(!ln && !stats, RAJNI_EINVAL,
                  "rajni_gemm_bf16: LN_FOLD / ROW_STATS need N %% %d == 0, ldd/ldres multiples of 16 and 32-byte aligned rows "
                  "(N=%d ldd=%lld ldres=%lld flags=%d)", BN, p.N, p.ldd, p.ldres, p.flags);
    return launch_gemm_mode<BN, CG, MODE_GENERIC, false>(A, W, p, ws, ws_bytes, stream);
}

// Tile width.  Generic epilogue: minimise padded columns (the 64-wide tile runs at ~2/3 rate, shared-memory bound).
// `exact` (hot epilogues, no column-tail path): among the widths that divide N, the CTA-pair tiles (256 or 192 wide,
// 256 rows) are preferred; between those two the one with fewer, fuller waves over the 74 CTA pairs wins
// (e.g. N = 768, M = 44288: 173 x 3 tiles of 256 = 7.01 waves -> 8, but 173 x 4 tiles of 192 = 9.35 -> 10 x 3/4 = 7.5).
static int pick_bn(int N, int M, int K, bool exact, bool no192, bool sk_ws, bool force_sk = false) {
    if (exact) {
        static const char* force = getenv("RAJNI_GEMM_BN");                 // debugging aid: force a pair-tile width that divides N
        if (force && M > BM && N % atoi(force) == 0 && (atoi(force) == 256 || (atoi(force) == 192 && !no192) || atoi(force) == 128)) return -atoi(force);
        const bool pair = M > BM;
        int best = 0;
        double best_cost = 0;
        for (int bn : {256, 192, 128}) {
            if (!pair || N % bn || (no192 && bn == 192)) continue;
            const long long tiles = (long long)((M + 2 * BM - 1) / (2 * BM)) * (N / bn);
            const int pairs = num_sms() / 2;
            double waves = (double)((tiles + pairs - 1) / pairs);
            if (bn == 256 && sk_ws) {
                // the 256-wide tile can split its leftover tiles along K (stream-K): the last wave then costs a fraction
                int sp = 0;
                const int kb = (K + BK - 1) / BK;
                if (sk_decide((int)tiles, pairs, kb, force_sk, &sp) > 0)
                    waves = (double)(tiles / pairs) + (double)((tiles % pairs) * kb / sp + 20) / kb;
            }
            // the 192-wide tile re-reads A once more per row block: it has to save 8 % of the wave time to be chosen
            // (the 128-wide pair tile re-reads A twice as often and halves the work per accumulator hand-over: 20 %)
            const double cost = waves * bn * (bn == 192 ? 1.08 : bn == 128 ? 1.2 : 1.0);
            if (!best || cost < best_cost) { best = bn; best_cost = cost; }
        }
        if (best) return -best;                     // negative: CTA-pair tile
        return N % 256 == 0 ? 256 : N % 128 == 0 ? 128 : 64;
    }
    auto cost = [&](int bn) { long long padded = (long long)((N + bn - 1) / bn) * bn; return bn == 64 ? padded * 3 / 2 : padded; };
    int bn = 256;
    if (cost(128) < cost(bn)) bn = 128;
    if (cost(64) < cost(bn)) bn = 64;
    return bn;
}

}  // namespace rajni

using namespace rajni;

// Slot width of the row statistics: 64 columns when N is a multiple of 128 (the producer then uses 256- or 128-wide tiles only,
// whose epilogue warps own whole 64-column slots), else 32 (N = 192: the 192-wide tile's warps own 96 columns).
static int stat_shift_for(int N) { return N % 128 == 0 ? 6 : 5; }

extern "C" int rajni_gemm_row_stats_slots(int N) {
    if (N <= 0 || N % 64 != 0) return 0;            // ROW_STATS needs whole tiles
    return N >> stat_shift_for(N);
}

extern "C" size_t rajni_gemm_workspace_bytes(void) { return sk_workspace_bytes(); }

// Host-side query (no launch): how many tiles a hot-epilogue GEMM of this shape would split along K given a workspace,
// and over how many CTA pairs.  0 = no stream-K (tile count already a multiple of the pairs, K too short, or no gain).
extern "C" int rajni_gemm_stream_k_plan(int M, int N, int K, int flags, int* sk_pairs) {
    if (sk_pairs) *sk_pairs = 0;
    if (M <= BM || N <= 0 || N % 256 != 0 || K <= 0 || (flags & RAJNI_EPI_OUT_F32)) return 0;
    // the entry point's own tile choice; only the 256-wide CTA-pair tile with a hot epilogue splits
    const bool exact = (flags & (RAJNI_EPI_LN_FOLD | RAJNI_EPI_ROW_STATS)) != 0;
    const bool force = (flags & RAJNI_HINT_STREAM_K) != 0;
    const int bn = pick_bn(N, M, K, exact, (flags & RAJNI_EPI_ROW_STATS) && stat_shift_for(N) == 6, true, force);
    if (bn != -256 && bn != 256) return 0;
    int sp = 0;
    const int tiles = ((M + 2 * BM - 1) / (2 * BM)) * (N / 256);
    const int R = sk_decide(tiles, num_sms() / 2, (K + BK - 1) / BK, force, &sp);
    if (sk_pairs && R > 0) *sk_pairs = sp;
    return R;
}

extern "C" int rajni_gemm_bf16_ex(const rajni_gemm_args* a, void* stream) {
    RAJNI_REQUIRE(a != nullptr, RAJNI_EINVAL, "rajni_gemm_bf16_ex: null argument block");
    const int M = a->M, N = a->N, K = a->K, flags = a->flags;
    RAJNI_REQUIRE(a->A && a->W && a->D, RAJNI_EINVAL, "rajni_gemm_bf16: null pointer");
    RAJNI_REQUIRE(M > 0 && N > 0 && K > 0 && K % 8 == 0, RAJNI_EINVAL, "rajni_gemm_bf16: M=%d N=%d K=%d (K must be a multiple of 8)", M, N, K);
    RAJNI_REQUIRE(!(flags & RAJNI_EPI_BIAS) || a->bias, RAJNI_EINVAL, "rajni_gemm_bf16: bias flag without bias");
    RAJNI_REQUIRE(!(flags & RAJNI_EPI_RESIDUAL) || a->residual, RAJNI_EINVAL, "rajni_gemm_bf16: residual flag without residual");
    RAJNI_REQUIRE(a->ldd >= N && a->ldd % 4 == 0 && (!(flags & RAJNI_EPI_RESIDUAL) || a->ldres % 4 == 0), RAJNI_EINVAL,
                  "rajni_gemm_bf16: ldd=%lld ldres=%lld must be multiples of 4 and ldd >= N", a->ldd, a->ldres);
    if (flags & RAJNI_EPI_LN_FOLD)
        RAJNI_REQUIRE(a->ln_stats && a->ln_wsum && a->ln_slots > 0 && a->ln_stats_ld >= M && (flags & RAJNI_EPI_BIAS) && !(flags & RAJNI_EPI_OUT_F32),
                      RAJNI_EINVAL, "rajni_gemm_bf16: LN_FOLD needs ln_stats, ln_wsum, ln_slots > 0, ln_stats_ld >= M, a bias and bf16 output");
    if (flags & RAJNI_EPI_ROW_STATS)
        RAJNI_REQUIRE(a->row_stats && a->row_stats_ld > 0 && (flags & RAJNI_EPI_RESIDUAL) && !(flags & RAJNI_EPI_OUT_F32), RAJNI_EINVAL,
                      "rajni_gemm_bf16: ROW_STATS needs row_stats, row_stats_ld and the bias+residual bf16 epilogue");
    GemmParams p{};
    p.bias = a->bias; p.D = a->D;
    p.residual = static_cast<const __nv_bfloat16*>(a->residual);
    p.res_row_map = a->res_row_map; p.out_row_map = a->out_row_map;
    p.ldd = a->ldd; p.ldres = a->ldres;
    p.M = M; p.N = N; p.K = K; p.flags = flags & ~RAJNI_HINT_REVERSE_M;
    p.reverse_m = (flags & RAJNI_HINT_REVERSE_M) != 0;
    p.ln_stats = reinterpret_cast<const float2*>(a->ln_stats);
    p.ln_wsum = a->ln_wsum;
    p.ln_stats_ld = a->ln_stats_ld;
    p.ln_slots = a->ln_slots;
    p.ln_inv_k = 1.0f / (float)K;
    p.ln_eps = a->ln_eps;
    p.row_stats = (flags & RAJNI_EPI_ROW_STATS) ? reinterpret_cast<float2*>(a->row_stats) : nullptr;
    p.row_stats_ld = a->row_stats_ld;
    p.stat_shift = stat_shift_for(N);
    const bool exact = (flags & (RAJNI_EPI_LN_FOLD | RAJNI_EPI_ROW_STATS)) != 0;
    RAJNI_REQUIRE(!exact || N % 64 == 0, RAJNI_EINVAL, "rajni_gemm_bf16: LN_FOLD / ROW_STATS need N %% 64 == 0 (N=%d)", N);
    // (a producer of 64-column statistics slots cannot use the 192-wide tile)
    int bn = pick_bn(N, M, K, exact, (flags & RAJNI_EPI_ROW_STATS) && stat_shift_for(N) == 6,
                     a->workspace != nullptr && (size_t)a->workspace_bytes >= sk_workspace_bytes(), (flags & RAJNI_HINT_STREAM_K) != 0);   // < 0: exact CTA-pair tile of width -bn
    auto s = static_cast<cudaStream_t>(stream);
    // wide problems run as CTA pairs (256 x 256 tiles); narrow ones keep single-CTA tiles
    static const bool force_cg1 = getenv("RAJNI_GEMM_CG1") != nullptr;     // debugging aid
    if (bn < 0 && force_cg1) bn = (-bn == 192) ? 64 : -bn;
    switch (bn) {
        case -256: return launch_gemm<256, 2>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
        case -192: return launch_gemm<192, 2>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
        case -128: return launch_gemm<128, 2>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
        case 256: return (M > BM && !force_cg1) ? launch_gemm<256, 2>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s) : launch_gemm<256, 1>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
        case 128: return launch_gemm<128, 1>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
        default: return launch_gemm<64, 1>(a->A, a->W, p, a->workspace, (size_t)a->workspace_bytes, s);
    }
}

extern "C" int rajni_gemm_bf16(const void* A, const void* W, const float* bias, void* D,
                               int M, int N, int K, int flags,
                               const void* residual, long long ldres, const int32_t* res_row_map,
                               long long ldd, const int32_t* out_row_map, void* stream) {
    RAJNI_REQUIRE(!(flags & (RAJNI_EPI_LN_FOLD | RAJNI_EPI_ROW_STATS)), RAJNI_EINVAL,
                  "rajni_gemm_bf16: LN_FOLD / ROW_STATS need rajni_gemm_bf16_ex");
    rajni_gemm_args a{};
    a.A = A; a.W = W; a.bias = bias; a.D = D;
    a.M = M; a.N = N; a.K = K; a.flags = flags;
    a.residual = residual; a.ldres = ldres; a.res_row_map = res_row_map;
    a.ldd = ldd; a.out_row_map = out_row_map;
    return rajni_gemm_bf16_ex(&a, stream);
}
