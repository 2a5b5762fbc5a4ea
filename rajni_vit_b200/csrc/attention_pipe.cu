// Pipelined tcgen05 attention over kept tokens (Np <= 224 keys, head dim 64): every 224-px configuration.
//
//   out[b, i, h*64:(h+1)*64] = softmax_j( q_i . k_j * scale ) v_j        attention.py:45-54
//   token j of image b is read from global qkv row row_map[b*Np + j]     attention.py:42-43 (gather fused)
//
// One CTA per SM walks a sequence of 128-query TILES (an (image, head) item has one tile when Np <= 128, else two that
// share K/V).  Each stage has its own warps and the score tile is multi-buffered in TMEM:
//
//   warps 0-7  EXP     thread = (query row, half of the key columns).  The thread pulls its WHOLE half row of S (<= 112
//                      fp32) out of TMEM with one wait - a tcgen05.ld costs ~150 cycles alone and ~450 next to the tensor
//                      pipe, whatever its size, so S is read exactly once and in one go (profiles/r2_pipe_probe.txt) - takes
//                      the row maximum from registers, swaps it with the other half's through shared memory (one 64-thread
//                      named barrier), then p = exp2(s*scale*log2e - max) -> bf16 P back into TMEM over S, partial row sum
//                      to shared memory.  Exact two-pass softmax, like the reference.  (160 registers: setmaxnreg.)
//   warps 8-11 EPILOGUE thread = query row: O(g) = P V out of TMEM, times 1/rowsum, bf16, swizzled shared memory, one TMA
//                      store per warp (3-d map clipped at the image's Np rows).
//   warp 12    MMA     one lane issues S(g) = Q K^T (SS, 4 k-steps) and O(g) = P V (TS: A = P from TMEM, V MN-major)
//   warps 13-15 LOAD   dense call: one thread, three TMA boxes per item (3-d map: rows past the image are ZERO-filled, so
//                      one image's Inf/NaN can never reach another's output); gathered call: cp.async row gather by row_map
//
// TMEM (512 columns): nbuf score buffers of s_stride columns (2 at Np_pad 208 ... 3 at Np_pad <= 128), then one or two
// 64-column O buffers: S(g+1) is computed while the exp warps work on tile g and P(g-1) V runs.
//
// One-tile items of at most 112 keys run the exp warps in FULL-ROW mode (ap_exp_full): a thread holds its whole row of S, so
// no maximum is exchanged, and warps 0-3 take the even tiles, warps 4-7 the odd ones - the two exp warps of a scheduler are
// half a period apart, one's TMEM wait / maximum / P store under the other's exponentials (dense 87 tokens: 30.8 us against
// 43.5 us for attention_tc; gathered calls stay with attention_tc's seven loader warps).
#include <cuda.h>

#include <type_traits>

#include "common.cuh"

namespace rajni {

constexpr int kApHelpWarp0 = 8;
#ifndef AP_MMA_WARP
#define AP_MMA_WARP 15
#endif
// The MMA issuer sits on scheduler 3 (warp id % 4): its neighbours there are the exp warps of TMEM lanes 96..127, which have
// no rows at all in the second tile of a 129..224-token item - an issuer next to busy exp warps gets so few issue slots that
// queueing one P V takes 2200 cycles instead of 1300 (profiles/r2_attention_pipe.md).
constexpr int kApMmaWarp = AP_MMA_WARP;
constexpr int kApLoaderWarp0 = 12;                                             // three loader warps: 12..14 (or 13..15)
constexpr int kApWg3Warp0 = 12;
constexpr int kApLoaderThreads = 96;
constexpr int kApLoaderGroups = kApLoaderThreads / 8;                          // 8 lanes move one token's 128-byte head slice
constexpr int kApSweeps = (224 + kApLoaderGroups - 1) / kApLoaderGroups;       // sweeps of the groups over <= 224 token rows
constexpr int kApThreads = 512;
constexpr int kApMaxStages = 4;
constexpr int kApMaxBufs = 4;
constexpr int kApSumSlots = 8;
#ifndef AP_POLY_EVERY
#define AP_POLY_EVERY 0
#endif
constexpr int kApPolyEvery = AP_POLY_EVERY;               // one exponential in this many is a polynomial on the FMA pipe (0: all on MUFU)
constexpr int kApOutStage = 4 * 4096;                                          // 32 rows x 128 B per helper warp
constexpr int kApAuxBytes = 2 * 2 * 128 * 4 + kApSumSlots * 2 * 128 * 4;       // half-row maxima (2 parities), partial row sums
constexpr int kApBarBytes = 320;
constexpr int kApSmemBudget = 227 * 1024 - 1024 - kApOutStage - kApAuxBytes - kApBarBytes;

#ifdef RAJNI_ATTN_TRACE
__device__ int g_ap_dbg;
__device__ long long g_ap_trace[64 * 16];
#define AP_TRACE(g, slot) do { if (blockIdx.x == 0 && (g) < 64) g_ap_trace[(g) * 16 + (slot)] = clock64(); } while (0)
#else
#define AP_TRACE(g, slot) do { } while (0)
#endif

struct AttnPipeParams {
    const __nv_bfloat16* qkv;
    const int32_t* row_map;
    int N_src, Np, Np_pad, C, H, BH, tpi;      // tpi = 128-row tiles per (image, head) item
    int nbuf, s_stride, n_obuf, o_col;         // score buffer b at column b*s_stride; O buffer ob at o_col + 64*ob
    int split;                                  // key columns [0, split) -> exp warps 0-3, [split, Np_pad) -> warps 4-7
    int fullrow;                                // one-tile items of <= 112 keys: a thread takes its WHOLE row, warps 0-3 the even tiles, 4-7 the odd ones
    int plane_bytes, stages, reverse;
    int dbg;                                    // experiments (tools/probes, RAJNI_ATTN_TRACE builds only): skip parts of the work
    float scale_log2;
};

__device__ __forceinline__ void ap_bar_sync(int id, int threads) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(threads) : "memory");
}
// Register re-partitioning between warpgroups (4 consecutive warps): the load/MMA and the epilogue warpgroups give registers
// back, the exp warpgroups (a half row of S = 112 registers) take them.  8*160 + 4*112 + 4*80 = 2048 = 64 K / 32.
template <int N> __device__ __forceinline__ void ap_reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" :: "n"(N)); }
template <int N> __device__ __forceinline__ void ap_reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(N)); }

// warp-uniform non-blocking barrier probe (lane 0 tests, everybody gets its answer)
__device__ __forceinline__ bool ap_test_uniform(uint64_t* bar, uint32_t parity) {
    return __shfl_sync(0xffffffffu, (int)mbar_test(bar, parity), 0) != 0;
}

__device__ __forceinline__ int ap_item(const AttnPipeParams& p, int n) {
    const int it = (int)blockIdx.x + n * (int)gridDim.x;
    return p.reverse ? p.BH - 1 - it : it;
}

// position of a tile in the CTA's sequence, kept with counters instead of divisions
struct ApCursor {
    int g = 0, n = 0, j = 0;          // tile index, item index, tile inside the item
    int buf = 0, stage = 0;
    uint32_t buf_ph = 0, stage_ph = 0;
    __device__ __forceinline__ void advance(const AttnPipeParams& p) {
        ++g;
        if (++buf == p.nbuf) { buf = 0; buf_ph ^= 1; }
        if (++j == p.tpi) {
            j = 0;
            ++n;
            if (++stage == p.stages) { stage = 0; stage_ph ^= 1; }
        }
    }
};

// 2^x on the FMA/ALU pipes (x >= -125 after the clamp): round x to the nearest integer with the 1.5*2^23 trick, a cubic
// for 2^f on f in [-0.5, 0.5] (relative error 2.2e-4, a twentieth of a bf16 ulp), the integer added into the exponent field.
// One exponential in kApPolyEvery goes this way: MUFU.EX2 (16 results/clk/SM) is what bounds the exp warps, the FMA pipe idles.
__device__ __forceinline__ float ap_ex2_poly(float x) {
    x = fmaxf(x, -125.f);
    const float t = x + 12582912.f;
    const float f = x - (t - 12582912.f);
    float q = fmaf(0.05286743f, f, 0.24215189f);
    q = fmaf(q, f, 0.69358677f);
    q = fmaf(q, f, 0.99996275f);
    return __uint_as_float(__float_as_uint(q) + (__float_as_uint(t) << 23));
}

// One exp-warp thread's share of a tile: the half row [cb, cb + 32*N32 + 16*HAS16) of S (TMEM row `sb`) -> P at `pcol`.
// Straight-line for a given (N32, HAS16): no branch between the 16-column groups, so MUFU.EX2 never drains.
//   s[0..95] = the 32-column pieces, s[96..111] = the 16-column piece.  The thread holds its WHOLE half row before the row
//   maximum is taken: one wait for all loads (a tcgen05.ld costs ~150 cycles alone whatever its size), `taken_bar` tells
//   the MMA issuer that S has left TMEM.  Columns >= Np (fewer than 16, all in the half's last 16 columns) are set to -inf
//   up front, so neither the maximum nor exp2 needs a mask: exp2(-inf) = 0.  P pair k overwrites register k, consumed by
//   then; P goes back with at most three stores (a tcgen05.st holds the warp ~100 cycles whatever its size).
//   drop16: the half's first 16 columns are also the other half's last (both halves run the same width, see the kernel);
//   they are written (identical values) but not summed.
// Returns the half row's sum of p.
template <int N32, int HAS16>
__device__ __forceinline__ float ap_exp_half(uint32_t sb, int cb, uint32_t pcol, int Np, float sl2, float* pm_mine, const float* pm_other,
                                             int bar_id, int bar_n, uint64_t* taken_bar, bool drop16, int lane, bool trace_lane, int g) {
    constexpr int NCOL = 32 * N32 + 16 * HAS16;
    constexpr int LAST = HAS16 ? 96 : 32 * N32 - 16;                          // registers of the half's last 16 columns
    constexpr int W16 = 16 * N32;                                             // P pairs of the 16-column piece go to s[W16..]
    uint32_t s[112];
#pragma unroll
    for (int i = 0; i < N32; ++i) tmem_ld32(sb + cb + 32 * i, *reinterpret_cast<uint32_t(*)[32]>(&s[32 * i]));
    if (HAS16) tmem_ld16(sb + cb + 32 * N32, *reinterpret_cast<uint32_t(*)[16]>(&s[96]));
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(taken_bar);
    if (trace_lane) AP_TRACE(g, 4);
    if (cb + NCOL > Np) {
#pragma unroll
        for (int i = 0; i < 16; ++i) if (cb + NCOL - 16 + i >= Np) s[LAST + i] = 0xff800000u;      // -inf
    }
    // ---- row maximum of this half (four independent chains), then of the row (the other half's through shared memory)
    float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int i = 0; i < 32 * N32; i += 2) m4[(i >> 1) & 3] = fmax3(m4[(i >> 1) & 3], __uint_as_float(s[i]), __uint_as_float(s[i + 1]));
    if (HAS16) {
#pragma unroll
        for (int i = 0; i < 16; i += 2) m4[(i >> 1) & 3] = fmax3(m4[(i >> 1) & 3], __uint_as_float(s[96 + i]), __uint_as_float(s[97 + i]));
    }
    const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
    *pm_mine = mx;
    ap_bar_sync(bar_id, bar_n);                                               // the two warps that share these 32 rows
    const float mb = fmaxf(mx, *pm_other) * sl2;
    if (trace_lane) AP_TRACE(g, 5);
#ifdef RAJNI_ATTN_TRACE
    if (g_ap_dbg & 2) return mb;
#endif
    float sum0 = 0.f, sum1 = 0.f;
    // p = exp2(s * scale * log2e - max) for registers R0..R0+N -> bf16 pairs at W0..; column c of the row takes the
    // polynomial when c % kApPolyEvery == kApPolyEvery - 1 (cb and R0 are multiples of 16, so the register index decides)
    auto exp_run = [&](auto r0_c, auto w0_c, auto n_c) {
        constexpr int R0 = decltype(r0_c)::value, W0 = decltype(w0_c)::value, N = decltype(n_c)::value;
#pragma unroll
        for (int j = 0; j < N; j += 2) {
            const float x0 = fmaf(__uint_as_float(s[R0 + j]), sl2, -mb), x1 = fmaf(__uint_as_float(s[R0 + j + 1]), sl2, -mb);
            const float e0 = ex2_approx(x0);
            const float e1 = (kApPolyEvery > 0 && (j + 1) % (kApPolyEvery > 0 ? kApPolyEvery : 1) == kApPolyEvery - 1) ? ap_ex2_poly(x1) : ex2_approx(x1);
            sum0 += e0;
            sum1 += e1;
            s[W0 + (j >> 1)] = float2_to_bf16x2(e0, e1);
        }
    };
    using std::integral_constant;
    if (N32 > 0) {
        exp_run(integral_constant<int, 0>{}, integral_constant<int, 0>{}, integral_constant<int, 16>{});
        if (drop16) { sum0 = 0.f; sum1 = 0.f; }
        exp_run(integral_constant<int, 16>{}, integral_constant<int, 8>{}, integral_constant<int, 32 * N32 - 16>{});
    }
    if (HAS16) {
        exp_run(integral_constant<int, 96>{}, integral_constant<int, W16>{}, integral_constant<int, 16>{});
        if (N32 == 0 && drop16) { sum0 = 0.f; sum1 = 0.f; }
    }
    if (trace_lane) AP_TRACE(g, 10);
    // P pairs are contiguous in s[0 .. NCOL/2): 32 + 16 + 8 columns at most
    if (NCOL >= 64) tmem_st32(pcol, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
    if ((NCOL / 2) & 16) tmem_st16(pcol + ((NCOL / 2) & 32), *reinterpret_cast<uint32_t(*)[16]>(&s[(NCOL / 2) & 32]));
    if ((NCOL / 2) & 8) tmem_st8(pcol + ((NCOL / 2) & 48), *reinterpret_cast<uint32_t(*)[8]>(&s[(NCOL / 2) & 48]));
    return sum0 + sum1;
}

// Full-row variant for one-tile items of at most 112 keys (K16 = Np_pad / 16): the thread holds its whole row of S, so
// there is no second half to exchange a maximum with, and the two exp warps of a scheduler work on DIFFERENT tiles (even /
// odd): one warp's TMEM wait, maximum and P store run under the other's exponentials instead of both marching in step.
// The row sum is still taken in two parts, [0, SPLIT) and [SPLIT, NCOL) with SPLIT as in the two-half scheme, each with
// its even / odd column chains, so the result has the same bits as ap_exp_half's (and attention_tc's).
template <int K16>
__device__ __forceinline__ void ap_exp_full(uint32_t sb, uint32_t pcol, int Np, float sl2, uint64_t* taken_bar, int lane,
                                            float& sum_a, float& sum_b) {
    constexpr int NCOL = 16 * K16, N32 = NCOL / 32, HAS16 = K16 & 1;
    constexpr int SPLIT = ((NCOL / 2) + 15) & ~15;
    uint32_t s[NCOL];
#pragma unroll
    for (int i = 0; i < N32; ++i) tmem_ld32(sb + 32 * i, *reinterpret_cast<uint32_t(*)[32]>(&s[32 * i]));
    if (HAS16) tmem_ld16(sb + 32 * N32, *reinterpret_cast<uint32_t(*)[16]>(&s[32 * N32]));
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(taken_bar);
    if (NCOL > Np) {
#pragma unroll
        for (int i = 0; i < 16; ++i) if (NCOL - 16 + i >= Np) s[NCOL - 16 + i] = 0xff800000u;      // -inf
    }
    float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int i = 0; i < NCOL; i += 2) m4[(i >> 1) & 3] = fmax3(m4[(i >> 1) & 3], __uint_as_float(s[i]), __uint_as_float(s[i + 1]));
    const float mb = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * sl2;
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int j = 0; j < NCOL; j += 2) {
        if (j == SPLIT) { sum_a = sum0 + sum1; sum0 = 0.f; sum1 = 0.f; }
        const float e0 = ex2_approx(fmaf(__uint_as_float(s[j]), sl2, -mb)), e1 = ex2_approx(fmaf(__uint_as_float(s[j + 1]), sl2, -mb));
        sum0 += e0;
        sum1 += e1;
        s[j >> 1] = float2_to_bf16x2(e0, e1);
    }
    if (SPLIT < NCOL) sum_b = sum0 + sum1;
    else { sum_a = sum0 + sum1; sum_b = 0.f; }
    constexpr int W = NCOL / 2;                                               // 32-bit words of P
    if (W & 32) tmem_st32(pcol, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
    if (W & 16) tmem_st16(pcol + (W & 32), *reinterpret_cast<uint32_t(*)[16]>(&s[W & 32]));
    if (W & 8) tmem_st8(pcol + (W & 48), *reinterpret_cast<uint32_t(*)[8]>(&s[W & 48]));
}

__global__ void __launch_bounds__(kApThreads, 1)
attention_pipe_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_out, const AttnPipeParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const int stage_bytes = 3 * p.plane_bytes;
    // [stages][Q|K|V planes] [output staging: 4 warps x 4 KB] [half-row maxima][partial row sums][barriers]
    // (a tile's Q operand is read as 128 rows from row 0 / 128 of the Q plane: the over-read lands in the stage's K plane)
    const uint32_t out_stage0 = smem_base + p.stages * stage_bytes;
    float* pmax = reinterpret_cast<float*>(smem_gen + p.stages * stage_bytes + kApOutStage);     // [2 parities][2 halves][128] half-row maxima
    float* sums = pmax + 2 * 2 * 128;                                                              // [8 slots][2 halves][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sums + kApSumSlots * 2 * 128);
    uint64_t* qk_full = bars;                        // [4] loader -> MMA
    uint64_t* v_full = bars + 4;                     // [4] loader -> MMA
    uint64_t* stage_empty = bars + 8;                // [4] MMA -> loader (tcgen05.commit after the item's last P V): the V plane is free
    uint64_t* s_full = bars + 12;                    // [4 bufs] MMA -> exp warps (S ready)
    uint64_t* s_taken = bars + 16;                   // [4 bufs] exp warps -> MMA (S is in registers: the tensor pipe may start P V)
    uint64_t* p_full = bars + 20;                    // [4 bufs] exp warps -> MMA (P in TMEM)
    uint64_t* o_full = bars + 24;                    // [2] MMA -> helpers
    uint64_t* o_empty = bars + 26;                   // [2] helpers -> MMA (O read out)
    uint64_t* qk_empty = bars + 28;                  // [4] MMA -> loader (commit after the item's last S): the Q and K planes are free -
                                                     //     a tile time or two before the V plane, and Q/K are 2/3 of the next item's bytes
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 32);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == kApMmaWarp) {
        tmem_alloc(tmem_slot, 512);
        if (lane == 0) {
            for (int i = 0; i < kApMaxStages; ++i) {
                // gathered: one cp.async-completion arrival per loader thread; dense: one arrival + TMA transaction bytes
                mbar_init(&qk_full[i], p.row_map ? kApLoaderThreads : 1);
                mbar_init(&v_full[i], p.row_map ? kApLoaderThreads : 1);
                mbar_init(&stage_empty[i], 1);
                mbar_init(&qk_empty[i], 1);
            }
            for (int i = 0; i < kApMaxBufs; ++i) {
                mbar_init(&s_full[i], 1);
                mbar_init(&p_full[i], p.fullrow ? 4 : 8);            // one arrival per exp warp (of the tile's parity)
                mbar_init(&s_taken[i], p.fullrow ? 4 : 8);
            }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&o_full[i], 1);
                mbar_init(&o_empty[i], 4);
            }
            mbar_fence_init();
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch();
    griddep_wait();
    const int n_mine = (p.BH - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;     // items of this CTA
    const int G = n_mine * p.tpi;                                                          // tiles of this CTA
    const int Np = p.Np, Np_pad = p.Np_pad;

    if (warp >= kApWg3Warp0) {
      // warpgroup 3 (MMA issuer + loaders) hands registers back: ONE setmaxnreg site for its four warps
      ap_reg_dec<80>();
      const int lw = warp - kApWg3Warp0 - (warp > kApMmaWarp ? 1 : 0);          // loader warp index 0..2 (the MMA warp aside)
      if (warp != kApMmaWarp && p.row_map == nullptr) {
        // ================= dense loader: one TMA box per plane; rows past the image's N_src are zero-filled =================
        if (lw == 0 && lane == 0) {
            tma_prefetch_desc(&tmap_qkv);
            const uint32_t plane_tx = (uint32_t)Np_pad * 128u;
            int stage = 0;
            uint32_t phase = 0;
            for (int n = 0; n < n_mine; ++n) {
                const int item = ap_item(p, n);
                const int b = item / p.H, h = item - b * p.H;
                uint8_t* sq = smem_gen + stage * stage_bytes;
                mbar_wait(&qk_empty[stage], phase ^ 1);
                mbar_expect_tx(&qk_full[stage], 2u * plane_tx);
                tma_load_3d(sq, &tmap_qkv, &qk_full[stage], h * 64, 0, b);
                tma_load_3d(sq + p.plane_bytes, &tmap_qkv, &qk_full[stage], p.C + h * 64, 0, b);
                mbar_wait(&stage_empty[stage], phase ^ 1);
                mbar_expect_tx(&v_full[stage], plane_tx);
                tma_load_3d(sq + 2 * p.plane_bytes, &tmap_qkv, &v_full[stage], 2 * p.C + h * 64, 0, b);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
      } else if (warp != kApMmaWarp) {
        // ================= gather loaders: 8 lanes move one token's 128-byte head slice per plane (cp.async) =================
        const int lt = lw * 32 + lane;
        const int grp = lt >> 3, chunk = lt & 7;
        const long long C3 = 3LL * p.C;
        int stage = 0;
        uint32_t phase = 0;
        for (int n = 0; n < n_mine; ++n) {
            const int item = ap_item(p, n);
            const int b = item / p.H, h = item - b * p.H;
            // global row of every token this lane group moves: the index loads are issued together, before the wait
            int grow[kApSweeps];
#pragma unroll
            for (int i = 0; i < kApSweeps; ++i) {
                const int j = grp + i * kApLoaderGroups;
                grow[i] = j < Np ? __ldg(p.row_map + (long long)b * Np + j) : -1;
            }
            const uint32_t sq = smem_base + stage * stage_bytes, sk = sq + p.plane_bytes, sv = sk + p.plane_bytes;
            const __nv_bfloat16* base = p.qkv + h * 64 + chunk * 8;
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {                    // pass 0: Q and K (what S needs), pass 1: V
                mbar_wait(pass == 0 ? &qk_empty[stage] : &stage_empty[stage], phase ^ 1);
#pragma unroll
                for (int i = 0; i < kApSweeps; ++i) {
                    const int j = grp + i * kApLoaderGroups;
                    if (j >= Np_pad) continue;
                    const bool ok = grow[i] >= 0;
                    const __nv_bfloat16* src = base + (long long)(ok ? grow[i] : 0) * C3;
                    const uint32_t off = j * 128 + ((chunk ^ (j & 7)) << 4);
                    if (pass == 0) {
                        if (ok) {                                     // rows past Np: dead query rows / masked key columns
                            cp_async16(sq + off, src, 16);
                            cp_async16(sk + off, src + p.C, 16);
                        }
                    } else {
                        cp_async16(sv + off, src + 2 * p.C, ok ? 16 : 0);      // zero-filled: 0 * V must stay 0
                    }
                }
                cp_async_arrive_noinc(pass == 0 ? &qk_full[stage] : &v_full[stage]);
            }
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      } else if (warp == kApMmaWarp) {
        // ================= MMA issuer =================
        // The tensor pipe executes in issue order:  ... PV(g-1) S(g+1) PV(g) S(g+2) ...  S(g) may be issued once
        // PV(g-nbuf), which read P out of the same buffer, is queued; PV(g) once P(g) is complete and its O buffer is free.
        if (lane == 0) {
            const uint32_t idesc_s = umma_idesc_bf16(128, Np_pad, 0, 0);
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);          // B = V is MN-major
            const int nk = Np_pad / 16, nk0 = p.split / 16;
            // P of key columns [0, split) sits at the buffer's start; the second half's P (keys Np_pad - split ...) starts at
            // column `split`, so P of key `split` is (2 split - Np_pad) / 2 columns further in
            const uint32_t p2 = (uint32_t)(p.split + ((2 * p.split - Np_pad) >> 1));
            const uint64_t qd0 = umma_desc_sw128(smem_base, 16, 1024);
            const uint64_t kd0 = umma_desc_sw128(smem_base + p.plane_bytes, 16, 1024);
            const uint64_t vd0 = umma_desc_sw128(smem_base + 2 * p.plane_bytes, 16, 1024);
            ApCursor s, v;
            int ob = 0;
            uint32_t o_ph0 = 1, o_ph1 = 1;                                    // parity of the o_empty phase the next PV waits for
            // (a fresh barrier passes a wait on parity 1: the first use of each O buffer does not wait)
            auto issue_s = [&]() {
                mbar_wait(&qk_full[s.stage], s.stage_ph);
                tc_fence_after();
                AP_TRACE(s.g, 0);
                const uint64_t qd = qd0 + (uint64_t)((s.stage * stage_bytes + s.j * (128 * 128)) >> 4);
                const uint64_t kd = kd0 + (uint64_t)((s.stage * stage_bytes) >> 4);
                const uint32_t d = tmem_base + s.buf * p.s_stride;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_bf16(d, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc_s, k != 0);
                umma_commit(&s_full[s.buf]);
                if (s.j == p.tpi - 1) umma_commit(&qk_empty[s.stage]);         // the item's last S: its Q and K planes may be refilled
                AP_TRACE(s.g, 1);
                s.advance(p);
            };
            // Fixed issue order with BLOCKING waits (a polling issuer takes issue slots from the exp warps of its scheduler):
            //   S(0) .. S(nbuf-1),  then  PV(g), S(g+nbuf)  for every tile g
            for (int i = 0; i < p.nbuf && s.g < G; ++i) issue_s();
            for (; v.g < G; v.advance(p)) {
                mbar_wait(&p_full[v.buf], v.buf_ph);
                // The exp warps read S(v+1) right after P(v); a tcgen05.ld next to the P V products (A operand from TMEM)
                // takes ~1000 cycles instead of ~300, and slows the products too (profiles/r2_attention_pipe.md), so the
                // products wait the few hundred cycles until S(v+1) is in registers and then run under the exponentials.
                if (v.g + 1 < G) {
                    int nb = v.buf + 1;
                    uint32_t nph = v.buf_ph;
                    if (nb == p.nbuf) { nb = 0; nph ^= 1; }
                    mbar_wait(&s_taken[nb], nph);
                }
                mbar_wait(&v_full[v.stage], v.stage_ph);
                mbar_wait(&o_empty[ob], ob ? o_ph1 : o_ph0);
                tc_fence_after();
                AP_TRACE(v.g, 2);
                const uint64_t vd = vd0 + (uint64_t)((v.stage * stage_bytes) >> 4);
                const uint32_t pb = tmem_base + v.buf * p.s_stride;
                const uint32_t d = tmem_base + p.o_col + ob * 64;
                uint64_t vdk = vd;
                for (int k = 0; k < nk0; ++k, vdk += (2048 >> 4)) umma_bf16_ts(d, pb + k * 8, vdk, idesc_o, k != 0);
                for (int k = 0; k < nk - nk0; ++k, vdk += (2048 >> 4)) umma_bf16_ts(d, pb + p2 + k * 8, vdk, idesc_o, 1);
                AP_TRACE(v.g, 12);
                umma_commit(&o_full[ob]);
                if (v.j == p.tpi - 1) umma_commit(&stage_empty[v.stage]);     // the item's last product: the stage may be refilled
                AP_TRACE(v.g, 3);
                if (ob) o_ph1 ^= 1; else o_ph0 ^= 1;
                if (++ob == p.n_obuf) ob = 0;
                if (s.g < G) issue_s();                                       // into the buffer this PV has just released
            }
        }
      }
    } else if (warp >= kApHelpWarp0) {
        // ================= epilogue warps: O(g) = P V out of TMEM, normalise, store =================
        ap_reg_dec<112>();
        const int hq = warp - kApHelpWarp0;                                  // TMEM lane quadrant
        const int row = hq * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(hq * 32) << 16);
        const uint32_t s_out = out_stage0 + hq * 4096;
        ApCursor e;
        int ob = 0, slot = 0;
        uint32_t o_ph0 = 0, o_ph1 = 0;
        for (; e.g < G; e.advance(p)) {
            mbar_wait(&o_full[ob], ob ? o_ph1 : o_ph0);
            tc_fence_after();
            if (hq == 0 && lane == 0) AP_TRACE(e.g, 6);
#ifdef RAJNI_ATTN_TRACE
            const bool live = e.j * 128 + hq * 32 < Np && !(p.dbg & 4);
#else
            const bool live = e.j * 128 + hq * 32 < Np;
#endif
            uint32_t o0[32], o1[32];
            if (live) {
                const uint32_t ocol = lane_base + p.o_col + ob * 64;
                tmem_ld32(ocol, o0);
                tmem_ld32(ocol + 32, o1);
                tmem_ld_wait();
                tc_fence_before();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&o_empty[ob]);
            if (live) {
                const float inv = 1.f / (sums[(slot * 2 + 0) * 128 + row] + sums[(slot * 2 + 1) * 128 + row]);
                if (lane == 0) bulk_wait_group_read<0>();                 // the previous store has read the staging buffer
                __syncwarp();
                const uint32_t srow = s_out + lane * 128;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint32_t (&src)[32] = c < 4 ? o0 : o1;
                    const int j = (c & 3) * 8;
                    sts128(srow + ((c ^ (lane & 7)) << 4),
                              float2_to_bf16x2(__uint_as_float(src[j]) * inv, __uint_as_float(src[j + 1]) * inv),
                              float2_to_bf16x2(__uint_as_float(src[j + 2]) * inv, __uint_as_float(src[j + 3]) * inv),
                              float2_to_bf16x2(__uint_as_float(src[j + 4]) * inv, __uint_as_float(src[j + 5]) * inv),
                              float2_to_bf16x2(__uint_as_float(src[j + 6]) * inv, __uint_as_float(src[j + 7]) * inv));
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    const int item = ap_item(p, e.n);
                    const int b = item / p.H, h = item - b * p.H;
                    tma_store_3d(&tmap_out, s_out, h * 64, e.j * 128 + hq * 32, b);
                    bulk_commit_group();
                }
            }
            if (hq == 0 && lane == 0) AP_TRACE(e.g, 7);
            if (ob) o_ph1 ^= 1; else o_ph0 ^= 1;
            if (++ob == p.n_obuf) ob = 0;
            if (++slot == kApSumSlots) slot = 0;
        }
        if (lane == 0) bulk_wait_group<0>();                                  // output stores complete before the CTA retires
    } else {
        // ================= exp warps: thread = (query row, half of the key columns) =================
        ap_reg_inc<160>();
        const int q = warp & 3, half = warp >> 2;
        const int row = q * 32 + lane;
        // Both halves run the SAME width (one code path resident in the instruction cache): `split` columns, the second half
        // starting at Np_pad - split; where the two overlap (16 columns) the second half does not count them in its sum.
        // Its P goes to column `split` on, clear of the columns the first half still reads.
        const int cb = half ? Np_pad - p.split : 0;
        const int nch = p.split >> 4;                                         // 16-column groups of a half (1..7)
        const bool drop16 = half && 2 * p.split > Np_pad;
        const bool has_cols = !half || p.split < Np_pad;                      // (a 16-column row has no second half)
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        const float sl2 = p.scale_log2;
        ApCursor c;
        int slot = 0;
        if (p.fullrow) {
            // one-tile items, whole rows: this warp takes the tiles of its parity only (see ap_exp_full)
            const int k16 = Np_pad >> 4;
            for (; c.g < G; c.advance(p)) {
                if ((c.g & 1) == half) {
                    mbar_wait(&s_full[c.buf], c.buf_ph);
                    if (q * 32 < Np) {
                        tc_fence_after();
                        const uint32_t sb = lane_base + c.buf * p.s_stride;
                        float sa = 0.f, sbm = 0.f;
                        switch (k16) {                                        // warp-uniform: one straight-line body per width
                            case 7: ap_exp_full<7>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            case 6: ap_exp_full<6>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            case 5: ap_exp_full<5>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            case 4: ap_exp_full<4>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            case 3: ap_exp_full<3>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            case 2: ap_exp_full<2>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                            default: ap_exp_full<1>(sb, sb, Np, sl2, &s_taken[c.buf], lane, sa, sbm); break;
                        }
                        sums[(slot * 2 + 0) * 128 + row] = sa;
                        sums[(slot * 2 + 1) * 128 + row] = sbm;
                        tmem_st_wait();
                        tc_fence_before();
                    } else {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&s_taken[c.buf]);
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&p_full[c.buf]);
                }
                if (++slot == kApSumSlots) slot = 0;
            }
        } else
        for (; c.g < G; c.advance(p)) {
            mbar_wait(&s_full[c.buf], c.buf_ph);
            if (warp == 0 && lane == 0) AP_TRACE(c.g, 8);
#ifdef RAJNI_ATTN_TRACE
            if (p.dbg & 1) { __syncwarp(); if (lane == 0) { mbar_arrive(&s_taken[c.buf]); mbar_arrive(&p_full[c.buf]); } if (++slot == kApSumSlots) slot = 0; continue; }
#endif
            if (c.j * 128 + q * 32 < Np && has_cols) {
                tc_fence_after();
                const uint32_t sb = lane_base + c.buf * p.s_stride;
                float* pm = pmax + (c.g & 1) * 256;
                float* pm_mine = pm + half * 128 + row;
                const float* pm_other = p.split < Np_pad ? pm + (half ^ 1) * 128 + row : pm_mine;
                const int bar_n = p.split < Np_pad ? 64 : 32;
                const bool tl = warp == 0 && lane == 0;
                float sum;
#define AP_HALF(N32_, H16_) ap_exp_half<N32_, H16_>(sb, cb, sb + (half ? p.split : 0), Np, sl2, pm_mine, pm_other, 1 + q + (bar_n == 32 ? 4 * half : 0), \
                                                    bar_n, &s_taken[c.buf], drop16, lane, tl, c.g)
                switch (nch) {                                                // warp-uniform: one straight-line body per width
                    case 7: sum = AP_HALF(3, 1); break;
                    case 6: sum = AP_HALF(3, 0); break;
                    case 5: sum = AP_HALF(2, 1); break;
                    case 4: sum = AP_HALF(2, 0); break;
                    case 3: sum = AP_HALF(1, 1); break;
                    case 2: sum = AP_HALF(1, 0); break;
                    default: sum = AP_HALF(0, 1); break;
                }
#undef AP_HALF
                sums[(slot * 2 + half) * 128 + row] = sum;
                tmem_st_wait();
                tc_fence_before();
            } else {
                if (c.j * 128 + q * 32 < Np) sums[(slot * 2 + half) * 128 + row] = 0.f;       // live rows, a half without columns
                __syncwarp();
                if (lane == 0) mbar_arrive(&s_taken[c.buf]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[c.buf]);
            if (warp == 0 && lane == 0) AP_TRACE(c.g, 9);
            if (++slot == kApSumSlots) slot = 0;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kApMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// returns 1 if this kernel handled the call, 0 if the shape is outside its range, <0 on error
int launch_attention_pipe(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                          int C, int H, float scale, int reverse, cudaStream_t stream) {
    const int Np_pad = (Np + 15) & ~15;
    if (Np_pad > 224) return 0;
    AttnPipeParams p{};
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.row_map = row_map;
    p.N_src = N_src; p.Np = Np; p.Np_pad = Np_pad; p.C = C; p.H = H;
    p.reverse = reverse;
#ifdef RAJNI_ATTN_TRACE
    p.dbg = getenv("AP_DEBUG") ? atoi(getenv("AP_DEBUG")) : 0;
    cudaMemcpyToSymbol(g_ap_dbg, &p.dbg, sizeof(int));
#endif
    p.BH = B * H;
    p.tpi = Np > 128 ? 2 : 1;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.s_stride = (Np_pad + 31) & ~31;
    p.n_obuf = 2 * p.s_stride + 128 <= 512 ? 2 : 1;
    p.nbuf = (512 - 64 * p.n_obuf) / p.s_stride;
    if (p.nbuf > kApMaxBufs) p.nbuf = kApMaxBufs;
    p.o_col = 512 - 64 * p.n_obuf;
    p.fullrow = (p.tpi == 1 && Np_pad <= 112) ? 1 : 0;
    p.split = p.fullrow ? Np_pad : ((Np_pad / 2) + 15) & ~15;
    p.plane_bytes = (Np_pad * 128 + 1023) & ~1023;
    p.stages = kApSmemBudget / (3 * p.plane_bytes);
    if (p.stages > kApMaxStages) p.stages = kApMaxStages;
    // One-tile items: S(g + nbuf) needs the Q/K of item g + nbuf while P V(g) still holds item g's stage, i.e. nbuf + 1 items in
    // flight.  With as many score buffers as stages the (blocking, fixed-order) issuer would sit out a whole load latency per
    // tile waiting for a stage that P V(g) has yet to release: 96-key items ran 46.6 us with 4 buffers, slower than 112-key ones
    // with 3 (34.5 us).
    if (p.tpi == 1 && p.nbuf > p.stages - 1) p.nbuf = p.stages - 1;
    RAJNI_REQUIRE(p.stages >= 2 && p.nbuf >= 2, RAJNI_EINVAL, "attention_pipe: Np=%d leaves %d stage(s), %d score buffer(s)", Np, p.stages, p.nbuf);
    // the last stage's Q operand of tile 1 is read 128 rows deep from row 128: keep that inside the allocation
    const int smem = p.stages * 3 * p.plane_bytes + kApOutStage + kApAuxBytes + kApBarBytes + 1024;
    CUtensorMap tmap;
    if (row_map) {
        if (int rc = make_tmap_bf16_3d_box(&tmap, out, B, Np, C, 32)) return rc;        // placeholder (unused by the gather loaders)
    } else {
        if (int rc = make_tmap_bf16_3d_ld(&tmap, qkv, B, N_src, 3LL * C, Np_pad)) return rc;
    }
    CUtensorMap tmap_out;
    RAJNI_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15u) == 0, RAJNI_EINVAL, "attention_pipe: out must be 16-byte aligned (TMA store)");
    if (int rc = make_tmap_bf16_3d_box(&tmap_out, out, B, Np, C, 32)) return rc;
    static int smem_granted[kMaxDevices] = {};
    if (int rc = raise_smem_limit("attention_pipe", attention_pipe_kernel, smem, smem_granted)) return rc;
    int grid = p.BH < num_sms() ? p.BH : num_sms();
    static const int cta_cap = getenv("RAJNI_ATTN_MAX_CTAS") ? atoi(getenv("RAJNI_ATTN_MAX_CTAS")) : 0;      // experiments: share the GPU
    if (cta_cap > 0 && grid > cta_cap) grid = cta_cap;
    const int rc = launch_checked("attention_pipe", attention_pipe_kernel, dim3(grid), dim3(kApThreads), (size_t)smem, stream, 1,
                                  tmap, tmap_out, p);
    return rc ? rc : 1;
}

}  // namespace rajni
