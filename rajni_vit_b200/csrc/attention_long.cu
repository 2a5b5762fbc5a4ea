// tcgen05 attention over kept tokens for sequences that do not fit one TMEM score tile (Np > 256, head dim 64):
// the 577-token configuration (deit_base_patch16_384) and its pruned lengths 507 / 446 / 357 / 257.
//
//   out[b, i, h*64:(h+1)*64] = softmax_j( q_i . k_j * scale ) v_j        attention.py:45-54
//   token j of image b is read from global qkv row row_map[b*Np + j]     attention.py:42-43 (gather fused)
//
// Work item = (image, head, 128-query tile); one CTA per SM loops over items (query tile fastest, so the CTAs that
// share a head's K/V run together and re-read them from L2).  Keys are processed in blocks of 224, twice:
//   pass 1:  S_j = Q K_j^T  ->  running row maximum                         (scores only)
//   pass 2:  S_j = Q K_j^T  ->  P_j = exp2((S_j - max) scale log2 e), row sums, P_j written over S_j as bf16
//            O += P_j V_j   (TS MMA: A = P_j from TMEM, B = V_j MN-major from shared memory)
// Recomputing S (4 k-steps) is cheaper than rescaling O in TMEM whenever the maximum moves, and it keeps the softmax
// exactly two-pass like the reference (no online rescale).
// Roles (384 threads):
//   warps 0-7  : softmax + epilogue; each warp owns a 16-row window of the tile through the 16-lane tcgen05.ld/st
//                shapes (register layout = mma accumulator fragment, verified in tools/probes/tmem16_probe.cu)
//   warp 8     : tcgen05.mma issuer (one lane); S_{j+1} is issued before P_j V_j so it overlaps the softmax of block j
//   warps 9-11 : loaders: cp.async row gather of the head's 128-byte Q/K/V slices into 128-byte-swizzled shared memory
// TMEM (512 columns): S buffers at [0,224) and [224,448), O at [448,512).
#include <cuda.h>

#include "common.cuh"

namespace rajni {

constexpr int kAlSoftmaxWarps = 8;
constexpr int kAlMmaWarp = 8;
constexpr int kAlLoaderWarp0 = 9;
constexpr int kAlLoaderThreads = 96;               // 3 warps: 12 warps in all = 3 per scheduler, 168 registers per thread
constexpr int kAlThreads = (kAlSoftmaxWarps + 1) * 32 + kAlLoaderThreads;    // 384
constexpr int kAlKB = 224;                         // keys per block
constexpr int kAlStages = 3;
constexpr int kAlPlane = kAlKB * 128;              // bytes of one K (or V) block
constexpr int kAlStageBytes = 2 * kAlPlane;
constexpr int kAlQBytes = 128 * 128;            // one Q tile; two of them (the next item's Q is prefetched)
constexpr int kAlOCol = 2 * kAlKB;                 // 448
constexpr int kAlSmem = 2 * kAlQBytes + kAlStages * kAlStageBytes + 256 + 1024;

struct AttnLongParams {
    const __nv_bfloat16* qkv;
    const int32_t* row_map;
    __nv_bfloat16* out;
    int N_src, Np, C, H, BH, QT, n_items, nb;      // QT = query tiles per head, nb = key blocks
    int reverse;
    float scale_log2;
};

__global__ void __launch_bounds__(kAlThreads, 1)
attention_long_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_kv, const AttnLongParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t s_q = smem_base, s_ring = smem_base + 2 * kAlQBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_gen + 2 * kAlQBytes + kAlStages * kAlStageBytes);
    uint64_t* full_bar = bars;              // [3] loader warp -> MMA (32 cp.async completions)
    uint64_t* empty_bar = bars + 3;         // [3] MMA -> loaders (tcgen05.commit)
    uint64_t* q_full = bars + 6;            // [2] loader warp -> MMA
    uint64_t* q_empty = bars + 8;           // [2] MMA -> loaders
    uint64_t* s_full = bars + 10;           // [2] MMA -> softmax (S_j ready)
    uint64_t* s_free = bars + 12;           // [2] softmax -> MMA (pass 1: S_j has been read, 256 arrivals)
    uint64_t* p_full = bars + 14;           // [2] softmax -> MMA (pass 2: P_j written, 256 arrivals)
    uint64_t* o_full = bars + 16;           //     MMA -> softmax
    uint64_t* o_free = bars + 17;           //     softmax -> MMA (O read out, 256 arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == kAlMmaWarp) {
        tmem_alloc(tmem_slot, 512);
        if (lane == 0) {
            // gathered: 32 cp.async-completion arrivals (one loader warp per step); dense: one arrival + TMA transaction bytes
            const uint32_t fill = p.row_map ? 32u : 1u;
            for (int i = 0; i < kAlStages; ++i) { mbar_init(&full_bar[i], fill); mbar_init(&empty_bar[i], 1); }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&q_full[i], fill);
                mbar_init(&q_empty[i], 1);
                mbar_init(&s_full[i], 1);
                mbar_init(&s_free[i], 256);
                mbar_init(&p_full[i], 256);
            }
            mbar_init(o_full, 1);
            mbar_init(o_free, 256);
            mbar_fence_init();
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch();
    griddep_wait();
    const int n_mine = (p.n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int Np = p.Np, nb = p.nb;

    if (warp >= kAlLoaderWarp0 && p.row_map == nullptr) {
        // ================= dense loader: the head's tokens are consecutive global rows -> TMA boxes, one thread =================
        // (3-d map [image][token][3C]: rows past the image's tokens are zero-filled, never the next image's)
        if (tid == kAlLoaderWarp0 * 32) {
            tma_prefetch_desc(&tmap_q);
            tma_prefetch_desc(&tmap_kv);
            int rs = 0;
            for (int n = 0; n < n_mine; ++n) {
                int item = blockIdx.x + n * gridDim.x;
                if (p.reverse) item = p.n_items - 1 - item;
                const int qt = item % p.QT, bh = item / p.QT;
                const int b = bh / p.H, h = bh - b * p.H;
                const int qb = n & 1;
                mbar_wait(&q_empty[qb], ((n >> 1) & 1) ^ 1);
                mbar_expect_tx(&q_full[qb], kAlQBytes);
                tma_load_3d(smem_gen + qb * kAlQBytes, &tmap_q, &q_full[qb], h * 64, qt * 128, b);      // rows past the image: zero-filled
                for (int pass = 0; pass < 2; ++pass) {
                    for (int j = 0; j < nb; ++j, ++rs) {
                        const int stage = rs % kAlStages;
                        mbar_wait(&empty_bar[stage], ((rs / kAlStages) & 1) ^ 1);
                        uint8_t* sk = smem_gen + 2 * kAlQBytes + stage * kAlStageBytes;
                        mbar_expect_tx(&full_bar[stage], pass ? 2 * kAlPlane : kAlPlane);
                        tma_load_3d(sk, &tmap_kv, &full_bar[stage], p.C + h * 64, j * kAlKB, b);
                        if (pass) tma_load_3d(sk + kAlPlane, &tmap_kv, &full_bar[stage], 2 * p.C + h * 64, j * kAlKB, b);
                    }
                }
            }
        }
    } else if (warp >= kAlLoaderWarp0) {
        // ================= gather loaders =================
        // A cp.async.mbarrier.arrive holds its thread until the copies have landed (~3000 cycles per block measured), so
        // the loader warps move WHOLE load steps concurrently: warp s (s < 3) owns ring stage s and loads every block
        // that goes there (one warp per stage keeps the 1-bit barrier parity unambiguous); warp 0 also loads the Q tiles.
        // Inside a warp 8 lanes move one token's 128-byte head slice, 4 tokens per sweep.
        const int lw = warp - kAlLoaderWarp0;
        const int grp = lane >> 3, chunk = lane & 7;
        const long long C3 = 3LL * p.C;
        int rs = 0;                                      // ring step counter (K blocks of pass 1, K+V blocks of pass 2)
        for (int n = 0; n < n_mine; ++n) {
            int item = blockIdx.x + n * gridDim.x;
            if (p.reverse) item = p.n_items - 1 - item;
            const int qt = item % p.QT, bh = item / p.QT;
            const int b = bh / p.H, h = bh - b * p.H;
            const __nv_bfloat16* head = p.qkv + h * 64 + chunk * 8;
            auto token_row = [&](int j) -> long long {       // global qkv row of token j of image b
                return p.row_map ? (long long)__ldg(p.row_map + (long long)b * Np + j) : (long long)b * p.N_src + j;
            };
            // ---- Q tile of item n into Q buffer n & 1 (rows past Np are zero-filled: finite scores, never stored)
            if (lw == 0) {
                const int qb = n & 1;
                mbar_wait(&q_empty[qb], ((n >> 1) & 1) ^ 1);
                long long grow[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int q = qt * 128 + grp + 4 * i;
                    grow[i] = q < Np ? token_row(q) : -1;
                }
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int r = grp + 4 * i;
                    const bool ok = grow[i] >= 0;
                    cp_async16(s_q + qb * kAlQBytes + r * 128 + ((chunk ^ (r & 7)) << 4), head + (ok ? grow[i] : 0) * C3, ok ? 16 : 0);
                }
                cp_async_arrive_noinc(&q_full[qb]);
            }
            // ---- key blocks: pass 1 needs K only, pass 2 K and V
            for (int pass = 0; pass < 2; ++pass) {
                for (int j = 0; j < nb; ++j, ++rs) {
                    const int stage = rs % kAlStages;
                    if (stage != lw) continue;
                    mbar_wait(&empty_bar[stage], ((rs / kAlStages) & 1) ^ 1);
                    const uint32_t sk = s_ring + stage * kAlStageBytes, sv = sk + kAlPlane;
                    const int rows = min(kAlKB, ((Np - j * kAlKB) + 15) & ~15);      // rows the MMAs of this block touch
                    for (int r0 = 0; r0 < rows; r0 += 32) {                            // 8 sweeps of 4 tokens: indices first, then copies
                        long long grow[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int r = r0 + grp + 4 * i, key = j * kAlKB + r;
                            grow[i] = (r < rows && key < Np) ? token_row(key) : -1;
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int r = r0 + grp + 4 * i;
                            if (r < rows) {
                                const bool ok = grow[i] >= 0;
                                const __nv_bfloat16* src = head + (ok ? grow[i] : 0) * C3;
                                const uint32_t off = r * 128 + ((chunk ^ (r & 7)) << 4);
                                cp_async16(sk + off, src + p.C, ok ? 16 : 0);
                                if (pass == 1) cp_async16(sv + off, src + 2 * p.C, ok ? 16 : 0);   // 0 * V must stay 0 past Np
                            }
                        }
                    }
                    cp_async_arrive_noinc(&full_bar[stage]);
                }
            }
        }
    } else if (warp == kAlMmaWarp) {
        // ================= MMA issuer =================
        if (lane == 0) {
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);             // B = V is MN-major
            const uint64_t qd0 = umma_desc_sw128(s_q, 16, 1024);
            uint64_t qd = qd0;
            int stage = 0;
            uint32_t phase = 0;
            uint32_t sfree_cnt[2] = {0, 0}, pfull_cnt[2] = {0, 0};
            bool pending[2] = {false, false};                                    // a pass-1 S in this buffer is still being read
            // S_j = Q K_j^T into score buffer `buf`; returns the ring stage it consumed
            auto issue_s = [&](int j, int buf, bool pass1) -> int {
                const int st = stage;
                mbar_wait(&full_bar[st], phase);
                if (++stage == kAlStages) { stage = 0; phase ^= 1; }
                if (pending[buf]) {
                    mbar_wait(&s_free[buf], sfree_cnt[buf] & 1);
                    ++sfree_cnt[buf];
                    pending[buf] = false;
                }
                fence_async_smem();              // cp.async (generic proxy) writes -> visible to the MMA's async-proxy reads
                tc_fence_after();
                const int cols = min(kAlKB, ((Np - j * kAlKB) + 15) & ~15);
                const uint32_t idesc_s = umma_idesc_bf16(128, cols, 0, 0);
                const uint64_t kd = umma_desc_sw128(s_ring + st * kAlStageBytes, 16, 1024);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_bf16(tmem_base + buf * kAlKB, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc_s, k != 0);
                umma_commit(&s_full[buf]);
                if (pass1) {
                    umma_commit(&empty_bar[st]);                                 // K block no longer needed
                    pending[buf] = true;
                }
                return st;
            };
            for (int n = 0; n < n_mine; ++n) {
                qd = qd0 + (uint64_t)(((n & 1) * kAlQBytes) >> 4);
                mbar_wait(&q_full[n & 1], (n >> 1) & 1);
                // ---- pass 1: scores only
                for (int j = 0; j < nb; ++j) issue_s(j, j & 1, true);
                // ---- pass 2: S_{j+1} is queued before P_j V_j so that it overlaps the softmax of block j
                int st_cur = issue_s(0, 0, false);
                mbar_wait(o_free, (n & 1) ^ 1);                                  // previous item's O has been read out
                for (int j = 0; j < nb; ++j) {
                    int st_next = -1;
                    if (j + 1 < nb) st_next = issue_s(j + 1, (j + 1) & 1, false);
                    const int buf = j & 1;
                    mbar_wait(&p_full[buf], pfull_cnt[buf] & 1);
                    ++pfull_cnt[buf];
                    fence_async_smem();
                    tc_fence_after();
                    const int cols = min(kAlKB, ((Np - j * kAlKB) + 15) & ~15);
                    const uint64_t vd = umma_desc_sw128(s_ring + st_cur * kAlStageBytes + kAlPlane, 16, 1024);
                    for (int k = 0; k < cols / 16; ++k)
                        umma_bf16_ts(tmem_base + kAlOCol, tmem_base + buf * kAlKB + k * 8, vd + (uint64_t)(k * (2048 >> 4)), idesc_o,
                                     (j | k) != 0);
                    umma_commit(&empty_bar[st_cur]);                             // K_j / V_j may be overwritten
                    st_cur = st_next;
                }
                umma_commit(o_full);
                umma_commit(&q_empty[n & 1]);
            }
        }
    } else {
        // ================= softmax + epilogue: 8 warps, 16 rows each =================
        const int rbase = (warp & 3) * 32 + ((warp >> 2) & 1) * 16;
        const int r0 = rbase + (lane >> 2);                                       // this thread's rows: r0 and r0 + 8
        const int k2 = (lane & 3) * 2;                                            // column pair inside an 8-column group
        const uint32_t twin = tmem_base + ((uint32_t)rbase << 16);
        const float sl2 = p.scale_log2;
        uint32_t sfull_cnt[2] = {0, 0};
        for (int n = 0; n < n_mine; ++n) {
            int item = blockIdx.x + n * gridDim.x;
            if (p.reverse) item = p.n_items - 1 - item;
            const int qt = item % p.QT, bh = item / p.QT;
            const int b = bh / p.H, h = bh - b * p.H;
            const bool warp_live = qt * 128 + rbase < Np;                         // any valid query row in this warp
            // ---------------- pass 1: row maxima ----------------
            float mx0 = -INFINITY, mx1 = -INFINITY;
            for (int j = 0; j < nb; ++j) {
                const int buf = j & 1;
                mbar_wait(&s_full[buf], sfull_cnt[buf] & 1);
                ++sfull_cnt[buf];
                tc_fence_after();
                if (warp_live) {
                    const int ncol = min(kAlKB, Np - j * kAlKB);                  // valid key columns of this block
                    const uint32_t ts = twin + buf * kAlKB;
                    uint32_t va[32], vb[32];
                    auto max64 = [&](const uint32_t (&cur)[32], int c0) {
                        if (c0 + 64 <= ncol) {
#pragma unroll
                            for (int g = 0; g < 8; ++g) {
                                mx0 = fmax3(mx0, __uint_as_float(cur[4 * g]), __uint_as_float(cur[4 * g + 1]));
                                mx1 = fmax3(mx1, __uint_as_float(cur[4 * g + 2]), __uint_as_float(cur[4 * g + 3]));
                            }
                        } else {
#pragma unroll
                            for (int g = 0; g < 8; ++g) {
                                const int c = c0 + 8 * g + k2;
                                if (c < ncol) { mx0 = fmaxf(mx0, __uint_as_float(cur[4 * g])); mx1 = fmaxf(mx1, __uint_as_float(cur[4 * g + 2])); }
                                if (c + 1 < ncol) { mx0 = fmaxf(mx0, __uint_as_float(cur[4 * g + 1])); mx1 = fmaxf(mx1, __uint_as_float(cur[4 * g + 3])); }
                            }
                        }
                    };
                    // (a 64-column load may run past the block's columns: they are this CTA's own TMEM and are masked)
                    tmem_ld16x256_x8(ts, va);
                    for (int c0 = 0; c0 < ncol; c0 += 128) {
                        tmem_ld_wait();
                        if (c0 + 64 < ncol) tmem_ld16x256_x8(ts + c0 + 64, vb);
                        max64(va, c0);
                        if (c0 + 64 < ncol) {
                            tmem_ld_wait();
                            if (c0 + 128 < ncol) tmem_ld16x256_x8(ts + c0 + 128, va);
                            max64(vb, c0 + 64);
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(&s_free[buf]);
            }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            // ---------------- pass 2: P = exp2((S - max) scale log2 e), row sums ----------------
            const float mb0 = mx0 * sl2, mb1 = mx1 * sl2;
            float sum0 = 0.f, sum1 = 0.f;
            for (int j = 0; j < nb; ++j) {
                const int buf = j & 1;
                mbar_wait(&s_full[buf], sfull_cnt[buf] & 1);
                ++sfull_cnt[buf];
                tc_fence_after();
                if (warp_live) {
                    const int ncol = min(kAlKB, Np - j * kAlKB);
                    const int ncol_pad = (ncol + 15) & ~15;
                    const uint32_t ts = twin + buf * kAlKB;
                    // one 8-column group: this thread's 2 rows x 2 columns -> one packed P word per row
                    auto exp_group = [&](uint32_t s00, uint32_t s01, uint32_t s10, uint32_t s11, int c, bool masked, uint32_t& p0, uint32_t& p1) {
                        float e00 = ex2_approx(fmaf(__uint_as_float(s00), sl2, -mb0)), e01 = ex2_approx(fmaf(__uint_as_float(s01), sl2, -mb0));
                        float e10 = ex2_approx(fmaf(__uint_as_float(s10), sl2, -mb1)), e11 = ex2_approx(fmaf(__uint_as_float(s11), sl2, -mb1));
                        if (masked) {                                             // key columns past Np contribute nothing
                            if (c + 1 >= ncol) { e01 = 0.f; e11 = 0.f; }
                            if (c >= ncol) { e00 = 0.f; e10 = 0.f; }
                        }
                        sum0 += e00 + e01;
                        sum1 += e10 + e11;
                        p0 = float2_to_bf16x2(e00, e01);
                        p1 = float2_to_bf16x2(e10, e11);
                    };
                    // The P of S columns [c0, c0+64) lands on columns [c0/2, c0/2+32) of the same 16 lanes: behind what this
                    // warp still has to read, and no other warp touches these lanes.  64-column loads: a tcgen05.ld costs
                    // 150-330 cycles whatever its size; 32 exp2 per thread hide it.
                    auto exp64 = [&](const uint32_t (&cur)[32], int c0) {
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            uint32_t pk[8];
                            const int cb = c0 + 32 * hh;
                            if (cb + 32 <= ncol) {
#pragma unroll
                                for (int g = 0; g < 4; ++g)
                                    exp_group(cur[16 * hh + 4 * g], cur[16 * hh + 4 * g + 1], cur[16 * hh + 4 * g + 2], cur[16 * hh + 4 * g + 3],
                                              0, false, pk[2 * g], pk[2 * g + 1]);
                            } else {
#pragma unroll
                                for (int g = 0; g < 4; ++g)
                                    exp_group(cur[16 * hh + 4 * g], cur[16 * hh + 4 * g + 1], cur[16 * hh + 4 * g + 2], cur[16 * hh + 4 * g + 3],
                                              cb + 8 * g + k2, true, pk[2 * g], pk[2 * g + 1]);
                            }
                            tmem_st16x128_x4(ts + (cb >> 1), pk);
                        }
                    };
                    uint32_t xa[32], xb[32];
                    const int full_end = ncol_pad & ~63;                          // columns covered by whole 64-column chunks
                    if (full_end > 0) tmem_ld16x256_x8(ts, xa);
                    for (int c0 = 0; c0 < full_end; c0 += 128) {
                        tmem_ld_wait();
                        if (c0 + 64 < full_end) tmem_ld16x256_x8(ts + c0 + 64, xb);
                        exp64(xa, c0);
                        if (c0 + 64 < full_end) {
                            tmem_ld_wait();
                            if (c0 + 128 < full_end) tmem_ld16x256_x8(ts + c0 + 128, xa);
                            exp64(xb, c0 + 64);
                        }
                    }
                    for (int c0 = full_end; c0 < ncol_pad; c0 += 16) {            // up to three 16-column tail pieces
                        uint32_t vt[8], pk[4];
                        tmem_ld16x256_x2(ts + c0, vt);
                        tmem_ld_wait();
#pragma unroll
                        for (int g = 0; g < 2; ++g)
                            exp_group(vt[4 * g], vt[4 * g + 1], vt[4 * g + 2], vt[4 * g + 3], c0 + 8 * g + k2, true, pk[2 * g], pk[2 * g + 1]);
                        tmem_st16x128_x2(ts + (c0 >> 1), pk);
                    }
                    tmem_st_wait();
                }
                tc_fence_before();
                mbar_arrive(&p_full[buf]);
            }
            sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
            sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
            sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
            sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
            // ---------------- O / rowsum -> bf16 -> global ----------------
            mbar_wait(o_full, n & 1);
            tc_fence_after();
            if (warp_live) {
                uint32_t o[32];
                tmem_ld16x256_x8(twin + kAlOCol, o);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(o_free);
                const int q0 = qt * 128 + r0, q1 = q0 + 8;
                __nv_bfloat16* dst = p.out + ((long long)b * Np + q0) * p.C + h * 64 + k2;
                if (q0 < Np) {
                    const float inv = 1.f / sum0;
#pragma unroll
                    for (int g = 0; g < 8; ++g)
                        *reinterpret_cast<uint32_t*>(dst + 8 * g) =
                            float2_to_bf16x2(__uint_as_float(o[4 * g]) * inv, __uint_as_float(o[4 * g + 1]) * inv);
                }
                if (q1 < Np) {
                    const float inv = 1.f / sum1;
                    dst += 8LL * p.C;
#pragma unroll
                    for (int g = 0; g < 8; ++g)
                        *reinterpret_cast<uint32_t*>(dst + 8 * g) =
                            float2_to_bf16x2(__uint_as_float(o[4 * g + 2]) * inv, __uint_as_float(o[4 * g + 3]) * inv);
                }
            } else {
                tc_fence_before();
                mbar_arrive(o_free);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kAlMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// returns 1 if handled, <0 on error
int launch_attention_long(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                          int C, int H, float scale, int reverse, cudaStream_t stream) {
    AttnLongParams p{};
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.row_map = row_map;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.N_src = N_src; p.Np = Np; p.C = C; p.H = H;
    p.BH = B * H;
    p.QT = (Np + 127) / 128;
    p.nb = (Np + kAlKB - 1) / kAlKB;
    p.reverse = reverse;
    p.scale_log2 = scale * 1.4426950408889634f;
    const long long items = (long long)p.BH * p.QT;
    RAJNI_REQUIRE(items < (1LL << 31), RAJNI_EINVAL, "attention_long: too many work items");
    p.n_items = (int)items;
    static int smem_granted[kMaxDevices] = {};
    if (int rc = raise_smem_limit("attention_long", attention_long_kernel, kAlSmem, smem_granted)) return rc;
    CUtensorMap tq, tkv;
    if (int rc = make_tmap_bf16_3d_ld(&tq, qkv, B, N_src, 3LL * C, 128)) return rc;           // per image: a box never reads the next image
    if (int rc = make_tmap_bf16_3d_ld(&tkv, qkv, B, N_src, 3LL * C, kAlKB)) return rc;
    const int grid = p.n_items < num_sms() ? p.n_items : num_sms();
    const int rc = launch_checked("attention_long", attention_long_kernel, dim3(grid), dim3(kAlThreads), (size_t)kAlSmem, stream, 1,
                                  tq, tkv, p);
    return rc ? rc : 1;
}

}  // namespace rajni
