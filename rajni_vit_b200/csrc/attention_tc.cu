// Persistent, warp-specialised tcgen05 attention over kept tokens (Np <= 256 keys, head dim 64).
//
//   out[b, i, h*64:(h+1)*64] = softmax_j( q_i . k_j * scale ) v_j        attention.py:45-54
//   token j of image b is read from global qkv row row_map[b*Np + j]     attention.py:42-43 (gather fused)
//
// One CTA per SM loops over work units.  A unit fills the two 128-row score tiles of the SM:
//   Np > 128 : one (image, head); tile 0 = queries 0..127, tile 1 = queries 128..Np-1, shared K/V
//   Np <= 128: two (image, head) pairs, one per tile, each with its own K/V
//   Np <= 64 : k = 2..8 consecutive images are PACKED into one tile (host side: launch_attention_tc); the softmax masks every
//              row to the keys of its own image (kPacked)
// Roles (512 threads):
//   warps 0-3 / 4-7 : softmax + epilogue of tile 0 / tile 1 (thread = query row = TMEM lane)
//   warp 8          : tcgen05.mma issuer (one lane), an event loop over the two tiles
//   warps 9-15      : loaders into 128-byte-swizzled shared memory, 2-4 stages deep, Q/K and V on separate
//                     barriers.  Dense call (no row map): one TMA box per plane.  Gathered call: cp.async row
//                     gather of the head's Q/K/V slices (128 B per token from arbitrary global rows), so the
//                     kept-token gather needs no separate pass over HBM
// Per tile:  S = Q K^T (SS MMA, fp32 in TMEM) -> two passes over the TMEM row (max; exp2/sum) ->
//            P written back over S as packed bf16 -> O = P V (TS MMA: A from TMEM, V MN-major from smem)
//            -> O/rowsum -> bf16 -> swizzled shared memory -> one TMA store per warp (32 rows x 128 B, clipped at Np).
// TMEM: 512 columns = 2 tiles x 256: S at [0,Np_pad), P at [0,Np_pad/2), O at [192,256) when Np_pad <= 192
// (then S of the next unit never waits for the O read-out), else at [128,192).
// Measured on B200 (tools/probes/mma_probe.cu): a tcgen05.mma with M=128 costs >= 94 cycles whatever N is,
// so the N=64 PV products run at a third of the tensor peak; with MUFU.EX2 at 16/clk/SM the softmax costs
// about as much.  The kernel is built to overlap the two, not to reach the GEMM roofline.
#include <cuda.h>

#include "common.cuh"

namespace rajni {

constexpr int kAtSoftmaxWarps = 8;
constexpr int kAtMmaWarp = 8;
constexpr int kAtLoaderWarp0 = 9;
// 7 loader warps: 16 warps in all still leave 128 registers per thread, and the cp.async row gather of the pruned blocks is
// bound by what each warp keeps in flight (4 loader warps: 119 us at 197 -> 173 tokens; the dense call needs one TMA thread)
constexpr int kAtLoaderThreads = 224;
constexpr int kAtLoaderGroups = kAtLoaderThreads / 8;                         // 8 lanes move one token's 128-byte head slice
constexpr int kAtSlots = (128 + kAtLoaderGroups - 1) / kAtLoaderGroups;       // sweeps of the groups over 128 token rows
constexpr int kAtThreads = (kAtSoftmaxWarps + 1) * 32 + kAtLoaderThreads;     // 512
constexpr int kAtMaxStages = 4;
constexpr int kAtTileCols = 256;
constexpr int kAtOutStage = kAtSoftmaxWarps * 32 * 128;                        // output staging: 32 rows x 128 B per softmax warp
constexpr int kAtSmemBudget = 224 * 1024 - kAtOutStage;                        // stages; barriers and alignment on top

struct AttnTcParams {
    const __nv_bfloat16* qkv;
    const int32_t* row_map;
    __nv_bfloat16* out;
    int N_src, Np, Np_pad, C, H, BH, two_tiles, n_units;
    int seg;                    // tokens per image inside a PACKED tile (several short images share a tile); == Np when not packed
    int o_col, o_outside;       // TMEM column of O inside a tile; o_outside = O does not overlap S's columns
    int split_col;              // > 0 (needs o_outside): P V starts once P's columns [0, split_col) are written, the rest follows
    int ksplit;                 // key column where attention_pipe.cu splits a row between its two exp warps (row-sum order)
    int plane_bytes, stages;    // bytes of one Q/K/V plane of a stage (1024-aligned); pipeline depth
    int reverse;                // walk the (image, head) items last-to-first (L2 reuse hint)
    float scale_log2;
};

// (image*H + head) handled by tile `t` of unit `u`, or -1
__device__ __forceinline__ int unit_item(const AttnTcParams& p, int u, int t) {
    const int item = p.two_tiles ? u : 2 * u + t;
    if (item >= p.BH) return -1;
    return p.reverse ? p.BH - 1 - item : item;
}

template <bool kPacked>
__global__ void __launch_bounds__(kAtThreads, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_out, const AttnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const int stage_bytes = 3 * p.plane_bytes;
    // [stages][Q|K|V planes] [output staging: 8 warps x 4 KB] [barriers]
    // (tile 1's Q operand is read as 128 rows from row 128 of its plane: the over-read lands in the stage's K plane)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_gen + p.stages * stage_bytes + kAtOutStage);
    uint64_t* qk_full = bars;                      // [4] loader -> MMA   (TMA transaction bytes of Q and K)
    uint64_t* v_full = bars + kAtMaxStages;        // [4] loader -> MMA   (V)
    uint64_t* empty_bar = bars + 2 * kAtMaxStages; // [4] MMA -> loader   (tcgen05.commit)
    uint64_t* s_full = bars + 3 * kAtMaxStages;    // [2 tiles] MMA -> softmax (S ready)
    uint64_t* p_full = s_full + 2;                 // [2 tiles] softmax -> MMA (P in TMEM, 128 arrivals)
    uint64_t* o_full = s_full + 4;                 // [2 tiles] MMA -> softmax (O ready)
    uint64_t* o_empty = s_full + 6;                // [2 tiles] softmax -> MMA (O read out)
    uint64_t* p_half = s_full + 8;                 // [2 tiles] softmax -> MMA (first split_col columns of P in TMEM)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 10);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == kAtMmaWarp) {
        tmem_alloc(tmem_slot, 512);
        if (lane == 0) {
            for (int i = 0; i < kAtMaxStages; ++i) {
                // gathered: one cp.async-completion arrival per loader thread; dense: one arrival + TMA transaction bytes
                mbar_init(&qk_full[i], p.row_map ? kAtLoaderThreads : 1);
                mbar_init(&v_full[i], p.row_map ? kAtLoaderThreads : 1);
                mbar_init(&empty_bar[i], 1);
            }
            for (int i = 0; i < 2; ++i) {
                mbar_init(&s_full[i], 1);
                mbar_init(&p_full[i], 128);
                mbar_init(&p_half[i], 128);
                mbar_init(&o_full[i], 1);
                mbar_init(&o_empty[i], 128);
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
    const int n_mine = (p.n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // units of this CTA

    if (warp >= kAtLoaderWarp0 && p.row_map == nullptr) {
        // ================= dense loader: the head's tokens are consecutive global rows -> one TMA box per plane =================
        if (tid == kAtLoaderWarp0 * 32) {
            tma_prefetch_desc(&tmap_qkv);
            const uint32_t plane_tx = (uint32_t)p.Np_pad * 128u;
            int stage = 0;
            uint32_t phase = 0;
            for (int n = 0; n < n_mine; ++n) {
                const int u = blockIdx.x + n * gridDim.x;
                const int nsub = p.two_tiles ? 1 : (unit_item(p, u, 1) >= 0 ? 2 : 1);
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_expect_tx(&qk_full[stage], 2u * plane_tx * nsub);
                mbar_expect_tx(&v_full[stage], plane_tx * nsub);
                uint8_t* sq = smem_gen + stage * stage_bytes;
                for (int pl = 0; pl < 3; ++pl)                              // Q, K first (S needs them), then V
                    for (int t = 0; t < nsub; ++t) {
                        const int item = unit_item(p, u, t);
                        const int b = item / p.H, h = item - b * p.H;
                        // 3-d map [image][token][3C]: rows past the image's tokens are zero-filled, never the next image's
                        tma_load_3d(sq + pl * p.plane_bytes + t * (128 * 128), &tmap_qkv, pl < 2 ? &qk_full[stage] : &v_full[stage],
                                    pl * p.C + h * 64, 0, b);
                    }
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp >= kAtLoaderWarp0) {
        // ================= gather loaders: 8 lanes move one token's 128-byte head slice per plane (cp.async) =================
        // (TMA tile::gather4 does the same gather in hardware but sustains only ~7.5 B/clk/SM on 128-byte rows -
        //  measured with tools/probes - so the copies are issued as 16-byte cp.async instead.)
        const int lt = tid - kAtLoaderWarp0 * 32;
        const int grp = lt >> 3, chunk = lt & 7;
        const long long C3 = 3LL * p.C;
        const int nsub = p.two_tiles ? 1 : 2;
        int stage = 0;
        uint32_t phase = 0;
        for (int n = 0; n < n_mine; ++n) {
            const int u = blockIdx.x + n * gridDim.x;
            // global row of every token this lane group moves: all index loads are issued together,
            // before (and independent of) the wait for the stage to drain
            int grow[2 * kAtSlots], hcol[2];
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int item = t < nsub ? unit_item(p, u, t) : -1;
                const int b = item >= 0 ? item / p.H : 0;
                hcol[t] = item >= 0 ? (item - b * p.H) * 64 + chunk * 8 : -1;
#pragma unroll
                for (int i = 0; i < kAtSlots; ++i) {
                    // slot t*kAtSlots+i: second sub-item, or (two_tiles) the next sweeps over the one head
                    const int j = grp + (p.two_tiles ? t * kAtSlots + i : i) * kAtLoaderGroups;
                    const int it2 = p.two_tiles ? unit_item(p, u, 0) : item;
                    const int b2 = p.two_tiles ? it2 / p.H : b;
                    int r = -1;
                    if (it2 >= 0 && j < p.Np && (p.two_tiles || j < 128)) r = p.row_map ? __ldg(p.row_map + (long long)b2 * p.Np + j) : b2 * p.N_src + j;
                    grow[t * kAtSlots + i] = r;
                }
            }
            if (p.two_tiles) hcol[1] = hcol[0];
            mbar_wait(&empty_bar[stage], phase ^ 1);
            const uint32_t sq = smem_base + stage * stage_bytes, sk = sq + p.plane_bytes, sv = sk + p.plane_bytes;
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {                    // pass 0: Q and K (what S needs), pass 1: V
#pragma unroll
                for (int k = 0; k < 2 * kAtSlots; ++k) {
                    const int t = k / kAtSlots;
                    const int j = grp + (p.two_tiles ? k : k - t * kAtSlots) * kAtLoaderGroups;
                    if (hcol[t] < 0 || j >= p.Np_pad || (!p.two_tiles && j >= 128)) continue;
                    const bool ok = grow[k] >= 0;
                    const __nv_bfloat16* src = p.qkv + (long long)(ok ? grow[k] : 0) * C3 + hcol[t];
                    const int r = (p.two_tiles ? 0 : t * 128) + j;
                    const uint32_t off = r * 128 + ((chunk ^ (r & 7)) << 4);
                    if (pass == 0) {
                        if (ok) {
                            cp_async16(sq + off, src, 16);
                            cp_async16(sk + off, src + p.C, 16);
                        }
                    } else {
                        cp_async16(sv + off, src + 2 * p.C, ok ? 16 : 0);     // rows past Np are zero-filled: 0 * V must stay 0
                    }
                }
                cp_async_arrive_noinc(pass == 0 ? &qk_full[stage] : &v_full[stage]);
            }
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == kAtMmaWarp) {
        // ================= MMA issuer: event loop over the two tiles =================
        // Per tile the tensor pipe runs  S(n) .. [softmax] .. PV(n) S(n+1) .. [softmax] .. ; the two tiles are
        // out of phase, so the issuer polls (never blocks on) the barrier of whichever tile is ready next.
        if (lane == 0) {
            const uint32_t idesc_s = umma_idesc_bf16(128, p.Np_pad, 0, 0);
            const uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);          // B = V is MN-major
            const uint32_t kv_stride = p.two_tiles ? 0 : 128 * 128;           // tile 1's K/V rows when a unit holds two heads
            const int nk = p.Np_pad / 16;
            // descriptors of stage 0 / tile 0; other stages and tiles are plain adds on the 16-byte address field
            const uint64_t qd0 = umma_desc_sw128(smem_base, 16, 1024);
            const uint64_t kd0 = umma_desc_sw128(smem_base + p.plane_bytes, 16, 1024);
            const uint64_t vd0 = umma_desc_sw128(smem_base + 2 * p.plane_bytes, 16, 1024);
            int cnt[2] = {n_mine, n_mine};
            if (unit_item(p, blockIdx.x + (n_mine - 1) * gridDim.x, 1) < 0) cnt[1] = n_mine - 1;
            int s_next[2] = {0, 0}, pv_next[2] = {0, 0};
            // stage and phase of the next S / PV of each tile (counters instead of divisions by p.stages)
            int s_stage[2] = {0, 0}, pv_stage[2] = {0, 0};
            uint32_t s_phase[2] = {0, 0}, pv_phase[2] = {0, 0};
            uint32_t pv_cnt = 0;                                              // PVs issued per stage, 4 bits each
            int qk_seen = 0, v_seen = 0;                                      // units whose Q/K (V) have been seen landed
            bool half_done[2] = {false, false};                               // the first part of the current P V is queued
            while (pv_next[0] < cnt[0] || pv_next[1] < cnt[1]) {
                bool did = false;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const uint32_t tt = tmem_base + t * kAtTileCols;
                    int n = pv_next[t];
                    if (p.split_col && !half_done[t] && n < cnt[t] && s_next[t] > n && mbar_test(&p_half[t], n & 1) &&
                        (n == 0 || mbar_test(&o_empty[t], (n - 1) & 1))) {
                        // the first columns of P(n, t) are in TMEM: start P V under the rest of the exp pass
                        const int st = pv_stage[t];
                        bool ok = true;
                        if (v_seen <= n) {
                            if (mbar_test(&v_full[st], pv_phase[t])) v_seen = n + 1;
                            else ok = false;
                        }
                        if (ok) {
                            tc_fence_after();
                            const uint64_t vd = vd0 + (uint64_t)((st * stage_bytes + t * kv_stride) >> 4);
                            for (int k = 0; k < p.split_col / 16; ++k)
                                umma_bf16_ts(tt + p.o_col, tt + k * 8, vd + (uint64_t)(k * (2048 >> 4)), idesc_o, k != 0);
                            half_done[t] = true;
                            did = true;
                        }
                    }
                    if (n < cnt[t] && s_next[t] > n && mbar_test(&p_full[t], n & 1) &&
                        (n == 0 || !p.o_outside || mbar_test(&o_empty[t], (n - 1) & 1))) {
                        // P(n, t) is in TMEM and O(n-1, t) has been read out
                        const int st = pv_stage[t];
                        bool ok = true;
                        if (v_seen <= n) {
                            if (mbar_test(&v_full[st], pv_phase[t])) v_seen = n + 1;
                            else ok = false;
                        }
                        if (ok) {
                            tc_fence_after();
                            const uint64_t vd = vd0 + (uint64_t)((st * stage_bytes + t * kv_stride) >> 4);
                            for (int k = half_done[t] ? p.split_col / 16 : 0; k < nk; ++k)
                                umma_bf16_ts(tt + p.o_col, tt + k * 8, vd + (uint64_t)(k * (2048 >> 4)), idesc_o, k != 0);
                            half_done[t] = false;
                            umma_commit(&o_full[t]);
                            pv_next[t] = n + 1;
                            if (++pv_stage[t] == p.stages) { pv_stage[t] = 0; pv_phase[t] ^= 1; }
                            const int tiles_n = (n == n_mine - 1 && cnt[1] < n_mine) ? 1 : 2;
                            const int sh = st * 4;
                            pv_cnt += 1u << sh;
                            if (((pv_cnt >> sh) & 15u) == (uint32_t)tiles_n) {
                                umma_commit(&empty_bar[st]);                  // the stage may be refilled
                                pv_cnt &= ~(15u << sh);
                            }
                            did = true;
                        }
                    }
                    n = s_next[t];
                    if (n < cnt[t] && pv_next[t] == n) {                      // PV(n-1, t) is queued: P's columns are free
                        const int st = s_stage[t];
                        bool ok = true;
                        if (qk_seen <= n) {
                            if (mbar_test(&qk_full[st], s_phase[t])) qk_seen = n + 1;
                            else ok = false;
                        }
                        if (ok && !p.o_outside && n > 0) ok = mbar_test(&o_empty[t], (n - 1) & 1);   // O sits inside S's columns
                        // stagger the tiles by half a period: tile 1 starts once tile 0 has finished its first softmax, so
                        // from then on one tile's exp2 pass (MUFU) overlaps the other's PV/S products instead of its exp2 pass
                        if (ok && t == 1 && n == 0 && cnt[0] > 0) ok = mbar_test(&p_full[0], 0);
                        if (ok) {
                            tc_fence_after();
                            const uint64_t qd = qd0 + (uint64_t)((st * stage_bytes + t * (128 * 128)) >> 4);
                            const uint64_t kd = kd0 + (uint64_t)((st * stage_bytes + t * kv_stride) >> 4);
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma_bf16(tt, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc_s, k != 0);
                            umma_commit(&s_full[t]);
                            s_next[t] = n + 1;
                            if (++s_stage[t] == p.stages) { s_stage[t] = 0; s_phase[t] ^= 1; }
                            did = true;
                        }
                    }
                }
                if (!did) __nanosleep(32);
            }
        }
    } else {
        // ================= softmax + epilogue: thread = query row = TMEM lane =================
        const int t = warp >> 2;
        const int row = (warp & 3) * 32 + lane;                               // row inside the tile
        const uint32_t trow = tmem_base + t * kAtTileCols + ((uint32_t)((warp & 3) * 32) << 16);
        const int Np = p.Np, Np_pad = p.Np_pad;
        const float sl2 = p.scale_log2;
        for (int n = 0; n < n_mine; ++n) {
            const int item = unit_item(p, blockIdx.x + n * gridDim.x, t);
            if (item < 0) break;
            const uint32_t ph = n & 1;
            const int q = (p.two_tiles ? t * 128 : 0) + row;                   // query index inside the image
            const bool warp_live = q - lane < Np;                              // any valid row in this warp
            const int item_b = item / p.H, item_h = item - item_b * p.H;       // (before the wait for S: off the critical path)
            mbar_wait(&s_full[t], ph);
            tc_fence_after();
            float sum = 1.f;
            if (warp_live) {
                uint32_t va[32], vb[32];
                // Key window of this row: all Np keys, or - packed tile: the rows are the tokens of Np / seg short images,
                // S holds every image against every image - the seg keys of the row's own image (block-diagonal mask).
                // [wlo, whi) is the union over the warp's rows (consecutive rows: lane 0 has the lowest window).
                int lo = 0, hi = Np, wlo = 0, whi = Np;
                if (kPacked) {
                    lo = (min(q, Np - 1) / p.seg) * p.seg;
                    hi = lo + p.seg;
                    wlo = __shfl_sync(0xffffffffu, lo, 0);
                    whi = __shfl_sync(0xffffffffu, hi, 31);
                }
                // ---- pass 1: row maximum, two 32-column loads in flight per wait
                float mx = -INFINITY;
                auto max32 = [&](const uint32_t (&cur)[32], int c0) {
                    if (c0 >= lo && c0 + 32 <= hi) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) mx = fmax3(mx, __uint_as_float(cur[j]), __uint_as_float(cur[j + 1]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) if (c0 + j >= lo && c0 + j < hi) mx = fmaxf(mx, __uint_as_float(cur[j]));
                    }
                };
                for (int c0 = wlo & ~63; c0 < whi; c0 += 64) {
                    tmem_ld32(trow + c0, va);
                    if (c0 + 32 < whi) tmem_ld32(trow + c0 + 32, vb);
                    tmem_ld_wait();
                    max32(va, c0);
                    if (c0 + 32 < whi) max32(vb, c0 + 32);
                }
                // ---- pass 2: p = exp2((s - max) * scale * log2 e), row sum, bf16 P back into TMEM.
                // P chunk c lands on columns [16c, 16c+16): always behind the S columns still to be read.
                // The row sum is taken in the order attention_pipe.cu takes it - even and odd columns of the key halves
                // [0, ksplit) and [ksplit, Np_pad) separately, (A0 + A1) + (B0 + B1) - so that the two kernels agree bit for
                // bit and a keep_ratio of 1.0 (gathered call) reproduces the un-pruned block (dense call) exactly.
                const float mb = mx * sl2;
                const int ksplit = p.ksplit;
                float sa0 = 0.f, sa1 = 0.f, sb0 = 0.f, sb1 = 0.f;
                auto add16 = [&](const float (&e)[32], int off, bool in_a) {
                    if (in_a) {
#pragma unroll
                        for (int j = 0; j < 16; j += 2) { sa0 += e[off + j]; sa1 += e[off + j + 1]; }
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j += 2) { sb0 += e[off + j]; sb1 += e[off + j + 1]; }
                    }
                };
                auto exp_step = [&](const uint32_t (&cur)[32], uint32_t (&nxt)[32], int c0) {
                    tmem_ld_wait();
                    if (c0 + 32 < Np_pad) tmem_ld32(trow + c0 + 32, nxt);      // may run <= 16 columns past Np_pad: still this tile's
                    float e[32];
                    if (Np_pad - c0 >= 32) {
                        uint32_t pk[16];
                        if (c0 >= lo && c0 + 32 <= hi) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) e[j] = ex2_approx(fmaf(__uint_as_float(cur[j]), sl2, -mb));
                        } else if (kPacked && (c0 + 32 <= wlo || c0 >= whi)) {   // no row of this warp has keys here (packed tile): P = 0
#pragma unroll
                            for (int j = 0; j < 32; ++j) e[j] = 0.f;
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) e[j] = (c0 + j >= lo && c0 + j < hi) ? ex2_approx(fmaf(__uint_as_float(cur[j]), sl2, -mb)) : 0.f;
                        }
#pragma unroll
                        for (int j = 0; j < 32; j += 2) pk[j >> 1] = float2_to_bf16x2(e[j], e[j + 1]);
                        add16(e, 0, c0 < ksplit);
                        add16(e, 16, c0 + 16 < ksplit);
                        tmem_st16(trow + (c0 >> 1), pk);
                    } else {                                                   // 16-column tail
                        uint32_t pk[8];
#pragma unroll
                        for (int j = 0; j < 16; ++j) e[j] = (c0 + j >= lo && c0 + j < hi) ? ex2_approx(fmaf(__uint_as_float(cur[j]), sl2, -mb)) : 0.f;
#pragma unroll
                        for (int j = 0; j < 16; j += 2) pk[j >> 1] = float2_to_bf16x2(e[j], e[j + 1]);
                        add16(e, 0, c0 < ksplit);
                        tmem_st8(trow + (c0 >> 1), pk);
                    }
                };
                // (with split_col: once P's first split_col columns are in TMEM the issuer starts P V on them)
                auto half_ready = [&]() {
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(&p_half[t]);
                };
                const int split = p.split_col;
                tmem_ld32(trow, va);
                for (int c0 = 0; c0 < Np_pad; c0 += 64) {
                    exp_step(va, vb, c0);
                    if (c0 + 32 == split) half_ready();
                    if (c0 + 32 < Np_pad) exp_step(vb, va, c0 + 32);
                    if (c0 + 64 == split) half_ready();
                }
                tmem_st_wait();
                sum = (sa0 + sa1) + (sb0 + sb1);
            } else if (p.split_col) {
                mbar_arrive(&p_half[t]);
            }
            tc_fence_before();
            mbar_arrive(&p_full[t]);
            // ---- O = P V done -> normalise, store
            if (warp_live) {                  // while P V runs: the previous store must have read the staging buffer
                if (lane == 0) bulk_wait_group_read<0>();
                __syncwarp();
            }
            mbar_wait(&o_full[t], ph);
            tc_fence_after();
            if (warp_live) {
                uint32_t o0[32], o1[32];
                tmem_ld32(trow + p.o_col, o0);
                tmem_ld32(trow + p.o_col + 32, o1);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&o_empty[t]);
                // The warp's 32 rows x 128 B go out as ONE TMA store (3-d map: rows past the image's Np are clipped), staged
                // in shared memory with the 128-byte swizzle.  (Against 32-byte st.global per row: -3 % kernel time.)
                const uint32_t s_out = smem_base + p.stages * stage_bytes + warp * 4096;
                const float inv = 1.f / sum;
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
                    tma_store_3d(&tmap_out, s_out, item_h * 64, q - lane, item_b);
                    bulk_commit_group();
                }
            } else {
                tc_fence_before();
                mbar_arrive(&o_empty[t]);
            }
        }
    }
    if (warp < kAtSoftmaxWarps && lane == 0) bulk_wait_group<0>();           // output stores complete before the CTA retires
    tc_fence_before();
    __syncthreads();
    if (warp == kAtMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// returns 1 if the tcgen05 kernel handled the call, 0 if the shape is outside its range, <0 on error
int launch_attention_tc(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                        int C, int H, float scale, int reverse, cudaStream_t stream) {
    if (Np > 256) return 0;
    // Short images share a tile: k consecutive images (k divides B, k * Np <= 128) are presented to the kernel as ONE image
    // of k * Np tokens - their rows are consecutive in qkv, in row_map and in out, so only the view changes - and the softmax
    // masks every row to the seg = Np keys of its own image.  A tile costs ~2 us whatever it holds (the chain S -> softmax ->
    // P V -> O is latency-bound), so vit_large's 14..64-token blocks run k = 2..8 times fewer of them.  The images of a tile
    // share one P V product: P is exactly 0 outside the row's image, so finite inputs give the same result as separate tiles
    // (up to the order of the fp32 accumulation), but a NaN/Inf value row reaches the images packed with it (0 * NaN).
    int seg = Np;
    static const bool nopack = getenv("RAJNI_ATTN_NOPACK") != nullptr;
    if (!nopack && Np <= 64) {
        int k = 128 / Np;
        while (k > 1 && B % k) --k;
        if (k > 1) { B /= k; N_src *= k; Np *= k; }
    }
    AttnTcParams p{};
    p.seg = seg;
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.row_map = row_map;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.N_src = N_src; p.Np = Np; p.C = C; p.H = H;
    p.reverse = reverse;
    p.BH = B * H;
    p.Np_pad = (Np + 15) & ~15;
    p.two_tiles = Np > 128;
    p.n_units = p.two_tiles ? p.BH : (p.BH + 1) / 2;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.ksplit = ((p.Np_pad / 2) + 15) & ~15;
    p.o_outside = p.Np_pad <= 192;
    p.o_col = p.o_outside ? 192 : 128;
    p.split_col = (p.o_outside && p.Np_pad >= 64) ? ((p.Np_pad / 2 + 31) & ~31) : 0;
    if (p.split_col >= p.Np_pad) p.split_col = 0;
    // a plane holds the Q (or K, or V) rows of a stage; tile 1's Q rows / the second head start at row 128
    const int plane_rows = p.two_tiles ? p.Np_pad : 128 + p.Np_pad;
    p.plane_bytes = (plane_rows * 128 + 1023) & ~1023;
    p.stages = kAtSmemBudget / (3 * p.plane_bytes);
    if (p.stages > kAtMaxStages) p.stages = kAtMaxStages;
    RAJNI_REQUIRE(p.stages >= 2, RAJNI_EINVAL, "attention_tc: Np=%d leaves room for %d stage(s)", Np, p.stages);
    const int smem = p.stages * 3 * p.plane_bytes + kAtOutStage + 256 + 1024;
    CUtensorMap tmap;
    if (int rc = make_tmap_bf16_3d_ld(&tmap, qkv, B, N_src, 3LL * C, p.Np_pad)) return rc;
    CUtensorMap tmap_out;
    RAJNI_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15u) == 0, RAJNI_EINVAL, "attention_tc: out must be 16-byte aligned (TMA store)");
    if (int rc = make_tmap_bf16_3d_box(&tmap_out, out, B, Np, C, 32)) return rc;
    const bool packed = seg < Np;
    auto kern = packed ? attention_tc_kernel<true> : attention_tc_kernel<false>;
    static int smem_granted[2][kMaxDevices] = {};
    if (int rc = raise_smem_limit("attention_tc", kern, smem, smem_granted[packed])) return rc;
    const int grid = p.n_units < num_sms() ? p.n_units : num_sms();
    const int rc = launch_checked("attention_tc", kern, dim3(grid), dim3(kAtThreads), (size_t)smem, stream, 1, tmap, tmap_out, p);
    return rc ? rc : 1;
}

}  // namespace rajni
