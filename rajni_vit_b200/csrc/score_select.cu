// Fused token scoring + selection for one image per CTA.
//
//   score  : rajni/wrapper/importance.py:5-34   (CLS attention x sigmoid(z-scored value norm))
//   select : rajni/wrapper/attention.py:31-39   (top-k of scores[:,1:], ascending, CLS prepended); generalised to P0
//            prefix tokens (CLS, or CLS + distillation token): top-k of scores[:,P0:], tokens 0..P0-1 prepended
//   carry  : rajni/wrapper/attention.py:58      (next_scores = scores[keep_idx])
//
// HBM-bound: the only large traffic is ONE pass over the K and V planes of the
// image's qkv tile (2*N*C bf16, contiguous 4C bytes per token), read with 16-byte
// streaming loads, one warp per token row.  Everything else lives in shared memory:
// per-head CLS logits [H][N], the head-averaged value rows [N][64] (fp32, so the
// centred norm is computed exactly like the reference without a second HBM pass),
// and the selection state (radix-select histogram, flags, prefix sums).
// Sequences whose logits and value rows do not fit there (score_smem_bytes over 227 KB: N > ~720 at 12 heads, e.g. the
// 785 tokens of a ViT-B/8) take the two-launch path of rajni_score_select_split: score_stream_kernel leaves them in the
// caller's workspace and score_tail_ws_kernel reads them in place (from L2), keeping only O(N) arrays in shared memory.
// bf16 tiles in, fp32 arithmetic throughout (SURVEY.md section 4.5).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace rajni {

constexpr int kSelThreads = 512;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kHeadDim = 64;
constexpr int kVmSmemStride = kHeadDim + 1;     // value rows in shared memory: thread-per-row reads without bank conflicts

// Optional event trace (tools/probes/score_trace.cu builds this file with -DRAJNI_SCORE_TRACE): globaltimer stamps (ns) of
// one CTA's thread 0.
#ifdef RAJNI_SCORE_TRACE
__device__ long long g_sc_trace[64 * 16];
__device__ int g_sc_trace_cta;
__device__ __forceinline__ long long sc_now() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define SC_TRACE(row, slot) do { if (threadIdx.x == 0 && (int)blockIdx.x == g_sc_trace_cta && (row) < 64) g_sc_trace[(row) * 16 + (slot)] = sc_now(); } while (0)
#else
#define SC_TRACE(row, slot) do { } while (0)
#endif

struct ScoreSelectParams {
    const __nv_bfloat16* qkv;   // [B,N,3C] or null (select-only)
    const float* scores_in;     // [B,N] when qkv == null
    float* scores_out;          // [B,N] or null
    int32_t* keep_idx;          // [B,keep+P0] or null (score-only)
    float* next_scores;         // [B,keep+P0]
    int32_t* row_map;           // [B*(keep+P0)] or null
    const float* pre_logit;     // [B][pad4(H*N)] CLS logits already computed by score_stream_kernel, or null
    const float* pre_vm;        // [B][N*64] head-averaged value rows already computed, or null
    int N, C, H, keep;
    int P0;                     // prefix tokens, always kept (1: CLS; 2: CLS + distillation token)
    float eps;
};

// shared memory of one image's tail (statistics + selection)
struct SelSmem {
    float* score;        // [N]
    float* scratch;      // [512] reduction scratch
    uint32_t* hist;      // [256]
    int* misc;           // [4]
    int* warp_off;       // [32]
    float* mu;           // [64]
    float* hstat;        // [64] per-head softmax sums
    float* r;            // [N rounded up to 4] first: 16-byte aligned
    float* logit;        // [H][N]
    float* tail;         // whatever follows (the fused kernel keeps the value rows here)
};
__device__ __forceinline__ SelSmem carve_sel_smem(float* smem, int N, int H) {
    SelSmem s;
    s.r = smem;                                    // 16-byte aligned, room for N rounded up to 4 (the selection keys)
    s.score = s.r + ((N + 3) & ~3);
    s.scratch = s.score + N;
    s.hist = reinterpret_cast<uint32_t*>(s.scratch + 512);
    s.misc = reinterpret_cast<int*>(s.hist + 256);
    s.warp_off = s.misc + 4;
    s.mu = reinterpret_cast<float*>(s.warp_off + 32);
    s.hstat = s.mu + 64;
    s.logit = s.hstat + 64;
    s.tail = s.logit + (size_t)H * N;
    return s;
}

// The tail's arithmetic is written for 512 "virtual" threads (16 virtual warps) so that a CTA of NT = 512 or 256 real threads
// produces the same bits: thread t plays virtual threads t, t + NT, ...; a virtual warp is always one real warp.
// Sum over the virtual threads of f(v): warp tree, then the 16 warp totals through a second warp tree.
// barrier of the NT threads that run a tail: the whole CTA, or (overlapped kernel) its compute warps on named barrier 1
template <int NT>
__device__ __forceinline__ void tail_sync() {
    if (NT == kSelThreads) __syncthreads();
    else asm volatile("bar.sync 1, %0;" :: "n"(NT) : "memory");
}

template <int NT, typename F>
__device__ __forceinline__ float block_sum(F f, float* scratch) {
    const int lane = threadIdx.x & 31;
    tail_sync<NT>();                       // scratch may still be read from a previous call
    for (int v = threadIdx.x; v < kSelThreads; v += NT) {
        const float x = warp_sum(f(v));
        if (lane == 0) scratch[v >> 5] = x;
    }
    tail_sync<NT>();
    float t = (lane < kSelWarps) ? scratch[lane] : 0.f;
    return warp_sum(t);                    // every warp reduces the same 16 values
}

// order-preserving float -> uint key (larger float => larger key); any NaN, whatever its sign bit, gets the largest key:
// torch.topk treats NaN as greater than every number (attention.py:35)
__device__ __forceinline__ uint32_t float_key(float f) {
    uint32_t u = __float_as_uint(f + 0.0f);        // -0.0 -> +0.0: they compare equal in the reference
    if ((u & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Select the `keep` largest of score[P0..N-1] (ties: lower index first), always keep tokens 0..P0-1,
// and emit ascending indices.  All threads of the CTA call this; score[] is in smem.
template <int NT>
__device__ void select_and_emit(const float* score, uint32_t* s_hist, int* s_misc, int* s_warp_off,
                                const ScoreSelectParams& p, int b) {
    const int N = p.N, keep = p.keep, P0 = p.P0, tid = threadIdx.x;
    // ---- radix select: key of the keep-th largest patch score, 8 bits per pass
    uint32_t prefix = 0, mask = 0;
    int remaining = keep;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += NT) s_hist[i] = 0;
        tail_sync<NT>();
        for (int n = P0 + tid; n < N; n += NT) {
            uint32_t k = float_key(score[n]);
            if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & 0xff], 1u);
        }
        tail_sync<NT>();
        if (tid < 32) {
            // warp 0: each lane owns 8 consecutive bins, highest bins in lane 0
            uint32_t c[8];
            uint32_t lane_total = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) { c[i] = s_hist[255 - (tid * 8 + i)]; lane_total += c[i]; }
            uint32_t incl = lane_total;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += t;
            }
            uint32_t before = incl - lane_total;          // elements in strictly higher bins of other lanes
            if (before < (uint32_t)remaining && incl >= (uint32_t)remaining) {
                uint32_t run = before;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (run < (uint32_t)remaining && run + c[i] >= (uint32_t)remaining) {
                        s_misc[0] = 255 - (tid * 8 + i);   // the digit
                        s_misc[1] = remaining - (int)run;  // still to take inside that bin
                    }
                    run += c[i];
                }
            }
        }
        tail_sync<NT>();
        prefix |= (uint32_t)s_misc[0] << shift;
        mask |= 0xffu << shift;
        remaining = s_misc[1];
        tail_sync<NT>();
    }
    const uint32_t thresh = prefix;        // exact key of the keep-th largest
    // `remaining` of the elements equal to thresh are kept, lowest index first.

    // ---- flags + ascending compaction. Thread t owns tokens [t*ipt, (t+1)*ipt).
    const int ipt = (N + NT - 1) / NT;
    const int n0 = tid * ipt;
    int n_gt = 0, n_eq = 0;
    for (int i = 0; i < ipt; ++i) {
        int n = n0 + i;
        if (n < P0) {
            n_gt += 1;                      // prefix tokens are always kept (counted as "greater")
        } else if (n < N) {
            uint32_t k = float_key(score[n]);
            n_gt += (k > thresh);
            n_eq += (k == thresh);
        }
    }
    // block exclusive scan of (n_gt, n_eq) packed: both < 2^15
    int packed = (n_gt << 16) | n_eq;
    int incl = packed;
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp_off[warp] = incl;
    tail_sync<NT>();
    if (warp == 0) {
        int w = (lane < NT / 32) ? s_warp_off[lane] : 0;
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        if (lane < NT / 32) s_warp_off[lane] = wi - w;   // exclusive warp offsets
    }
    tail_sync<NT>();
    int excl = incl - packed + s_warp_off[warp];
    int gt_before = excl >> 16, eq_before = excl & 0xffff;
    const int stride = keep + P0;
    for (int i = 0; i < ipt; ++i) {
        int n = n0 + i;
        if (n < N) {
            bool take;
            int pos;
            if (n < P0) {
                take = true;
                pos = gt_before;            // = n: only prefix tokens precede it
            } else {
                uint32_t k = float_key(score[n]);
                bool gt = k > thresh, eq = k == thresh;
                take = gt || (eq && eq_before < remaining);
                pos = gt_before + min(eq_before, remaining);
                eq_before += eq;
            }
            if (take) {
                p.keep_idx[(size_t)b * stride + pos] = n;
                p.next_scores[(size_t)b * stride + pos] = score[n];
                if (p.row_map) p.row_map[(size_t)b * stride + pos] = b * N + n;
            }
            gt_before += take && (n < P0 || float_key(score[n]) > thresh);
        }
    }
}

// One token row: CLS logits of every head (q pre-scaled) and the head-averaged value row.  Shared by the one-CTA-per-image
// kernel (destinations in shared memory) and the overlapped kernel (destinations in global scratch), so both produce
// bit-identical numbers.  Loads and arithmetic are separate so that a warp can have several rows in flight.
template <int CPL>
__device__ __forceinline__ void score_row_load(const __nv_bfloat16* row, int lane, int chunks, int C, bool live,
                                               uint4 (&kk)[CPL], uint4 (&vv)[CPL]) {
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        int j = lane + 32 * i;
        bool ok = live && j < chunks;
        kk[i] = ok ? ld_stream16(row + C + j * 8) : make_uint4(0, 0, 0, 0);
        vv[i] = ok ? ld_stream16(row + 2 * C + j * 8) : make_uint4(0, 0, 0, 0);
    }
}

template <int CPL>
__device__ __forceinline__ void score_row_math(const uint4 (&kk)[CPL], const uint4 (&vv)[CPL], const float (&q)[CPL][8],
                                               int lane, int H, int N, int n, float* logit_dst, float* vm_dst, int vm_stride, float inv_h) {
    float va[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        float2 k0 = bf16x2_to_float2(kk[i].x), k1 = bf16x2_to_float2(kk[i].y);
        float2 k2 = bf16x2_to_float2(kk[i].z), k3 = bf16x2_to_float2(kk[i].w);
        const float4 qa = make_float4(q[i][0], q[i][1], q[i][2], q[i][3]);
        const float4 qb = make_float4(q[i][4], q[i][5], q[i][6], q[i][7]);
        float dot = qa.x * k0.x;
        dot = fmaf(qa.y, k0.y, dot); dot = fmaf(qa.z, k1.x, dot); dot = fmaf(qa.w, k1.y, dot);
        dot = fmaf(qb.x, k2.x, dot); dot = fmaf(qb.y, k2.y, dot); dot = fmaf(qb.z, k3.x, dot);
        dot = fmaf(qb.w, k3.y, dot);
        // 8 lanes share a head (64 dims = 8 chunks)
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        dot += __shfl_xor_sync(0xffffffffu, dot, 4);
        int h = (lane >> 3) + 4 * i;
        if ((lane & 7) == 0 && h < H) logit_dst[(size_t)h * N + n] = dot;
        float2 v0 = bf16x2_to_float2(vv[i].x), v1 = bf16x2_to_float2(vv[i].y);
        float2 v2 = bf16x2_to_float2(vv[i].z), v3 = bf16x2_to_float2(vv[i].w);
        va[0] += v0.x; va[1] += v0.y; va[2] += v1.x; va[3] += v1.y;
        va[4] += v2.x; va[5] += v2.y; va[6] += v3.x; va[7] += v3.y;
    }
    // lanes l, l+8, l+16, l+24 hold the same 8 dims of different heads
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        va[e] += __shfl_xor_sync(0xffffffffu, va[e], 8);
        va[e] += __shfl_xor_sync(0xffffffffu, va[e], 16);
    }
    if (lane < 8) {
        float* dst = vm_dst + (size_t)n * vm_stride + lane * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) dst[e] = va[e] * inv_h;       // importance.py:24
    }
}

template <int CPL>
__device__ __forceinline__ void score_row(const __nv_bfloat16* row, const float (&q)[CPL][8], int lane, int chunks,
                                          int C, int H, int N, int n, float* logit_dst, float* vm_dst, int vm_stride, float inv_h) {
    uint4 kk[CPL], vv[CPL];
    score_row_load<CPL>(row, lane, chunks, C, true, kk, vv);
    score_row_math<CPL>(kk, vv, q, lane, H, N, n, logit_dst, vm_dst, vm_stride, inv_h);
}

// CLS query of the image, pre-scaled by 1/sqrt(64) (exact: power of two)
template <int CPL>
__device__ __forceinline__ void load_cls_query(const __nv_bfloat16* img, int lane, int chunks, float (&q)[CPL][8]) {
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        int j = lane + 32 * i;
        uint4 u = (j < chunks) ? ld_stream16(img + j * 8) : make_uint4(0, 0, 0, 0);
        float2 a = bf16x2_to_float2(u.x), bb = bf16x2_to_float2(u.y), c = bf16x2_to_float2(u.z), d = bf16x2_to_float2(u.w);
        q[i][0] = a.x * 0.125f; q[i][1] = a.y * 0.125f; q[i][2] = bb.x * 0.125f; q[i][3] = bb.y * 0.125f;
        q[i][4] = c.x * 0.125f; q[i][5] = c.y * 0.125f; q[i][6] = d.x * 0.125f; q[i][7] = d.y * 0.125f;
    }
}

// Selection for N <= 256 (every 224-px configuration): rank by counting instead of four radix passes with their twelve
// block barriers.  Thread n counts the patches with a larger key (keys in shared memory, read four at a time; the prefix
// slots and the padding hold key 0, which no score maps to); equal keys - rare - are found through a counter per rank and ordered by index
// in a second loop only their threads run.  Positions come from one ballot per warp.  Same output as select_and_emit.
template <int NT>
__device__ void select_rank_emit(const float* score, uint32_t* key, uint32_t* s_cnt, int* s_warp_cnt, const ScoreSelectParams& p, int b) {
    const int N = p.N, keep = p.keep, P0 = p.P0, tid = threadIdx.x, lane = tid & 31;
    const int N4 = (N + 3) & ~3;
    for (int n = tid; n < N4; n += NT) key[n] = (n >= P0 && n < N) ? float_key(score[n]) : 0u;
    for (int i = tid; i < 256; i += NT) s_cnt[i] = 0;
    tail_sync<NT>();
    const int n = tid;                                   // N <= 256 <= NT
    const bool live = n >= P0 && n < N;
    const uint32_t kn = live ? key[n] : 0xffffffffu;
    int gt = 0;
    if ((n & ~31) < N) {                                 // warps past the last token have nothing to count
        const uint4* k4 = reinterpret_cast<const uint4*>(key);
#pragma unroll 4
        for (int m = 0; m < N4 / 4; ++m) {
            const uint4 k = k4[m];
            gt += (k.x > kn) + (k.y > kn) + (k.z > kn) + (k.w > kn);
        }
    }
    if (live) atomicAdd(&s_cnt[gt], 1u);                 // gt <= N - P0 - 1 <= 254
    tail_sync<NT>();
    bool take = false;
    if (n < P0) {
        take = true;                                     // prefix tokens are always kept
    } else if (n < N) {
        int rank = gt;
        if (s_cnt[gt] > 1u && gt < keep) {               // tied with other patches: lower index first
            for (int m = P0; m < n; ++m) rank += (key[m] == kn);
        }
        take = rank < keep;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, take);
    if (lane == 0) s_warp_cnt[tid >> 5] = __popc(bal);
    tail_sync<NT>();
    if (take) {
        int pos = __popc(bal & ((1u << lane) - 1u));
        for (int w = 0; w < (tid >> 5); ++w) pos += s_warp_cnt[w];
        const size_t o = (size_t)b * (keep + P0) + pos;
        p.keep_idx[o] = n;
        p.next_scores[o] = score[n];
        if (p.row_map) p.row_map[o] = b * N + n;
    }
}

template <int NT>
__device__ __forceinline__ void select_any(const SelSmem& sm, const ScoreSelectParams& p, int b) {
    // sm.r is dead by now: its N (+3, the scratch after it is free too) words hold the keys
    if (p.N <= 256) select_rank_emit<NT>(sm.score, reinterpret_cast<uint32_t*>(sm.r), sm.hist, sm.warp_off, p, b);
    else select_and_emit<NT>(sm.score, sm.hist, sm.misc, sm.warp_off, p, b);
}

// squared distance of one value row (shared memory) from mu; four interleaved partial sums
__device__ __forceinline__ float row_dist2(const float* row, const float* mu) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int i = 0; i < kHeadDim / 4; ++i) {
        const float4 v = make_float4(row[4 * i], row[4 * i + 1], row[4 * i + 2], row[4 * i + 3]);
        const float d0 = v.x - mu[4 * i], d1 = v.y - mu[4 * i + 1], d2 = v.z - mu[4 * i + 2], d3 = v.w - mu[4 * i + 3];
        a0 = fmaf(d0, d0, a0); a1 = fmaf(d1, d1, a1); a2 = fmaf(d2, d2, a2); a3 = fmaf(d3, d3, a3);
    }
    return (a0 + a1) + (a2 + a3);
}

// The per-image tail: statistics of the value rows and the CLS logits, scores, selection.  The CTA's NT threads call it after a
// barrier that made sm.logit and vm (rows of kVmSmemStride floats, both in shared memory) complete.  Thread-per-token wherever
// the reference's reductions allow: ~9 block barriers in all.  (NT and the 512 "virtual threads" of block_sum: the overlapped
// kernel of tools/probes/score_overlap_persistent_experiment.patch runs the same tail on 448 threads with the same bits.)
// VS: float stride of the value rows (kVmSmemStride in shared memory, kHeadDim in the workspace).  sm.logit may point into the
// workspace too (score_tail_ws_kernel): same reads, same arithmetic, same bits.
template <int NT, int VS = kVmSmemStride>
__device__ void score_tail(const SelSmem& sm, const float* vm, const ScoreSelectParams& p, int b, int trace_row = 0) {
    const int N = p.N, H = p.H;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int vs = VS;
    const float inv_h = 1.0f / (float)H;
    SC_TRACE(32 + trace_row, 4);
    // ---- mean over tokens of the head-averaged value (importance.py:25): 8 interleaved partial sums per dim, then their sum
    {
        const int d = tid & 63;
        for (int g = tid >> 6; g < kSelThreads / 64; g += NT / 64) {
            float acc = 0.f;
            int n = g;
            for (; n < N; n += 8) acc += vm[(size_t)n * vs + d];
            sm.scratch[g * 64 + d] = acc;
        }
        tail_sync<NT>();
        if (tid < 64) {
            float t = 0.f;
#pragma unroll
            for (int gg = 0; gg < kSelThreads / 64; ++gg) t += sm.scratch[gg * 64 + tid];
            sm.mu[tid] = t / (float)N;
        }
        tail_sync<NT>();
    }
    SC_TRACE(32 + trace_row, 5);
    // ---- r[n] = || vm[n] - mu ||  (importance.py:27): thread per token
    for (int n = tid; n < N; n += NT) sm.r[n] = sqrtf(row_dist2(vm + (size_t)n * vs, sm.mu));
    SC_TRACE(32 + trace_row, 6);
    // ---- per-head softmax statistics over all N tokens (importance.py:20): warp per head
    for (int h = warp; h < H; h += NT / 32) {
        float* l = sm.logit + (size_t)h * N;
        float m = -INFINITY;
        for (int n = lane; n < N; n += 32) m = fmaxf(m, l[n]);
        m = warp_max(m);
        float s = 0.f;
        for (int n = lane; n < N; n += 32) {
            float e = expf(l[n] - m);
            l[n] = e;
            s += e;
        }
        s = warp_sum(s);
        if (lane == 0) sm.hstat[h] = s;
    }
    SC_TRACE(32 + trace_row, 7);
    // ---- z-score of r with the unbiased std (importance.py:28-32)
    const float* r = sm.r;
    const float mu = block_sum<NT>([&](int v) { float t = 0.f; for (int n = v; n < N; n += kSelThreads) t += r[n]; return t; },
                                   sm.scratch) / (float)N;
    const float var = block_sum<NT>([&](int v) { float t = 0.f; for (int n = v; n < N; n += kSelThreads) { float d = r[n] - mu; t += d * d; } return t; },
                                    sm.scratch) / (float)(N - 1);
    const float sd = sqrtf(var) + p.eps;
    SC_TRACE(32 + trace_row, 8);
    for (int n = tid; n < N; n += NT) {
        float a = 0.f;
        for (int h = 0; h < H; ++h) a += sm.logit[(size_t)h * N + n] / sm.hstat[h];
        a *= inv_h;                                                    // importance.py:21
        float z = (sm.r[n] - mu) / sd;
        float sc = a * (1.0f / (1.0f + expf(-z)));                     // importance.py:32-34
        sm.score[n] = sc;
        if (p.scores_out) p.scores_out[(size_t)b * N + n] = sc;
    }
    tail_sync<NT>();
    SC_TRACE(32 + trace_row, 9);
    if (p.keep_idx != nullptr) select_any<NT>(sm, p, b);
    SC_TRACE(32 + trace_row, 10);
}

// CPL = 16-byte chunks per lane per plane = ceil(C / 256).
// One CTA per image, everything in shared memory, no scratch: the stand-alone entry points (rajni_importance, rajni_select,
// rajni_score_select).  64 registers per thread so that two CTAs (two images) share an SM.  All images of a batch are
// resident at once and march in lock-step - pass, then tail - so the tail (~25 % of the time) is never hidden.  A persistent
// kernel that overlaps the two across images was built and measured (tools/probes/score_overlap_persistent_experiment.patch,
// profiles/r2_score_select.md): the tail's ~8 us latency is still exposed after the last image, so it did not win.
template <int CPL>
__global__ void __launch_bounds__(kSelThreads, 2) score_select_kernel(const ScoreSelectParams p) {
    extern __shared__ __align__(16) float smem[];
    const int N = p.N, C = p.C, H = p.H;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x;

    griddep_launch();
    griddep_wait();
    const SelSmem sm = carve_sel_smem(smem, N, H);
    if (p.qkv != nullptr) {
        float* s_vm = sm.tail;                     // [N][64] (scalar access only)
        const int chunks = C >> 3;                 // 16-byte chunks per plane row
        const __nv_bfloat16* img = p.qkv + (size_t)b * N * 3 * C;
        if (p.pre_logit != nullptr) {
            // split path: the K/V pass already ran (score_stream_kernel); fetch its per-token results (L2-resident) in one
            // round trip - every load of the copy is independent
            const float* gl1 = p.pre_logit + (size_t)b * (((size_t)H * N + 3) & ~(size_t)3);
            const float4* gl = reinterpret_cast<const float4*>(gl1);
            const float4* gv = reinterpret_cast<const float4*>(p.pre_vm + (size_t)b * N * kHeadDim);
            for (int i = tid; i < (H * N) / 4; i += kSelThreads) {
                const float4 v = __ldg(gl + i);
                sm.logit[4 * i] = v.x; sm.logit[4 * i + 1] = v.y; sm.logit[4 * i + 2] = v.z; sm.logit[4 * i + 3] = v.w;
            }
            for (int i = ((H * N) / 4) * 4 + tid; i < H * N; i += kSelThreads) sm.logit[i] = __ldg(gl1 + i);
#pragma unroll 8
            for (int i = tid; i < N * kHeadDim / 4; i += kSelThreads) {
                const float4 v = __ldg(gv + i);
                float* dst = s_vm + (i >> 4) * kVmSmemStride + 4 * (i & 15);
                dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
            }
        } else {
            float q[CPL][8];
            load_cls_query<CPL>(img, lane, chunks, q);
            // ---- the single HBM pass: one warp per token row, K plane then V plane
#pragma unroll 2
            for (int n = warp; n < N; n += kSelWarps)
                score_row<CPL>(img + (size_t)n * 3 * C, q, lane, chunks, C, H, N, n, sm.logit, s_vm, kVmSmemStride, 1.0f / (float)H);
        }
        __syncthreads();
        score_tail<kSelThreads>(sm, s_vm, p, b);
    } else {
        for (int n = tid; n < N; n += kSelThreads) sm.score[n] = p.scores_in[(size_t)b * N + n];
        __syncthreads();
        if (p.keep_idx != nullptr) select_any<kSelThreads>(sm, p, b);
    }
}

// Split path, kernel 1: when a batch has far fewer images than the GPU has SMs (vit_large at 32 images per GPU), one CTA
// per image leaves most SMs idle and each CTA latency-bound.  This kernel spreads the K/V pass over (image, 16-row block)
// CTAs and leaves the per-token results in global scratch; score_select_kernel then starts from them (pre_logit / pre_vm).
constexpr int kStreamThreads = 256;
constexpr int kStreamRows = 16;
template <int CPL>
__global__ void __launch_bounds__(kStreamThreads) score_stream_kernel(const __nv_bfloat16* qkv, float* logit_g, float* vm_g,
                                                                      int N, int C, int H) {
    griddep_launch();
    griddep_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.y, chunks = C >> 3;
    const __nv_bfloat16* img = qkv + (size_t)b * N * 3 * C;
    float q[CPL][8];
    load_cls_query<CPL>(img, lane, chunks, q);
    const float inv_h = 1.0f / (float)H;
    float* logit_dst = logit_g + (size_t)b * (((size_t)H * N + 3) & ~(size_t)3);     // per-image stride padded to 16 bytes
    float* vm_dst = vm_g + (size_t)b * N * kHeadDim;
    for (int n = blockIdx.x * kStreamRows + warp; n < min(N, (int)(blockIdx.x + 1) * kStreamRows); n += kStreamThreads / 32)
        score_row<CPL>(img + (size_t)n * 3 * C, q, lane, chunks, C, H, N, n, logit_dst, vm_dst, kHeadDim, inv_h);
}

// Split path, kernel 2 for long sequences: the per-image tail reading the CLS logits and value rows where score_stream_kernel
// left them (L2-resident: 61 MB at 256 images x 785 tokens x 12 heads) instead of staging them in shared memory, which then
// holds only the O(N) selection arrays.  The softmax exponentials overwrite the image's logits in the workspace.
__global__ void __launch_bounds__(kSelThreads) score_tail_ws_kernel(const ScoreSelectParams p, float* logit_g) {
    extern __shared__ __align__(16) float smem[];
    griddep_launch();
    griddep_wait();
    const int b = blockIdx.x;
    SelSmem sm = carve_sel_smem(smem, p.N, 0);
    sm.logit = logit_g + (size_t)b * (((size_t)p.H * p.N + 3) & ~(size_t)3);
    score_tail<kSelThreads, kHeadDim>(sm, p.pre_vm + (size_t)b * p.N * kHeadDim, p, b);
}

constexpr size_t kSmemLimit = 227 * 1024;

static size_t score_smem_bytes(int N, int H, bool with_logit, bool with_vm) {
    size_t floats = (size_t)((N + 3) & ~3) + N + 512 + 256 + 4 + 32 + 64 + 64;
    if (with_logit) floats += (size_t)H * N;
    if (with_vm) floats += (size_t)N * kVmSmemStride;
    return floats * sizeof(float);
}

static int launch_score_select(const ScoreSelectParams& p, int B, cudaStream_t stream) {
    const bool with_score = p.qkv != nullptr;
    size_t smem = score_smem_bytes(p.N, p.H, with_score, with_score);
    RAJNI_REQUIRE(smem <= kSmemLimit, RAJNI_EINVAL,
                  "score_select: N=%d H=%d needs %zu B of shared memory (rajni_score_select_split takes such shapes)", p.N, p.H, smem);
    int cpl = with_score ? (p.C + 255) / 256 : 1;
    void (*kern)(const ScoreSelectParams) = nullptr;
    switch (cpl) {
        case 1: kern = score_select_kernel<1>; break;
        case 2: kern = score_select_kernel<2>; break;
        case 3: kern = score_select_kernel<3>; break;
        case 4: kern = score_select_kernel<4>; break;
        default: RAJNI_REQUIRE(false, RAJNI_EINVAL, "score_select: C=%d > 1024 unsupported", p.C);
    }
    static int smem_granted[4][kMaxDevices] = {};
    if (int rc = raise_smem_limit("score_select", kern, (int)smem, smem_granted[cpl - 1])) return rc;
    return launch_checked("score_select", kern, dim3(B), dim3(kSelThreads), smem, stream, 1, p);
}

// true when one image's CLS logits and value rows do not fit the per-image kernel's shared memory
static bool needs_workspace_tail(int N, int H) { return score_smem_bytes(N, H, true, true) > kSmemLimit; }

static int launch_score_tail_ws(const ScoreSelectParams& p, float* logit_g, int B, cudaStream_t stream) {
    const size_t smem = score_smem_bytes(p.N, 0, false, false);
    static int smem_granted[kMaxDevices] = {};
    if (int rc = raise_smem_limit("score_tail_ws", score_tail_ws_kernel, (int)smem, smem_granted)) return rc;
    return launch_checked("score_tail_ws", score_tail_ws_kernel, dim3(B), dim3(kSelThreads), smem, stream, 1, p, logit_g);
}

static size_t split_workspace_floats(int B, int N, int H) {
    return (size_t)B * (((size_t)H * N + 3) & ~(size_t)3) + (size_t)B * N * kHeadDim;
}

// split path, kernel 1 (see score_stream_kernel)
static int launch_score_stream(const __nv_bfloat16* qkv, int B, int N, int C, int H, float* ws, cudaStream_t stream) {
    float* logit_g = ws;
    float* vm_g = ws + (size_t)B * (((size_t)H * N + 3) & ~(size_t)3);
    void (*kern)(const __nv_bfloat16*, float*, float*, int, int, int) = nullptr;
    switch ((C + 255) / 256) {
        case 1: kern = score_stream_kernel<1>; break;
        case 2: kern = score_stream_kernel<2>; break;
        case 3: kern = score_stream_kernel<3>; break;
        case 4: kern = score_stream_kernel<4>; break;
        default: RAJNI_REQUIRE(false, RAJNI_EINVAL, "score_select: C=%d > 1024 unsupported", C);
    }
    return launch_checked("score_stream", kern, dim3((N + kStreamRows - 1) / kStreamRows, B), dim3(kStreamThreads), 0, stream, 1,
                          qkv, logit_g, vm_g, N, C, H);
}

static int check_score_shape(int B, int N, int C, int H) {
    RAJNI_REQUIRE(B > 0 && N >= 2 && N <= 4096, RAJNI_EINVAL, "score: bad B=%d N=%d", B, N);
    RAJNI_REQUIRE(H > 0 && C == H * kHeadDim, RAJNI_EINVAL, "score: head dim must be 64 (C=%d H=%d)", C, H);
    return 0;
}

static int check_keep(const char* fn, int N, int P0, int keep) {
    RAJNI_REQUIRE(P0 >= 1 && P0 <= 2, RAJNI_EINVAL, "%s: prefix=%d (1: CLS, 2: CLS + distillation token)", fn, P0);
    RAJNI_REQUIRE(keep >= 1, RAJNI_EINVAL, "%s: keep=%d < 1", fn, keep);
    RAJNI_REQUIRE(keep <= N - P0, RAJNI_ERANGE, "selected index k out of range (keep=%d, patches=%d)", keep, N - P0);
    return 0;
}

static int select_prefix(const char* fn, const float* scores, int B, int N, int P0, int keep, int32_t* keep_idx,
                         float* next_scores, int32_t* row_map, cudaStream_t stream) {
    RAJNI_REQUIRE(scores && keep_idx && next_scores, RAJNI_EINVAL, "%s: null pointer", fn);
    RAJNI_REQUIRE(B > 0 && N >= 2 && N <= 16384, RAJNI_EINVAL, "%s: bad B=%d N=%d", fn, B, N);
    if (int rc = check_keep(fn, N, P0, keep)) return rc;
    ScoreSelectParams p{};
    p.scores_in = scores;
    p.keep_idx = keep_idx; p.next_scores = next_scores; p.row_map = row_map;
    p.N = N; p.C = 0; p.H = 0; p.keep = keep; p.P0 = P0; p.eps = 0.f;
    return launch_score_select(p, B, stream);
}

// workspace == null: the one-launch kernel; else the split path (K/V pass over (image, row-block) CTAs, then the tail).
// keep_idx == null: scores only.
static int score_select_prefix(const char* fn, const void* qkv, int B, int N, int C, int H, int P0, int keep, float eps,
                               float* scores, int32_t* keep_idx, float* next_scores, int32_t* row_map,
                               void* workspace, size_t workspace_bytes, cudaStream_t s) {
    RAJNI_REQUIRE(qkv && (keep_idx ? next_scores != nullptr : scores != nullptr), RAJNI_EINVAL, "%s: null pointer", fn);
    if (int rc = check_score_shape(B, N, C, H)) return rc;
    if (keep_idx != nullptr) {
        if (int rc = check_keep(fn, N, P0, keep)) return rc;
    }
    ScoreSelectParams p{};
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.scores_out = scores;
    p.keep_idx = keep_idx; p.next_scores = next_scores; p.row_map = row_map;
    p.N = N; p.C = C; p.H = H; p.keep = keep_idx ? keep : 0; p.P0 = P0; p.eps = eps;
    if (workspace == nullptr) return launch_score_select(p, B, s);
    RAJNI_REQUIRE(B <= 65535, RAJNI_EINVAL, "%s: B=%d exceeds the grid limit", fn, B);
    RAJNI_REQUIRE(workspace_bytes >= split_workspace_floats(B, N, H) * sizeof(float) && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                  RAJNI_EINVAL, "%s: workspace too small (%zu B) or not 16-byte aligned", fn, workspace_bytes);
    float* ws = static_cast<float*>(workspace);
    if (int rc = launch_score_stream(p.qkv, B, N, C, H, ws, s)) return rc;
    p.pre_logit = ws;
    p.pre_vm = ws + (size_t)B * (((size_t)H * N + 3) & ~(size_t)3);
    // RAJNI_SCORE_WS_TAIL=1 (read per call; tests): the long-sequence tail at any N, to compare it with the shared-memory one
    if (needs_workspace_tail(N, H) || getenv("RAJNI_SCORE_WS_TAIL") != nullptr) return launch_score_tail_ws(p, ws, B, s);
    return launch_score_select(p, B, s);
}

}  // namespace rajni

using namespace rajni;

extern "C" int rajni_importance(const void* qkv, int B, int N, int C, int H, float eps,
                                float* scores, void* stream) {
    RAJNI_REQUIRE(qkv && scores, RAJNI_EINVAL, "rajni_importance: null pointer");
    if (int rc = check_score_shape(B, N, C, H)) return rc;
    ScoreSelectParams p{};
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.scores_out = scores;
    p.N = N; p.C = C; p.H = H; p.keep = 0; p.eps = eps;
    return launch_score_select(p, B, static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_select_prefix(const float* scores, int B, int N, int prefix, int keep, int32_t* keep_idx,
                                   float* next_scores, int32_t* row_map, void* stream) {
    return select_prefix("rajni_select_prefix", scores, B, N, prefix, keep, keep_idx, next_scores, row_map,
                         static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_select(const float* scores, int B, int N, int keep, int32_t* keep_idx,
                            float* next_scores, int32_t* row_map, void* stream) {
    return select_prefix("rajni_select", scores, B, N, 1, keep, keep_idx, next_scores, row_map, static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_score_select_prefix(const void* qkv, int B, int N, int C, int H, int prefix, int keep, float eps,
                                         float* scores, int32_t* keep_idx, float* next_scores, int32_t* row_map,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    return score_select_prefix("rajni_score_select_prefix", qkv, B, N, C, H, prefix, keep, eps, scores, keep_idx, next_scores,
                               row_map, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_score_select(const void* qkv, int B, int N, int C, int H, int keep, float eps,
                                  float* scores, int32_t* keep_idx, float* next_scores,
                                  int32_t* row_map, void* stream) {
    RAJNI_REQUIRE(keep_idx, RAJNI_EINVAL, "rajni_score_select: null pointer");
    return score_select_prefix("rajni_score_select", qkv, B, N, C, H, 1, keep, eps, scores, keep_idx, next_scores, row_map,
                               nullptr, 0, static_cast<cudaStream_t>(stream));
}

extern "C" size_t rajni_score_select_workspace_bytes(int B, int N, int C, int H) {
    (void)C;
    if (B <= 0 || N <= 0 || H <= 0) return 0;
    return split_workspace_floats(B, N, H) * sizeof(float);
}

extern "C" int rajni_score_select_split(const void* qkv, int B, int N, int C, int H, int keep, float eps,
                                        float* scores, int32_t* keep_idx, float* next_scores, int32_t* row_map,
                                        void* workspace, size_t workspace_bytes, void* stream) {
    RAJNI_REQUIRE(workspace, RAJNI_EINVAL, "rajni_score_select_split: null pointer");
    return score_select_prefix("rajni_score_select_split", qkv, B, N, C, H, 1, keep, eps, scores, keep_idx, next_scores, row_map,
                               workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_score_select_needs_workspace(int N, int H) {
    return N > 0 && H > 0 && needs_workspace_tail(N, H) ? 1 : 0;
}
