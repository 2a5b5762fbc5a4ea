// HBM-bound row kernels: gather-compaction, LayerNorm, patch im2col.
// All use 16-byte vector accesses, contiguous along the fastest dimension per warp.
#include <type_traits>

#include "common.cuh"

namespace rajni {

// ------------------------------------------------------------------ gather rows
// dst[r,:] = src[row_map[r],:]   attention.py:42-43 (qkv rows), model.py:55-56 (residual rows)
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4* __restrict__ src,
                                                          const int32_t* __restrict__ row_map,
                                                          uint4* __restrict__ dst,
                                                          long long total_chunks, int chunks_per_row) {
    griddep_launch();
    griddep_wait();
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // 4 independent 16-byte loads in flight per thread
    for (; i + 3 * stride < total_chunks; i += 4 * stride) {
        uint4 v[4];
        long long idx[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            idx[u] = i + u * stride;
            int r = (int)(idx[u] / chunks_per_row);
            int c = (int)(idx[u] - (long long)r * chunks_per_row);
            v[u] = ld_stream16(src + (long long)__ldg(row_map + r) * chunks_per_row + c);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) st_stream16(dst + idx[u], v[u]);
    }
    for (; i < total_chunks; i += stride) {
        int r = (int)(i / chunks_per_row);
        int c = (int)(i - (long long)r * chunks_per_row);
        st_stream16(dst + i, ld_stream16(src + (long long)__ldg(row_map + r) * chunks_per_row + c));
    }
}

// ------------------------------------------------------------------ LayerNorm
// One warp per row, the row held in registers (CPL 16-byte chunks per lane), fp32 math:
// mean, then centred variance (biased, like nn.LayerNorm), y = (x-mean)*rstd*gamma+beta.
// STATS: also write the row's LayerNorm partial sums in the RAJNI_EPI_ROW_STATS layout that the LN-folded GEMMs read
// (slot 0 = (sum, sum of squares) of the stored bf16 row, the other slots zero, as write_prefix_rows does).  Every load
// of a row precedes its first store (the stores need the row's mean), so y may be x.
// OutT = float: the same values stored unrounded (a headless model's features), 8 columns as two 16-byte stores.
template <int CPL, bool STATS = false, typename OutT = __nv_bfloat16>
__global__ void __launch_bounds__(256) layernorm_kernel(const __nv_bfloat16* __restrict__ x, long long in_stride,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        float eps, OutT* __restrict__ y, long long out_stride, int rows, int C,
                                                        float2* __restrict__ row_stats, long long stats_ld, int stats_slots) {
    static_assert(!STATS || std::is_same<OutT, __nv_bfloat16>::value, "row statistics are those of a stored bf16 row");
    griddep_launch();
    griddep_wait();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int chunks = C >> 3;
    const __nv_bfloat16* xr = x + (long long)row * in_stride;
    float v[CPL][8];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        int j = lane + 32 * i;
        if (j < chunks) {
            uint4 u = ld_stream16(xr + j * 8);
            float2 a = bf16x2_to_float2(u.x), b = bf16x2_to_float2(u.y), c = bf16x2_to_float2(u.z), d = bf16x2_to_float2(u.w);
            v[i][0] = a.x; v[i][1] = a.y; v[i][2] = b.x; v[i][3] = b.y;
            v[i][4] = c.x; v[i][5] = c.y; v[i][6] = d.x; v[i][7] = d.y;
#pragma unroll
            for (int e = 0; e < 8; ++e) sum += v[i][e];
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[i][e] = 0.f;
        }
    }
    const float mean = warp_sum(sum) / (float)C;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        if (lane + 32 * i < chunks) {
#pragma unroll
            for (int e = 0; e < 8; ++e) { float d = v[i][e] - mean; sq += d * d; }
        }
    }
    const float rstd = rsqrtf(warp_sum(sq) / (float)C + eps);
    OutT* yr = y + (long long)row * out_stride;
    float osum = 0.f, osq = 0.f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
        int j = lane + 32 * i;
        if (j < chunks) {
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + j * 8));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + j * 8 + 4));
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + j * 8));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(beta + j * 8 + 4));
            if constexpr (std::is_same<OutT, float>::value) {
                const float4 o0 = make_float4((v[i][0] - mean) * rstd * g0.x + b0.x, (v[i][1] - mean) * rstd * g0.y + b0.y,
                                              (v[i][2] - mean) * rstd * g0.z + b0.z, (v[i][3] - mean) * rstd * g0.w + b0.w);
                const float4 o1 = make_float4((v[i][4] - mean) * rstd * g1.x + b1.x, (v[i][5] - mean) * rstd * g1.y + b1.y,
                                              (v[i][6] - mean) * rstd * g1.z + b1.z, (v[i][7] - mean) * rstd * g1.w + b1.w);
                st_stream16(yr + j * 8, *reinterpret_cast<const uint4*>(&o0));
                st_stream16(yr + j * 8 + 4, *reinterpret_cast<const uint4*>(&o1));
            } else {
                uint4 o;
                o.x = float2_to_bf16x2((v[i][0] - mean) * rstd * g0.x + b0.x, (v[i][1] - mean) * rstd * g0.y + b0.y);
                o.y = float2_to_bf16x2((v[i][2] - mean) * rstd * g0.z + b0.z, (v[i][3] - mean) * rstd * g0.w + b0.w);
                o.z = float2_to_bf16x2((v[i][4] - mean) * rstd * g1.x + b1.x, (v[i][5] - mean) * rstd * g1.y + b1.y);
                o.w = float2_to_bf16x2((v[i][6] - mean) * rstd * g1.z + b1.z, (v[i][7] - mean) * rstd * g1.w + b1.w);
                st_stream16(yr + j * 8, o);
                if (STATS) {
                    const uint32_t w[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float2 f = bf16x2_to_float2(w[k]);
                        osum += f.x + f.y;
                        osq += f.x * f.x + f.y * f.y;
                    }
                }
            }
        }
    }
    if (STATS) {
        osum = warp_sum(osum);
        osq = warp_sum(osq);
        for (int s = lane; s < stats_slots; s += 32)
            row_stats[(long long)s * stats_ld + row] = s == 0 ? make_float2(osum, osq) : make_float2(0.f, 0.f);
    }
}

// ------------------------------------------------------------------ average pooling + fc_norm
// y[b,:] = LN(mean(x[b*N + P0 .. b*N + N-1, :])): timm's head with global_pool='avg' (fc_norm over the mean of the patch
// tokens).  One cluster of kPoolCluster CTAs per image, CTA r owning columns [r*C/8, (r+1)*C/8): at 256 images that is
// 2048 CTAs to stream the rows, and the LayerNorm statistics of the mean row are combined over the cluster through DSMEM.
// Thread t sums chunk t % K (8 columns, K = C/64 chunks per CTA) over rows P0 + t/K, P0 + t/K + G, ... (G = 256/K row
// groups) in fp32, then the G partials of a column are added in group order and divided by N - P0.  The order depends on
// N, P0 and C only: an image's pooled row is bit-identical in any batch.
constexpr int kPoolCluster = 8;
constexpr int kPoolThreads = 256;
constexpr int kPoolUnroll = 4;              // row loads in flight per thread

__device__ __forceinline__ float ld_cluster_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

// Sum of v over the CTA (fixed order: lanes, then warps 0..7), then over the cluster's CTAs 0..7 (every CTA adds the same
// eight values in the same order, so all get the same bits).  slot: this CTA's shared word that its partial goes to.
__device__ __forceinline__ float pool_cluster_sum(float v, float* warp_part, float* slot) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kPoolThreads / 32; ++w) t += warp_part[w];
        *slot = t;
    }
    cluster_sync_all();
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < kPoolCluster; ++r) t += ld_cluster_f32(mapa_u32(smem_u32(slot), r));
    return t;
}

// OutT = float: the same values stored unrounded (a headless model's features).
template <typename OutT = __nv_bfloat16>
__global__ void __launch_bounds__(kPoolThreads, 4) mean_pool_layernorm_kernel(const __nv_bfloat16* __restrict__ x, int N, int P0, int C,
                                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                           float eps, OutT* __restrict__ y, long long out_stride) {
    __shared__ float part[kPoolThreads * 8];
    __shared__ float warp_part[kPoolThreads / 32];
    __shared__ float red[2];
    griddep_launch();
    griddep_wait();
    const int b = blockIdx.y;
    const int cs = C / kPoolCluster;                            // columns of this CTA (multiple of 8)
    const int K = cs >> 3, G = kPoolThreads / K;
    const int c0 = (int)cluster_ctarank() * cs;
    const int t = threadIdx.x, j = t % K, g = t / K;
    if (g < G) {
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        const __nv_bfloat16* base = x + (long long)b * N * C + c0 + j * 8;
        int n = P0 + g;
        for (; n + (kPoolUnroll - 1) * G < N; n += kPoolUnroll * G) {
            uint4 u[kPoolUnroll];
#pragma unroll
            for (int k = 0; k < kPoolUnroll; ++k) u[k] = ld_stream16(base + (long long)(n + k * G) * C);
#pragma unroll
            for (int k = 0; k < kPoolUnroll; ++k) {
                const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float2 f = bf16x2_to_float2(w[q]);
                    acc[2 * q] += f.x;
                    acc[2 * q + 1] += f.y;
                }
            }
        }
        for (; n < N; n += G) {
            const uint4 u = ld_stream16(base + (long long)n * C);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 f = bf16x2_to_float2(w[q]);
                acc[2 * q] += f.x;
                acc[2 * q + 1] += f.y;
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) part[g * cs + j * 8 + e] = acc[e];
    }
    __syncthreads();
    float m = 0.f;                                              // this thread's column of the mean row (t < cs)
    if (t < cs) {
        float s = 0.f;
        for (int q = 0; q < G; ++q) s += part[q * cs + t];
        m = s / (float)(N - P0);
    }
    const float mean = pool_cluster_sum(m, warp_part, &red[0]) / (float)C;
    const float d = t < cs ? m - mean : 0.f;
    const float rstd = rsqrtf(pool_cluster_sum(d * d, warp_part, &red[1]) / (float)C + eps);
    if (t < cs) {
        if constexpr (std::is_same<OutT, float>::value) y[(long long)b * out_stride + c0 + t] = d * rstd * gamma[c0 + t] + beta[c0 + t];
        else y[(long long)b * out_stride + c0 + t] = __float2bfloat16_rn(d * rstd * gamma[c0 + t] + beta[c0 + t]);
    }
    cluster_sync_all();                                         // no CTA leaves while another may still read its red[]
}

// ------------------------------------------------------------------ patch im2col (+ prefix rows)
// Prefix rows: the P0 rows in front of each image's patches (CLS, or CLS + distillation token), copied from a [P0, C] block
// the host prepared (token + its position embedding, or the token alone when the model adds no position to it), and
// their LayerNorm partial sums (slot 0 = the host's (sum, sum of squares) of the row, the other slots zero).
constexpr int kMaxPrefix = 2;
struct PrefixStats { float sum[kMaxPrefix], sumsq[kMaxPrefix]; };

__device__ __forceinline__ void write_prefix_rows(const uint4* __restrict__ prefix_rows, int P0, const PrefixStats& ps,
                                                  uint4* __restrict__ x, int C, int B, long long P,
                                                  float2* __restrict__ row_stats, long long stats_ld, int stats_slots) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int cchunks = C >> 3;
    const long long N0 = P + P0;                 // rows per image
    const long long pre = (long long)P0 * cchunks;
    for (long long i = t0; i < (long long)B * pre; i += stride) {
        const int b = (int)(i / pre);
        const int k = (int)(i - (long long)b * pre);          // r * cchunks + j: row-major in prefix_rows and in x alike
        x[(long long)b * N0 * cchunks + k] = __ldg(prefix_rows + k);
    }
    // LayerNorm partials of the prefix rows (the patch rows' partials come from the embed GEMM's epilogue)
    if (row_stats != nullptr) {
        const long long per = (long long)stats_slots * P0;
        for (long long i = t0; i < (long long)B * per; i += stride) {
            const int b = (int)(i / per);
            const int k = (int)(i - (long long)b * per);
            const int s = k / P0, r = k - s * P0;
            row_stats[(long long)s * stats_ld + (long long)b * N0 + r] = s == 0 ? make_float2(ps.sum[r], ps.sumsq[r]) : make_float2(0.f, 0.f);
        }
    }
}

// One thread moves one (patch, channel, ky) strip: 16 pixels in, 16 bf16 out (two 16-byte
// stores = one full 32-byte sector).  px is the fastest thread index, so a warp reads
// contiguous image rows.  Column order (c, ky, kx) matches Conv2d weight.view(C, -1).
// DT: 0 = bf16, 1 = fp32, 2 = uint8 pixels normalised here exactly as torchvision's ToTensor + Normalize do in fp32
// ((u / 255 - mean[c]) / std[c], IEEE divisions; run.py:62-70), so the bf16 result equals that of the fp32 pipeline.
struct ImageNorm { float mean[3], std[3]; };
template <int DT>
__global__ void __launch_bounds__(256) im2col16_kernel(const void* __restrict__ images, const ImageNorm norm, int B, int S,
                                                       __nv_bfloat16* __restrict__ cols,
                                                       const uint4* __restrict__ prefix_rows, int P0, const PrefixStats ps,
                                                       uint4* __restrict__ x, int C,
                                                       float2* __restrict__ row_stats, long long stats_ld, int stats_slots) {
    griddep_launch();
    griddep_wait();
    const int G = S >> 4;                       // patches per side
    const long long strips = (long long)B * G * 3 * 16 * G;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < strips; i += stride) {
        int px = (int)(i % G);
        long long t = i / G;
        int ky = (int)(t & 15); t >>= 4;
        int c = (int)(t % 3); t /= 3;
        int py = (int)(t % G);
        int b = (int)(t / G);
        const long long pix = (((long long)b * 3 + c) * S + (py * 16 + ky)) * S + px * 16;
        uint4 o0, o1;
        if (DT == 2) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(images) + pix));
            const float mean = norm.mean[c], sd = norm.std[c];
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
            uint32_t o[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float f[4];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    f[j] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)((w[k] >> (8 * j)) & 0xffu), 255.0f), mean), sd);
                o[2 * k] = float2_to_bf16x2(f[0], f[1]);
                o[2 * k + 1] = float2_to_bf16x2(f[2], f[3]);
            }
            o0 = make_uint4(o[0], o[1], o[2], o[3]);
            o1 = make_uint4(o[4], o[5], o[6], o[7]);
        } else if (DT == 1) {
            const float4* src = reinterpret_cast<const float4*>(static_cast<const float*>(images) + pix);
            float4 a = __ldg(src), bb = __ldg(src + 1), cc = __ldg(src + 2), d = __ldg(src + 3);
            o0 = make_uint4(float2_to_bf16x2(a.x, a.y), float2_to_bf16x2(a.z, a.w),
                            float2_to_bf16x2(bb.x, bb.y), float2_to_bf16x2(bb.z, bb.w));
            o1 = make_uint4(float2_to_bf16x2(cc.x, cc.y), float2_to_bf16x2(cc.z, cc.w),
                            float2_to_bf16x2(d.x, d.y), float2_to_bf16x2(d.z, d.w));
        } else {
            const uint4* src = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(images) + pix);
            o0 = __ldg(src);
            o1 = __ldg(src + 1);
        }
        const long long m = ((long long)b * G + py) * G + px;
        uint4* dst = reinterpret_cast<uint4*>(cols + m * 768 + c * 256 + ky * 16);
        dst[0] = o0;
        dst[1] = o1;
    }
    // prefix rows: x[b,0,:] = cls_token + pos_embed[0]   (model.py:35-37), and the distillation token's row after it
    write_prefix_rows(prefix_rows, P0, ps, x, C, B, (long long)G * G, row_stats, stats_ld, stats_slots);
}

// ------------------------------------------------------------------ patch im2col (+ prefix rows)
// Any patch size p that is a multiple of 8.  One thread moves one 8-pixel run of one (patch, channel, patch row): 8 pixels
// in, 16 bytes of bf16 out.  The run's index inside its (patch, channel) plane (p*p/8 runs) is the fastest thread index, so
// a warp stores 512 consecutive bytes of one cols row at p >= 16 and four 128-byte planes at p = 8: whole sectors at every
// p.  Reads are whole image-row segments of p pixels (at p = 8 the warp's four patches are neighbours, so uint8 pixels
// arrive as whole 32-byte sectors too).  Column order (c, ky, kx) matches Conv2d weight.view(C, -1).
// DT: 0 = bf16, 1 = fp32, 2 = uint8 pixels normalised here exactly as torchvision's ToTensor + Normalize do in fp32
// ((u / 255 - mean[c]) / std[c], IEEE divisions; run.py:62-70), so the bf16 result equals that of the fp32 pipeline.
constexpr int kIm2colUnroll = 4;            // independent runs in flight per thread

template <int DT>
__device__ __forceinline__ void im2col_load(const void* images, long long pix, uint4 (&r)[2]) {
    if (DT == 1) {
        const uint4* s = reinterpret_cast<const uint4*>(static_cast<const float*>(images) + pix);
        r[0] = __ldg(s);
        r[1] = __ldg(s + 1);
    } else if (DT == 2) {
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(static_cast<const uint8_t*>(images) + pix));
        r[0] = make_uint4(u.x, u.y, 0u, 0u);
    } else {
        r[0] = __ldg(reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(images) + pix));
    }
}

template <int DT>
__device__ __forceinline__ uint4 im2col_convert(const uint4 (&r)[2], const ImageNorm& norm, int c) {
    if (DT == 1) {
        const float4 a = make_float4(__uint_as_float(r[0].x), __uint_as_float(r[0].y), __uint_as_float(r[0].z), __uint_as_float(r[0].w));
        const float4 b = make_float4(__uint_as_float(r[1].x), __uint_as_float(r[1].y), __uint_as_float(r[1].z), __uint_as_float(r[1].w));
        return make_uint4(float2_to_bf16x2(a.x, a.y), float2_to_bf16x2(a.z, a.w),
                          float2_to_bf16x2(b.x, b.y), float2_to_bf16x2(b.z, b.w));
    } else if (DT == 2) {
        const float mean = norm.mean[c], sd = norm.std[c];
        const uint32_t w[2] = {r[0].x, r[0].y};
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            float f[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                f[j] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)((w[k] >> (8 * j)) & 0xffu), 255.0f), mean), sd);
            o[2 * k] = float2_to_bf16x2(f[0], f[1]);
            o[2 * k + 1] = float2_to_bf16x2(f[2], f[3]);
        }
        return make_uint4(o[0], o[1], o[2], o[3]);
    } else {
        return r[0];
    }
}

template <int DT>
__global__ void __launch_bounds__(256) im2col_kernel(const void* __restrict__ images, const ImageNorm norm, int B, int S, int p,
                                                     __nv_bfloat16* __restrict__ cols,
                                                     const uint4* __restrict__ prefix_rows, int P0, const PrefixStats ps,
                                                     uint4* __restrict__ x, int C,
                                                     float2* __restrict__ row_stats, long long stats_ld, int stats_slots) {
    griddep_launch();
    griddep_wait();
    const int G = S / p;                        // patches per side
    const int rpr = p >> 3;                     // runs per patch row
    const int rpp = p * rpr;                    // runs per (patch, channel) plane
    const long long plane = (long long)p * p;
    const int img_runs = G * G * 3 * rpp;       // = 3 S^2 / 8 < 2^31 (checked by the host)
    const long long runs = (long long)B * img_runs;
    const long long stride = (long long)gridDim.x * blockDim.x;
    // run i -> (q = run in plane, px, c, py, b), q fastest; returns the source pixel offset, sets the cols element offset.
    // One 64-bit division per run; the rest in 32 bits.
    auto locate = [&](long long i, long long& dst, int& c) {
        const int b = (int)(i / img_runs);
        unsigned t = (unsigned)(i - (long long)b * img_runs);
        const int q = (int)(t % (unsigned)rpp); t /= (unsigned)rpp;
        const int px = (int)(t % (unsigned)G); t /= (unsigned)G;
        c = (int)(t % 3u);
        const int py = (int)(t / 3u);
        const int ky = q / rpr, kx = (q - ky * rpr) * 8;
        dst = (((long long)b * G + py) * G + px) * 3 * plane + c * plane + (long long)q * 8;
        return (((long long)b * 3 + c) * S + (py * p + ky)) * S + px * p + kx;
    };
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (kIm2colUnroll - 1) * stride < runs; i += kIm2colUnroll * stride) {
        uint4 r[kIm2colUnroll][2];
        long long dst[kIm2colUnroll];
        int c[kIm2colUnroll];
#pragma unroll
        for (int u = 0; u < kIm2colUnroll; ++u) im2col_load<DT>(images, locate(i + u * stride, dst[u], c[u]), r[u]);
#pragma unroll
        for (int u = 0; u < kIm2colUnroll; ++u) *reinterpret_cast<uint4*>(cols + dst[u]) = im2col_convert<DT>(r[u], norm, c[u]);
    }
    for (; i < runs; i += stride) {
        uint4 r[2];
        long long dst;
        int c;
        im2col_load<DT>(images, locate(i, dst, c), r);
        *reinterpret_cast<uint4*>(cols + dst) = im2col_convert<DT>(r, norm, c);
    }
    // prefix rows: x[b,0,:] = cls_token + pos_embed[0]   (model.py:35-37), and the distillation token's row after it
    write_prefix_rows(prefix_rows, P0, ps, x, C, B, (long long)G * G, row_stats, stats_ld, stats_slots);
}

}  // namespace rajni

using namespace rajni;

extern "C" int rajni_gather_rows(const void* src, const int32_t* row_map, void* dst,
                                 int rows_out, int row_elems, void* stream) {
    RAJNI_REQUIRE(src && row_map && dst, RAJNI_EINVAL, "rajni_gather_rows: null pointer");
    RAJNI_REQUIRE(rows_out > 0 && row_elems > 0 && row_elems % 8 == 0, RAJNI_EINVAL,
                  "rajni_gather_rows: rows=%d row_elems=%d (must be a positive multiple of 8)", rows_out, row_elems);
    const int cpr = row_elems / 8;
    const long long total = (long long)rows_out * cpr;
    long long blocks = (total + 256 * 4 - 1) / (256 * 4);
    if (blocks > 148 * 16) blocks = 148 * 16;
    return launch_checked("gather_rows", gather_rows_kernel, dim3((int)blocks), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
                          static_cast<const uint4*>(src), row_map, static_cast<uint4*>(dst), total, cpr);
}

// The host side of the three LayerNorm entry points.  y: bf16 or fp32 rows at out_row_stride elements (a multiple of 16
// bytes, as the kernel stores 16-byte chunks).  STATS: also the rows' partial sums (bf16 rows only, see layernorm_kernel).
template <bool STATS, typename OutT>
static int launch_layernorm(const char* name, const char* kname, const void* x, long long in_row_stride, const float* gamma,
                            const float* beta, float eps, OutT* y, long long out_row_stride, int rows, int C,
                            float* row_stats, long long row_stats_ld, int stats_slots, void* stream) {
    constexpr int kOutAlign = 16 / sizeof(OutT);
    RAJNI_REQUIRE(x && gamma && beta && y && (!STATS || row_stats), RAJNI_EINVAL, "%s: null pointer", name);
    RAJNI_REQUIRE(rows > 0 && C > 0 && C % 8 == 0 && C <= 2048 && in_row_stride % 8 == 0 && out_row_stride % kOutAlign == 0 &&
                  out_row_stride >= C, RAJNI_EINVAL, "%s: rows=%d C=%d stride=%lld out stride=%lld unsupported", name, rows, C,
                  in_row_stride, out_row_stride);
    if (STATS)
        RAJNI_REQUIRE(stats_slots > 0 && row_stats_ld >= rows, RAJNI_EINVAL,
                      "%s: stats_slots=%d row_stats_ld=%lld (need slots > 0 and ld >= rows=%d)", name, stats_slots,
                      row_stats_ld, rows);
    const int cpl = (C / 8 + 31) / 32;
    const int wpb = 8;
    dim3 grid((rows + wpb - 1) / wpb), block(wpb * 32);
    auto kern = layernorm_kernel<8, STATS, OutT>;             // cpl 5..8
    switch (cpl) {
        case 1: kern = layernorm_kernel<1, STATS, OutT>; break;
        case 2: kern = layernorm_kernel<2, STATS, OutT>; break;
        case 3: kern = layernorm_kernel<3, STATS, OutT>; break;
        case 4: kern = layernorm_kernel<4, STATS, OutT>; break;
    }
    return launch_checked(kname, kern, grid, block, 0, static_cast<cudaStream_t>(stream), 1, static_cast<const __nv_bfloat16*>(x),
                          in_row_stride, gamma, beta, eps, y, out_row_stride, rows, C, reinterpret_cast<float2*>(row_stats),
                          row_stats_ld, stats_slots);
}

extern "C" int rajni_layernorm_strided(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                                       void* y, long long out_row_stride, int rows, int C, void* stream) {
    return launch_layernorm<false>("rajni_layernorm_strided", "layernorm", x, in_row_stride, gamma, beta, eps,
                                   static_cast<__nv_bfloat16*>(y), out_row_stride, rows, C, nullptr, 0, 0, stream);
}

extern "C" int rajni_layernorm_strided_f32(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                                           float* y, long long out_row_stride, int rows, int C, void* stream) {
    return launch_layernorm<false>("rajni_layernorm_f32", "layernorm_f32", x, in_row_stride, gamma, beta, eps, y,
                                   out_row_stride, rows, C, nullptr, 0, 0, stream);
}

extern "C" int rajni_layernorm_row_stats(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                                         void* y, long long out_row_stride, int rows, int C,
                                         float* row_stats, long long row_stats_ld, int stats_slots, void* stream) {
    return launch_layernorm<true>("rajni_layernorm_row_stats", "layernorm_row_stats", x, in_row_stride, gamma, beta, eps,
                                  static_cast<__nv_bfloat16*>(y), out_row_stride, rows, C, row_stats, row_stats_ld, stats_slots,
                                  stream);
}

template <typename OutT>
static int mean_pool_layernorm(const char* name, const char* kname, const void* x, int B, int N, int prefix, int C, const float* gamma, const float* beta,
                               float eps, OutT* y, long long out_row_stride, void* stream) {
    constexpr int kOutAlign = 16 / sizeof(OutT);
    RAJNI_REQUIRE(x && gamma && beta && y, RAJNI_EINVAL, "%s: null pointer", name);
    RAJNI_REQUIRE(B > 0 && B <= 65535 && prefix >= 1 && prefix <= kMaxPrefix && N > prefix && C > 0 && C % 64 == 0 && C <= 2048 &&
                  out_row_stride >= C && out_row_stride % kOutAlign == 0, RAJNI_EINVAL,
                  "%s: B=%d N=%d prefix=%d C=%d out stride=%lld unsupported (C a multiple of 64 up to 2048, "
                  "N > prefix, prefix 1 or 2)", name, B, N, prefix, C, out_row_stride);
    return launch_checked(kname, mean_pool_layernorm_kernel<OutT>, dim3(kPoolCluster, B), dim3(kPoolThreads), 0,
                          static_cast<cudaStream_t>(stream), kPoolCluster, static_cast<const __nv_bfloat16*>(x), N, prefix, C, gamma,
                          beta, eps, y, out_row_stride);
}

extern "C" int rajni_mean_pool_layernorm(const void* x, int B, int N, int prefix, int C, const float* gamma, const float* beta,
                                         float eps, void* y, long long out_row_stride, void* stream) {
    return mean_pool_layernorm("rajni_mean_pool_layernorm", "mean_pool_layernorm", x, B, N, prefix, C, gamma, beta, eps, static_cast<__nv_bfloat16*>(y),
                               out_row_stride, stream);
}

extern "C" int rajni_mean_pool_layernorm_f32(const void* x, int B, int N, int prefix, int C, const float* gamma, const float* beta,
                                             float eps, float* y, long long out_row_stride, void* stream) {
    return mean_pool_layernorm("rajni_mean_pool_layernorm_f32", "mean_pool_layernorm_f32", x, B, N, prefix, C, gamma, beta, eps, y, out_row_stride, stream);
}

extern "C" int rajni_patch_im2col_prefix(const void* images, int image_dtype, int B, int S, int patch,
                                         void* cols, const void* prefix_rows, int prefix, void* x, int C,
                                         float* row_stats, long long row_stats_ld, int stats_slots,
                                         const float* prefix_stats_host, const float* norm, void* stream) {
    RAJNI_REQUIRE(images && cols && prefix_rows && x, RAJNI_EINVAL, "rajni_patch_im2col_prefix: null pointer");
    RAJNI_REQUIRE(prefix >= 1 && prefix <= kMaxPrefix, RAJNI_EINVAL, "rajni_patch_im2col_prefix: prefix=%d (1: CLS, 2: CLS + distillation token)", prefix);
    RAJNI_REQUIRE(row_stats == nullptr || prefix_stats_host != nullptr, RAJNI_EINVAL, "rajni_patch_im2col_prefix: row_stats needs prefix_stats_host");
    PrefixStats ps{};
    if (row_stats != nullptr)
        for (int r = 0; r < prefix; ++r) {
            ps.sum[r] = prefix_stats_host[2 * r];
            ps.sumsq[r] = prefix_stats_host[2 * r + 1];
        }
    RAJNI_REQUIRE(image_dtype >= RAJNI_IMG_BF16 && image_dtype <= RAJNI_IMG_U8, RAJNI_EINVAL, "rajni_patch_im2col_prefix: image_dtype %d", image_dtype);
    RAJNI_REQUIRE(image_dtype != RAJNI_IMG_U8 || norm != nullptr, RAJNI_EINVAL, "rajni_patch_im2col_prefix: uint8 images need norm (mean[3], std[3])");
    ImageNorm nm{{0.f, 0.f, 0.f}, {1.f, 1.f, 1.f}};
    if (image_dtype == RAJNI_IMG_U8)
        for (int i = 0; i < 3; ++i) {
            nm.mean[i] = norm[i];
            nm.std[i] = norm[3 + i];
            RAJNI_REQUIRE(nm.std[i] > 0.f, RAJNI_EINVAL, "rajni_patch_im2col_prefix: std[%d] must be positive", i);
        }
    RAJNI_REQUIRE(patch >= 8 && patch % 8 == 0 && S > 0 && S <= 16384 && S % patch == 0 && B > 0 && C % 8 == 0, RAJNI_EINVAL,
                  "rajni_patch_im2col_prefix: patch=%d S=%d B=%d C=%d unsupported (patch must be a multiple of 8 dividing S <= 16384)", patch, S, B, C);
    const int G = S / patch;
    RAJNI_REQUIRE(row_stats == nullptr || (stats_slots > 0 && row_stats_ld >= (long long)B * (G * G + prefix)), RAJNI_EINVAL,
                  "rajni_patch_im2col_prefix: row_stats needs stats_slots > 0 and row_stats_ld >= B*(P+prefix)");
    auto s = static_cast<cudaStream_t>(stream);
    // p = 16 keeps its own kernel: 16-pixel strips, px fastest.  On a B200 at 256 images of 224 px it moves fp32 images in
    // 41.7 us against the any-patch kernel's 44.3 us, uint8 pixels in 54.5 against 78.6 us (profiles/r3_kbench.txt).
    if (patch == 16) {
        const long long strips = (long long)B * G * 3 * 16 * G;
        long long blocks = (strips + 255) / 256;
        if (blocks > 148 * 32) blocks = 148 * 32;
        auto kern = image_dtype == RAJNI_IMG_U8 ? im2col16_kernel<2> : image_dtype == RAJNI_IMG_F32 ? im2col16_kernel<1> : im2col16_kernel<0>;
        return launch_checked("patch_im2col", kern, dim3((int)blocks), dim3(256), 0, s, 1,
                              images, nm, B, S, static_cast<__nv_bfloat16*>(cols), static_cast<const uint4*>(prefix_rows), prefix, ps,
                              static_cast<uint4*>(x), C, reinterpret_cast<float2*>(row_stats), row_stats_ld, stats_slots);
    } else {
        const long long runs = (long long)B * G * G * 3 * patch * (patch / 8);
        long long blocks = (runs + 256 * kIm2colUnroll - 1) / (256 * kIm2colUnroll);
        if (blocks > 148 * 32) blocks = 148 * 32;
        auto kern = image_dtype == RAJNI_IMG_U8 ? im2col_kernel<2> : image_dtype == RAJNI_IMG_F32 ? im2col_kernel<1> : im2col_kernel<0>;
        return launch_checked("patch_im2col", kern, dim3((int)blocks), dim3(256), 0, s, 1,
                              images, nm, B, S, patch, static_cast<__nv_bfloat16*>(cols), static_cast<const uint4*>(prefix_rows), prefix, ps,
                              static_cast<uint4*>(x), C, reinterpret_cast<float2*>(row_stats), row_stats_ld, stats_slots);
    }
}
