// GPU JPEG decode of the baseline subset (include/rajni_jpeg.h), bit-identical to PIL.Image.open(f).convert("RGB").
//
// The arithmetic is libjpeg(-turbo)'s at Pillow's defaults, restated and pinned against Pillow in oracle/jpeg_oracle.py:
//   jpeg_huffman  one CTA per image, one decoding thread (the stream is sequential; the other lanes load the image's
//                 Huffman tables into shared memory and pull its bytes into L2).  A 64-bit bit buffer in registers,
//                 0xFF00 unstuffed on refill, a marker ends the data (zeros follow, as in libjpeg); DC prediction,
//                 EOB/ZRL, the extend rule; int16 coefficients in natural order.  Every read is bounded by the image's
//                 byte range and every write by its coefficient slot: a malformed stream ends as a status, never a fault.
//   jpeg_idct     dequantise + jpeg_idct_islow (CONST_BITS 13, PASS1_BITS 2, 64-bit products as in the C code), level
//                 shift and the range limit (mask to 10 bits, then the table = clamp of the sign-extended value + 128).
//   jpeg_color    fancy (triangle) upsampling of h2v1 / h2v2 chroma (first/last column rules, context rows replicated at
//                 the plane's top and bottom, plain replication when the chroma plane is at most 2 samples wide) and
//                 jdcolor's fixed-point YCbCr -> RGB; grayscale R = G = B = Y.  HWC uint8 frames.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "../../include/rajni_jpeg.h"

namespace rajni {

constexpr int kJpegMaxSide = 16384;
constexpr int kLutBits = 9;

// jpeg_natural_order: zig-zag position -> natural (row-major) index
__constant__ uint8_t c_natural[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63};
static const uint8_t h_natural[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63};

// One Huffman table as the decoder uses it: a 9-bit lookahead table and libjpeg's maxcode / valoffset for longer codes.
struct HuffDev {
    uint16_t lut[1 << kLutBits];   // (code length << 8) | symbol for codes of <= 9 bits, 0 = longer code
    int maxcode[18];               // largest code of each length (-1: none); [17] is a sentinel above every code
    int valoff[18];                // symbol index of a length-l code = code + valoff[l]
    uint8_t vals[256];
};
static_assert(sizeof(HuffDev) % 16 == 0, "HuffDev is copied to shared memory in 16-byte words");

constexpr int kMaxTabs = 6;        // distinct (class, id) tables one scan of <= 3 components can use

struct JpegJob {
    long long src, src_end;        // entropy-coded bytes of the image in `files`
    long long coef;                // int16 element offset of component 0's blocks in the coefficient area
    long long plane;               // byte offset of component 0's samples in the plane area
    long long frame;               // byte offset of the HWC frame in `frames`
    long long idct0, row0;         // first jpeg_idct CTA / jpeg_color CTA (one per row) of the image over the batch
    int w, h, ncomp, hs, vs, mcux, mcuy, restart;
    int bw[3], bh[3];              // blocks per row / column of each component as stored
    int dc[3], ac[3];              // index of each component's tables in this job's table list
    int tab0, ntab;                // first HuffDev of the job in the table area, and how many
    int q[3][64];                  // quantisation table of each component, natural order
};

// ------------------------------------------------------------------ entropy decode
struct BitReader {
    uint64_t buf;                  // MSB-aligned
    int n;                         // valid bits in buf
    int fake;                      // how many of them (the low end) are zero padding past the data (<= n + 8)
    const uint8_t* p;
    const uint8_t* end;
    bool marker;                   // p rests on the 0xFF that starts a marker
    bool over;                     // bits past the data have been consumed (sticky)
};

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

__device__ __forceinline__ void br_refill(BitReader& r) {
    // fast path: append the bytes before the next 0xFF in one step, from two aligned 8-byte loads (`files` is 8-byte
    // aligned, and the 16 bytes read lie below `end`)
    const uintptr_t a = reinterpret_cast<uintptr_t>(r.p);
    if (!r.marker && (a & ~(uintptr_t)7) + 16 <= reinterpret_cast<uintptr_t>(r.end)) {
        const uint64_t* w = reinterpret_cast<const uint64_t*>(a & ~(uintptr_t)7);
        const int sh = (int)(a & 7) * 8;
        const uint64_t lo = __ldg(w), hi = __ldg(w + 1);
        const uint64_t v = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;           // v's byte j = p[j]
        const uint64_t t = ~v;
        const uint64_t z = (t - 0x0101010101010101ull) & ~t & 0x8080808080808080ull;   // exact at the lowest 0xFF byte
        const int first_ff = z ? ((__ffsll((long long)z) - 1) >> 3) : 8;
        const int k = min((64 - r.n) >> 3, first_ff);
        if (k > 0) {
            const uint64_t be = ((uint64_t)bswap32((uint32_t)v) << 32) | bswap32((uint32_t)(v >> 32));   // p[0] on top
            r.buf |= (be >> (64 - 8 * k)) << (64 - r.n - 8 * k);
            r.n += 8 * k;
            r.p += k;
        }
    }
    while (r.n <= 56) {
        uint32_t c = 0;
        bool pad = true;
        if (!r.marker && r.p < r.end) {
            c = __ldg(r.p);
            pad = false;
            if (c != 0xFF) {
                ++r.p;
            } else {
                const uint8_t* q = r.p + 1;
                while (q < r.end && __ldg(q) == 0xFF) ++q;
                if (q < r.end && __ldg(q) == 0) {
                    r.p = q + 1;
                } else {
                    r.marker = true;
                    c = 0;
                    pad = true;
                }
            }
        }
        if (pad) {
            if (r.n < r.fake) r.over = true;
            r.fake = min(r.fake, r.n) + 8;
        }
        r.buf |= (uint64_t)c << (56 - r.n);
        r.n += 8;
    }
}

__device__ __forceinline__ bool br_overrun(const BitReader& r) { return r.over || r.n < r.fake; }

__device__ __forceinline__ uint32_t br_get(BitReader& r, int k) {      // k in 1..16, n >= k
    const uint32_t v = (uint32_t)(r.buf >> (64 - k));
    r.buf <<= k;
    r.n -= k;
    return v;
}

// -1 for a code no table entry matches
__device__ __forceinline__ int br_huff(BitReader& r, const HuffDev& t) {
    const uint32_t e = t.lut[r.buf >> (64 - kLutBits)];
    if (e) {
        const int len = e >> 8;
        r.buf <<= len;
        r.n -= len;
        return e & 0xFF;
    }
    int l = kLutBits + 1;
    int code = (int)(r.buf >> (64 - l));
    while (code > t.maxcode[l]) {
        ++l;
        if (l > 16) return -1;
        code = (int)(r.buf >> (64 - l));
    }
    r.buf <<= l;
    r.n -= l;
    return t.vals[(code + t.valoff[l]) & 0xFF];
}

__device__ __forceinline__ int huff_extend(uint32_t v, int s) {
    return (int)v < (1 << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v;
}

constexpr int kHuffThreads = 32;

__global__ void __launch_bounds__(kHuffThreads) jpeg_huffman_kernel(const uint8_t* __restrict__ files, const JpegJob* __restrict__ jobs,
                                                                    const HuffDev* __restrict__ tabs, int16_t* __restrict__ coef,
                                                                    int* __restrict__ status) {
    // no griddep_launch(): jpeg_idct's CTAs would otherwise fill the SMs early and wait beside the decoders, which run
    // for the whole kernel on one thread each
    griddep_wait();
    __shared__ __align__(16) HuffDev s_tab[kMaxTabs];
    const JpegJob& job = jobs[blockIdx.x];
    const int t = threadIdx.x;
    if (job.ntab == 0) return;                                   // not a GPU file
    {
        const uint4* src = reinterpret_cast<const uint4*>(tabs + job.tab0);
        uint4* dst = reinterpret_cast<uint4*>(s_tab);
        const int words = job.ntab * (int)(sizeof(HuffDev) / 16);
        for (int i = t; i < words; i += kHuffThreads) dst[i] = src[i];
        for (long long o = job.src + 128LL * t; o < job.src_end; o += 128LL * kHuffThreads) prefetch_l2(files + o);
    }
    __syncthreads();
    if (t != 0) return;

    BitReader r{0, 0, 0, files + job.src, files + job.src_end, false, false};
    const int nc = job.ncomp, restart = job.restart, mcux = job.mcux, hs0 = job.hs, vs0 = job.vs;
    const long long nmcu = (long long)mcux * job.mcuy;
    // the coefficient area is zeroed before this kernel: only nonzero coefficients are stored
    int16_t* const cp0 = coef + job.coef;
    int16_t* const cp1 = cp0 + (long long)job.bw[0] * job.bh[0] * 64;
    int16_t* const cp2 = nc == 3 ? cp1 + (long long)job.bw[1] * job.bh[1] * 64 : cp1;
    const int bw0 = job.bw[0], bw1 = nc == 3 ? job.bw[1] : 0;
    const HuffDev* const dct0 = s_tab + job.dc[0];
    const HuffDev* const act0 = s_tab + job.ac[0];
    const HuffDev* const dct1 = s_tab + (nc == 3 ? job.dc[1] : 0);
    const HuffDev* const act1 = s_tab + (nc == 3 ? job.ac[1] : 0);
    const HuffDev* const dct2 = s_tab + (nc == 3 ? job.dc[2] : 0);
    const HuffDev* const act2 = s_tab + (nc == 3 ? job.ac[2] : 0);
    int pred0 = 0, pred1 = 0, pred2 = 0;
    int rst = 0, left = restart;
    int err = RAJNI_JPEG_OK;
    for (long long m = 0; m < nmcu && !err; ++m) {
        if (restart) {
            if (left == 0) {                                     // process_restart: drop the buffer, expect RSTn
                if (br_overrun(r)) { err = RAJNI_JPEG_TRUNCATED; break; }
                r.buf = 0;
                r.n = r.fake = 0;
                r.marker = false;
                if (r.p >= r.end || __ldg(r.p) != 0xFF) { err = RAJNI_JPEG_BAD_RESTART; break; }
                while (r.p < r.end && __ldg(r.p) == 0xFF) ++r.p;
                if (r.p >= r.end || __ldg(r.p) != 0xD0 + (rst & 7)) { err = RAJNI_JPEG_BAD_RESTART; break; }
                ++r.p;
                ++rst;
                left = restart;
                pred0 = pred1 = pred2 = 0;
            }
            --left;
        }
        const int ux = (int)(m % mcux), uy = (int)(m / mcux);
#pragma unroll
        for (int c = 0; c < 3; ++c) {                            // unrolled: every per-component value is a register
            if (c >= nc || err) break;
            const int hs = (c == 0 && nc == 3) ? hs0 : 1, vs = (c == 0 && nc == 3) ? vs0 : 1;
            const HuffDev& dct = *(c == 0 ? dct0 : c == 1 ? dct1 : dct2);
            const HuffDev& act = *(c == 0 ? act0 : c == 1 ? act1 : act2);
            int& pred = c == 0 ? pred0 : c == 1 ? pred1 : pred2;
            int16_t* const cp = c == 0 ? cp0 : c == 1 ? cp1 : cp2;
            const int bw = c == 0 ? bw0 : bw1;
            for (int by = 0; by < vs && !err; ++by) {
                for (int bx = 0; bx < hs; ++bx) {
                    int16_t* const blk = cp + ((long long)(uy * vs + by) * bw + (ux * hs + bx)) * 64;
                    if (r.n < 32) br_refill(r);
                    int s = br_huff(r, dct);
                    if (s < 0) { err = RAJNI_JPEG_BAD_CODE; break; }
                    if (s) {
                        if (r.n < 32) br_refill(r);
                        pred += huff_extend(br_get(r, s), s);
                    }
                    blk[0] = (int16_t)pred;
                    for (int k = 1; k < 64;) {
                        if (r.n < 32) br_refill(r);
                        const int rs = br_huff(r, act);
                        if (rs < 0) { err = RAJNI_JPEG_BAD_CODE; break; }
                        const int run = rs >> 4;
                        s = rs & 15;
                        if (s) {
                            k += run;
                            if (k > 63) { err = RAJNI_JPEG_BAD_RUN; break; }
                            blk[c_natural[k]] = (int16_t)huff_extend(br_get(r, s), s);
                            ++k;
                        } else if (run == 15) {
                            k += 16;
                        } else {
                            break;
                        }
                    }
                    if (err) break;
                }
            }
        }
    }
    if (!err && br_overrun(r)) err = RAJNI_JPEG_TRUNCATED;      // the last MCU used bits past the data
    status[blockIdx.x] = err;
}

// ------------------------------------------------------------------ IDCT
constexpr int kIdctBlocks = 32;                                  // 8x8 blocks per CTA, 8 threads each

__device__ __forceinline__ long long descale(long long x, int n) { return (x + (1LL << (n - 1))) >> n; }

// jpeg_idct_islow's butterfly; o[] gets the 8 undescaled outputs
__device__ __forceinline__ void islow_1d(long long s0, long long s1, long long s2, long long s3, long long s4, long long s5,
                                         long long s6, long long s7, long long (&o)[8]) {
    long long z1 = (s2 + s6) * 4433;
    long long tmp2 = z1 + s6 * -15137;
    long long tmp3 = z1 + s2 * 6270;
    long long tmp0 = (s0 + s4) * 8192;
    long long tmp1 = (s0 - s4) * 8192;
    const long long t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
    tmp0 = s7; tmp1 = s5; tmp2 = s3; tmp3 = s1;
    z1 = tmp0 + tmp3;
    long long z2 = tmp1 + tmp2, z3 = tmp0 + tmp2, z4 = tmp1 + tmp3;
    const long long z5 = (z3 + z4) * 9633;
    tmp0 *= 2446;
    tmp1 *= 16819;
    tmp2 *= 25172;
    tmp3 *= 12299;
    z1 *= -7373;
    z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    tmp0 += z1 + z3;
    tmp1 += z2 + z4;
    tmp2 += z2 + z3;
    tmp3 += z1 + z4;
    o[0] = t10 + tmp3; o[7] = t10 - tmp3;
    o[1] = t11 + tmp2; o[6] = t11 - tmp2;
    o[2] = t12 + tmp1; o[5] = t12 - tmp1;
    o[3] = t13 + tmp0; o[4] = t13 - tmp0;
}

// the image a flattened-grid CTA belongs to: the last job whose first CTA is <= x (images without CTAs share their
// successor's first CTA, so the search lands on an image that has them)
template <bool kRows>
__device__ __forceinline__ int job_of(const JpegJob* __restrict__ jobs, int B, long long x) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((kRows ? jobs[mid].row0 : jobs[mid].idct0) <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(kIdctBlocks * 8) jpeg_idct_kernel(const JpegJob* __restrict__ jobs, int B, const int16_t* __restrict__ coef,
                                                                    uint8_t* __restrict__ planes, const int* __restrict__ status) {
    griddep_launch();
    griddep_wait();
    __shared__ __align__(16) int16_t s_coef[kIdctBlocks][64];
    __shared__ int s_ws[kIdctBlocks][64];
    const int jb = job_of<false>(jobs, B, blockIdx.x);              // one grid over every image's blocks
    const JpegJob& job = jobs[jb];
    if (job.ntab == 0 || status[jb] != RAJNI_JPEG_OK) return;
    long long nblk = 0;
    for (int c = 0; c < job.ncomp; ++c) nblk += (long long)job.bw[c] * job.bh[c];
    const long long first = ((long long)blockIdx.x - job.idct0) * kIdctBlocks;
    if (first >= nblk) return;
    const int t = threadIdx.x;
    // 32 blocks x 128 B of coefficients, 16 B per thread (components are contiguous: the blocks of one launch row are)
    {
        const long long b = first + (t >> 3);
        if (b < nblk) reinterpret_cast<uint4*>(s_coef)[t] = reinterpret_cast<const uint4*>(coef + job.coef + b * 64)[t & 7];
    }
    __syncthreads();
    const int lb = t >> 3, col = t & 7;
    const long long b = first + lb;
    if (b >= nblk) return;                                       // no barrier follows for these threads' blocks
    int c = 0;
    long long bi = b;
    while (c + 1 < job.ncomp && bi >= (long long)job.bw[c] * job.bh[c]) { bi -= (long long)job.bw[c] * job.bh[c]; ++c; }
    const int* q = job.q[c];
    // pass 1: column `col`
    {
        long long s[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) s[k] = (long long)s_coef[lb][k * 8 + col] * q[k * 8 + col];
        long long o[8];
        islow_1d(s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], o);
#pragma unroll
        for (int k = 0; k < 8; ++k) s_ws[lb][k * 8 + col] = (int)descale(o[k], 13 - 2);
    }
    __syncwarp(0xFFu << (t & 24));                               // a block's 8 threads are lanes 8i..8i+7 of one warp
    // pass 2: row `col`
    {
        const int* w = s_ws[lb] + col * 8;
        long long o[8];
        islow_1d(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o);
        uint32_t px[2] = {0, 0};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            int x = (int)(descale(o[k], 13 + 2 + 3) & 1023);
            x = (x < 512 ? x : x - 1024) + 128;
            x = x < 0 ? 0 : (x > 255 ? 255 : x);
            px[k >> 2] |= (uint32_t)x << (8 * (k & 3));
        }
        long long poff = job.plane;
        for (int cc = 0; cc < c; ++cc) poff += (long long)job.bw[cc] * job.bh[cc] * 64;
        const int pw = job.bw[c] * 8;
        const long long by = bi / job.bw[c], bx = bi % job.bw[c];
        *reinterpret_cast<uint2*>(planes + poff + (by * 8 + col) * pw + bx * 8) = make_uint2(px[0], px[1]);
    }
}

// ------------------------------------------------------------------ upsampling + colour
// jdcolor.c build_ycc_rgb_table, SCALEBITS 16
__device__ __forceinline__ int fix16(double v) { return (int)(v * 65536.0 + 0.5); }

__device__ __forceinline__ uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

// chroma sample at output (x, y): h1v1, fancy h2v1 or fancy h2v2 (jdsample.c), from a plane of pitch pw
__device__ __forceinline__ int chroma_at(const uint8_t* p, int pw, int x, int y, int hs, int vs, int cw, int ch) {
    if (hs == 1) return p[(long long)y * pw + x];
    const int j = x >> 1;
    if (cw <= 2) return p[(long long)(vs == 2 ? y >> 1 : y) * pw + j];
    if (vs == 1) {
        const uint8_t* row = p + (long long)y * pw;
        const int v = row[j];
        if (x & 1) return j == cw - 1 ? v : (3 * v + row[j + 1] + 2) >> 2;
        return j == 0 ? v : (3 * v + row[j - 1] + 1) >> 2;
    }
    const int i = y >> 1;
    int nb = (y & 1) ? i + 1 : i - 1;
    nb = nb < 0 ? 0 : (nb > ch - 1 ? ch - 1 : nb);
    const uint8_t* r0 = p + (long long)i * pw;
    const uint8_t* r1 = p + (long long)nb * pw;
    const int cs = 3 * r0[j] + r1[j];
    if (x & 1) return j == cw - 1 ? (4 * cs + 7) >> 4 : (3 * cs + 3 * r0[j + 1] + r1[j + 1] + 7) >> 4;
    return j == 0 ? (4 * cs + 8) >> 4 : (3 * cs + 3 * r0[j - 1] + r1[j - 1] + 8) >> 4;
}

constexpr int kColorThreads = 128;

__device__ __forceinline__ void color_px(const JpegJob& job, const uint8_t* __restrict__ planes, uint8_t* __restrict__ frames,
                                         int x, int y) {
    const int pw0 = job.bw[0] * 8;
    const uint8_t* yp = planes + job.plane;
    const int Y = yp[(long long)y * pw0 + x];
    uint8_t* o = frames + job.frame + ((long long)y * job.w + x) * 3;
    if (job.ncomp == 1) {
        o[0] = o[1] = o[2] = (uint8_t)Y;
        return;
    }
    const long long psz0 = (long long)job.bw[0] * job.bh[0] * 64, psz1 = (long long)job.bw[1] * job.bh[1] * 64;
    const int pw1 = job.bw[1] * 8;
    const int cw = (job.w + job.hs - 1) / job.hs, ch = (job.h + job.vs - 1) / job.vs;
    const int cb = chroma_at(yp + psz0, pw1, x, y, job.hs, job.vs, cw, ch);
    const int cr = chroma_at(yp + psz0 + psz1, pw1, x, y, job.hs, job.vs, cw, ch);
    const int r = Y + ((fix16(1.40200) * (cr - 128) + 32768) >> 16);
    const int g = Y + ((-fix16(0.34414) * (cb - 128) + 32768 + -fix16(0.71414) * (cr - 128)) >> 16);
    const int b = Y + ((fix16(1.77200) * (cb - 128) + 32768) >> 16);
    o[0] = clamp255(r);
    o[1] = clamp255(g);
    o[2] = clamp255(b);
}

// one CTA per row of every image (one grid over the batch's rows)
__global__ void __launch_bounds__(kColorThreads) jpeg_color_kernel(const JpegJob* __restrict__ jobs, int B, const uint8_t* __restrict__ planes,
                                                                   uint8_t* __restrict__ frames, const int* __restrict__ status) {
    griddep_launch();
    griddep_wait();
    const int jb = job_of<true>(jobs, B, blockIdx.x);
    const JpegJob& job = jobs[jb];
    const int y = (int)(blockIdx.x - job.row0);
    if (job.ntab == 0 || status[jb] != RAJNI_JPEG_OK || y >= job.h) return;
    for (int x = threadIdx.x; x < job.w; x += kColorThreads) color_px(job, planes, frames, x, y);
}

// ------------------------------------------------------------------ host: header parse
static void refuse(rajni_jpeg_info* info, const char* why) {
    info->gpu = 0;
    snprintf(info->why, sizeof(info->why), "%s", why);
}

// jpeg_make_d_derived_tbl's checks: counts fit, no code is all ones, DC symbols <= 15
static bool huff_valid(const uint8_t* bits, const uint8_t* vals, bool dc) {
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        code += bits[l - 1];
        k += bits[l - 1];
        if (code >= (1 << l)) return false;
        code <<= 1;
    }
    if (k > 256) return false;
    if (dc)
        for (int i = 0; i < k; ++i)
            if (vals[i] > 15) return false;
    return true;
}

static int parse(const uint8_t* d, long long n, rajni_jpeg_info* info) {
    memset(info, 0, sizeof(*info));
    info->file_bytes = n;
    if (!d || n < 4 || d[0] != 0xFF || d[1] != 0xD8) { refuse(info, "not a JPEG (no SOI)"); return 0; }
    if (d[n - 2] != 0xFF || d[n - 1] != 0xD9) { refuse(info, "no EOI at the end (truncated?)"); return 0; }
    bool have_q[4] = {}, have_h[8] = {}, have_frame = false, jfif = false, adobe = false;
    int transform = -1, ids[3] = {};
    long long i = 2;
    for (;;) {
        while (i < n && d[i] != 0xFF) ++i;
        while (i < n && d[i] == 0xFF) ++i;
        if (i >= n) { refuse(info, "no scan before the end of the file"); return 0; }
        const int m = d[i++];
        if (m == 0xD8 || m == 0xD9) { refuse(info, "SOI/EOI before the scan"); return 0; }
        if ((m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (i + 2 > n) { refuse(info, "truncated header"); return 0; }
        const long long len = (d[i] << 8) | d[i + 1];
        if (len < 2 || i + len > n) { refuse(info, "truncated segment"); return 0; }
        const uint8_t* s = d + i + 2;
        const long long sl = len - 2;
        i += len;
        if (m == 0xC0 || m == 0xC1) {
            if (have_frame || sl < 6) { refuse(info, "bad SOF"); return 0; }
            const int h = (s[1] << 8) | s[2], w = (s[3] << 8) | s[4], nc = s[5];
            if (s[0] != 8) { refuse(info, "not 8-bit samples"); return 0; }
            if (h == 0 || w == 0 || h > kJpegMaxSide || w > kJpegMaxSide) { refuse(info, "size out of range"); return 0; }
            if ((nc != 1 && nc != 3) || sl < 6 + 3 * nc) { refuse(info, "not 1 or 3 components"); return 0; }
            int hv[3][2];
            for (int c = 0; c < nc; ++c) {
                ids[c] = s[6 + 3 * c];
                hv[c][0] = s[7 + 3 * c] >> 4;
                hv[c][1] = s[7 + 3 * c] & 15;
                info->qt[c] = s[8 + 3 * c];
                if (info->qt[c] > 3) { refuse(info, "bad quantisation table id"); return 0; }
            }
            if (nc == 1) {
                if (hv[0][0] < 1 || hv[0][0] > 4 || hv[0][1] < 1 || hv[0][1] > 4) { refuse(info, "bad sampling factor"); return 0; }
                info->h_samp = info->v_samp = 1;
            } else {
                const bool chroma11 = hv[1][0] == 1 && hv[1][1] == 1 && hv[2][0] == 1 && hv[2][1] == 1;
                const bool luma = (hv[0][0] == 1 && hv[0][1] == 1) || (hv[0][0] == 2 && hv[0][1] == 1) || (hv[0][0] == 2 && hv[0][1] == 2);
                if (!chroma11 || !luma) { refuse(info, "sampling other than 4:4:4, 4:2:2, 4:2:0"); return 0; }
                info->h_samp = hv[0][0];
                info->v_samp = hv[0][1];
            }
            info->width = w;
            info->height = h;
            info->ncomp = nc;
            have_frame = true;
        } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4 && m != 0xC8) {
            refuse(info, m == 0xCC ? "arithmetic coding" : "progressive, lossless or arithmetic frame");
            return 0;
        } else if (m == 0xDB) {
            for (long long j = 0; j < sl;) {
                const int pq = s[j] >> 4, tq = s[j] & 15, size = pq ? 128 : 64;
                if (tq > 3 || pq > 1 || j + 1 + size > sl) { refuse(info, "bad DQT"); return 0; }
                for (int k = 0; k < 64; ++k)
                    info->quant[tq][h_natural[k]] = pq ? (uint16_t)((s[j + 1 + 2 * k] << 8) | s[j + 2 + 2 * k]) : s[j + 1 + k];
                have_q[tq] = true;
                j += 1 + size;
            }
        } else if (m == 0xC4) {
            for (long long j = 0; j < sl;) {
                if (j + 17 > sl) { refuse(info, "bad DHT"); return 0; }
                const int tc = s[j] >> 4, th = s[j] & 15;
                int cnt = 0;
                for (int l = 0; l < 16; ++l) cnt += s[j + 1 + l];
                if (tc > 1 || th > 3 || cnt > 256 || j + 17 + cnt > sl) { refuse(info, "bad DHT"); return 0; }
                const int slot = tc * 4 + th;
                memcpy(info->huff_bits[slot], s + j + 1, 16);
                memset(info->huff_vals[slot], 0, 256);
                memcpy(info->huff_vals[slot], s + j + 17, cnt);
                if (!huff_valid(info->huff_bits[slot], info->huff_vals[slot], tc == 0)) { refuse(info, "bad Huffman table"); return 0; }
                have_h[slot] = true;
                j += 17 + cnt;
            }
        } else if (m == 0xDD) {
            if (sl < 2) { refuse(info, "bad DRI"); return 0; }
            info->restart_interval = (s[0] << 8) | s[1];
        } else if (m == 0xE0) {
            if (sl >= 14 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xEE) {
            if (sl >= 12 && memcmp(s, "Adobe", 5) == 0) { adobe = true; transform = s[11]; }
        } else if (m == 0xDA) {
            if (!have_frame) { refuse(info, "SOS before SOF"); return 0; }
            const int ns = sl > 0 ? s[0] : 0;
            if (ns != info->ncomp || sl < 4 + 2 * ns) { refuse(info, "the first scan does not hold every component (multi-scan)"); return 0; }
            for (int c = 0; c < ns; ++c) {
                if (s[1 + 2 * c] != ids[c]) { refuse(info, "scan component order"); return 0; }
                info->dc[c] = s[2 + 2 * c] >> 4;
                info->ac[c] = s[2 + 2 * c] & 15;
                if (info->dc[c] > 3 || info->ac[c] > 3) { refuse(info, "bad Huffman table id"); return 0; }
            }
            if (s[1 + 2 * ns] != 0 || s[2 + 2 * ns] != 63 || s[3 + 2 * ns] != 0) { refuse(info, "not a sequential scan"); return 0; }
            info->scan_offset = i;
            break;
        }
    }
    if (info->ncomp == 3) {
        bool ycc;
        if (jfif) ycc = true;
        else if (adobe) {
            if (transform != 1) { refuse(info, "Adobe RGB or unknown transform"); return 0; }
            ycc = true;
        } else {
            ycc = !(ids[0] == 'R' && ids[1] == 'G' && ids[2] == 'B');
        }
        if (!ycc) { refuse(info, "RGB components"); return 0; }
    }
    for (int c = 0; c < info->ncomp; ++c)
        if (!have_q[info->qt[c]] || !have_h[info->dc[c]] || !have_h[4 + info->ac[c]]) {
            refuse(info, "a table the scan uses is not defined");
            return 0;
        }
    info->gpu = 1;
    return 1;
}

// ------------------------------------------------------------------ host: jobs and workspace
struct Layout {
    int bw[3], bh[3], mcux, mcuy;
    long long blocks;
};

static Layout layout_of(const rajni_jpeg_info& in) {
    Layout L{};
    if (in.ncomp == 1) {
        L.bw[0] = L.mcux = (in.width + 7) / 8;
        L.bh[0] = L.mcuy = (in.height + 7) / 8;
    } else {
        L.mcux = (in.width + 8 * in.h_samp - 1) / (8 * in.h_samp);
        L.mcuy = (in.height + 8 * in.v_samp - 1) / (8 * in.v_samp);
        L.bw[0] = L.mcux * in.h_samp;
        L.bh[0] = L.mcuy * in.v_samp;
        L.bw[1] = L.bw[2] = L.mcux;
        L.bh[1] = L.bh[2] = L.mcuy;
    }
    for (int c = 0; c < in.ncomp; ++c) L.blocks += (long long)L.bw[c] * L.bh[c];
    return L;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// workspace: status[B] | jobs[B] | tables | coefficients (int16) | planes (uint8)
struct WsPlan {
    size_t jobs, tabs, coef, planes, total;
    long long ntabs, blocks;
};

static WsPlan plan_of(const rajni_jpeg_info* infos, int B) {
    WsPlan p{};
    for (int b = 0; b < B; ++b) {
        if (!infos[b].gpu) continue;
        const Layout L = layout_of(infos[b]);
        p.blocks += L.blocks;
        p.ntabs += kMaxTabs;
    }
    p.jobs = align256((size_t)B * sizeof(int));
    p.tabs = p.jobs + align256((size_t)B * sizeof(JpegJob));
    p.coef = p.tabs + align256((size_t)p.ntabs * sizeof(HuffDev));
    p.planes = p.coef + align256((size_t)p.blocks * 128);
    p.total = p.planes + align256((size_t)p.blocks * 64);
    return p;
}

// jpeg_make_d_derived_tbl for the device layout
static void build_huff(const uint8_t* bits, const uint8_t* vals, HuffDev* t) {
    memset(t, 0, sizeof(*t));
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        t->maxcode[l] = -1;
        if (bits[l - 1]) {
            t->valoff[l] = k - code;
            for (int i = 0; i < bits[l - 1]; ++i, ++code, ++k)
                if (l <= kLutBits) {
                    const int lo = code << (kLutBits - l), hi = (code + 1) << (kLutBits - l);
                    for (int e = lo; e < hi; ++e) t->lut[e] = (uint16_t)((l << 8) | vals[k]);
                }
            t->maxcode[l] = code - 1;
        }
        code <<= 1;
    }
    t->maxcode[17] = 0x7fffffff;
    memcpy(t->vals, vals, 256);
}

}  // namespace rajni

using namespace rajni;

extern "C" int rajni_jpeg_version(void) { return RAJNI_JPEG_VERSION; }

extern "C" const char* rajni_jpeg_last_error(void) { return error_text(); }

extern "C" int rajni_jpeg_parse(const void* data_host, long long nbytes, rajni_jpeg_info* info) {
    if (!info) return 0;
    return parse(static_cast<const uint8_t*>(data_host), nbytes, info);
}

extern "C" size_t rajni_jpeg_workspace_bytes(const rajni_jpeg_info* infos_host, int B) {
    if (!infos_host || B <= 0) return 0;
    return plan_of(infos_host, B).total;
}

extern "C" int rajni_jpeg_decode(const void* files, const long long* file_offsets_host, const rajni_jpeg_info* infos_host, int B,
                                 void* frames, const long long* frame_offsets_host, void* workspace, size_t workspace_bytes,
                                 void* stream) {
    RAJNI_REQUIRE(files && file_offsets_host && infos_host && frames && frame_offsets_host && workspace, RAJNI_EINVAL,
                  "rajni_jpeg_decode: null pointer");
    RAJNI_REQUIRE(B > 0 && B <= 65535, RAJNI_EINVAL, "rajni_jpeg_decode: B=%d", B);
    RAJNI_REQUIRE((reinterpret_cast<uintptr_t>(files) & 7) == 0, RAJNI_EINVAL, "rajni_jpeg_decode: files must be 8-byte aligned");
    const WsPlan P = plan_of(infos_host, B);
    RAJNI_REQUIRE(workspace_bytes >= P.total, RAJNI_EINVAL, "rajni_jpeg_decode: workspace of %zu B, need %zu B", workspace_bytes, P.total);
    // host image of status | jobs | tables, one copy
    std::vector<uint8_t> host(P.coef, 0);
    int* st = reinterpret_cast<int*>(host.data());
    JpegJob* jobs = reinterpret_cast<JpegJob*>(host.data() + P.jobs);
    HuffDev* tabs = reinterpret_cast<HuffDev*>(host.data() + P.tabs);
    int tab = 0;
    long long coef = 0, plane = 0, idct_ctas = 0, rows = 0;
    for (int b = 0; b < B; ++b) {
        const rajni_jpeg_info& in = infos_host[b];
        JpegJob& j = jobs[b];
        j.idct0 = idct_ctas;
        j.row0 = rows;
        st[b] = RAJNI_JPEG_SKIPPED;
        if (!in.gpu) continue;
        RAJNI_REQUIRE(in.width >= 1 && in.width <= kJpegMaxSide && in.height >= 1 && in.height <= kJpegMaxSide &&
                      (in.ncomp == 1 || in.ncomp == 3) && in.scan_offset > 0 && in.scan_offset <= in.file_bytes,
                      RAJNI_EINVAL, "rajni_jpeg_decode: info %d was not filled by rajni_jpeg_parse", b);
        st[b] = RAJNI_JPEG_OK;
        const Layout L = layout_of(in);
        j.src = file_offsets_host[b] + in.scan_offset;
        j.src_end = file_offsets_host[b] + in.file_bytes;
        j.coef = coef;
        j.plane = plane;
        j.frame = frame_offsets_host[b];
        j.w = in.width;
        j.h = in.height;
        j.ncomp = in.ncomp;
        j.hs = in.h_samp;
        j.vs = in.v_samp;
        j.mcux = L.mcux;
        j.mcuy = L.mcuy;
        j.restart = in.restart_interval;
        j.tab0 = tab;
        int slots[8];
        for (int s = 0; s < 8; ++s) slots[s] = -1;
        for (int c = 0; c < in.ncomp; ++c) {
            j.bw[c] = L.bw[c];
            j.bh[c] = L.bh[c];
            const int want[2] = {in.dc[c], 4 + in.ac[c]};
            for (int w = 0; w < 2; ++w) {
                if (slots[want[w]] < 0) {
                    slots[want[w]] = j.ntab++;
                    build_huff(in.huff_bits[want[w]], in.huff_vals[want[w]], &tabs[tab + slots[want[w]]]);
                }
            }
            j.dc[c] = slots[want[0]];
            j.ac[c] = slots[want[1]];
            for (int k = 0; k < 64; ++k) j.q[c][k] = in.quant[in.qt[c]][k];
        }
        tab += kMaxTabs;
        coef += L.blocks * 64;
        plane += L.blocks * 64;
        idct_ctas += (L.blocks + kIdctBlocks - 1) / kIdctBlocks;
        rows += in.height;
    }
    auto s = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    cudaError_t e = cudaMemcpyAsync(ws, host.data(), host.size(), cudaMemcpyHostToDevice, s);
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "rajni_jpeg_decode: table copy: %s", cudaGetErrorString(e));
    e = cudaMemsetAsync(ws + P.coef, 0, P.planes - P.coef, s);       // jpeg_huffman stores only nonzero coefficients
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "rajni_jpeg_decode: coefficient memset: %s", cudaGetErrorString(e));
    if (P.blocks == 0) return RAJNI_OK;
    const JpegJob* djobs = reinterpret_cast<const JpegJob*>(ws + P.jobs);
    int* dstatus = reinterpret_cast<int*>(ws);
    int16_t* dcoef = reinterpret_cast<int16_t*>(ws + P.coef);
    uint8_t* dplanes = ws + P.planes;
    if (int rc = launch_checked("jpeg_huffman", jpeg_huffman_kernel, dim3(B), dim3(kHuffThreads), 0, s, 1,
                                static_cast<const uint8_t*>(files), djobs, reinterpret_cast<const HuffDev*>(ws + P.tabs), dcoef, dstatus))
        return rc;
    RAJNI_REQUIRE(idct_ctas <= 0x7fffffffLL && rows <= 0x7fffffffLL, RAJNI_EINVAL, "rajni_jpeg_decode: batch too large");
    if (int rc = launch_checked("jpeg_idct", jpeg_idct_kernel, dim3((unsigned)idct_ctas), dim3(kIdctBlocks * 8), 0, s, 1,
                                djobs, B, static_cast<const int16_t*>(dcoef), dplanes, static_cast<const int*>(dstatus)))
        return rc;
    return launch_checked("jpeg_color", jpeg_color_kernel, dim3((unsigned)rows), dim3(kColorThreads), 0, s, 1, djobs, B,
                          static_cast<const uint8_t*>(dplanes),
                          static_cast<uint8_t*>(frames), static_cast<const int*>(dstatus));
}

extern "C" int rajni_jpeg_status(const void* workspace, int B, int* status_host, void* stream) {
    RAJNI_REQUIRE(workspace && status_host && B > 0, RAJNI_EINVAL, "rajni_jpeg_status: null pointer or B=%d", B);
    auto s = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemcpyAsync(status_host, workspace, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "rajni_jpeg_status: %s", cudaGetErrorString(e));
    return RAJNI_OK;
}
