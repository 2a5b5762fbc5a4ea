// f3 (SURVEY 8f): the loader's Resize(256, bicubic) + CenterCrop(224) on the GPU, bit-identical to torchvision on PIL images.
//
//   transforms.Resize(256, interpolation=3) -> transforms.CenterCrop(224)           rajni/run.py:62-66
//
// The arithmetic is Pillow's (libImaging/Resample.c, restated and pinned in oracle/resize_oracle.py): separable resampling
// with an antialiasing bicubic window (support = 2 * max(scale, 1), a = -0.5), weights normalised in double and rounded to
// 22-bit fixed point, a HORIZONTAL pass to a uint8 temporary and a VERTICAL pass, each  clip8(((1 << 21) + sum p*k) >> 22).
// Output size and crop window are torchvision's (shorter edge -> 256, longer -> int(256*long/short); round-half-even origin).
// Only the crop's 224 columns / rows are ever computed.
//
// Three launches per batch of decoded uint8 HWC frames of arbitrary sizes (concatenated in one device buffer):
//   resize_plan_kernel   one CTA per image: window bounds + integer weights of the 224 columns and 224 rows, in DOUBLE with
//                        explicitly unfused multiplies/adds (the weights must match the CPU's to the last bit)
//   resize_h_kernel      temp[b][r][xx][c] for the source rows the crop needs            (HBM-bound: reads the frames once)
//   resize_v_kernel      out[b][c][yy][xx] uint8 planar - the tensor PILToTensor would give; the patch kernel then applies
//                        ToTensor + Normalize in fp32 (rajni_patch_im2col_prefix, RAJNI_IMG_U8)
#include "common.cuh"

namespace rajni {

constexpr int kRsPrecision = 32 - 8 - 2;      // Pillow PRECISION_BITS
constexpr int kRsMaxTaps = 96;                // ceil(2*scale)*2+1 <= 96: downscales up to ~23x (shorter edge up to ~6000 px)
constexpr int kRsCrop = 224;

struct ResizePlan {            // per image, in the workspace
    int r0, rows;              // first source row the crop needs, and how many
    int w, h;
    int kh_n, kv_n;            // taps per output column / row
};

// Pillow's bicubic_filter, a = -0.5, every operation rounded separately (x86-64 wheels have no FMA contraction)
__device__ __forceinline__ double rs_bicubic(double x) {
    if (x < 0.0) x = -x;
    if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dadd_rn(__dmul_rn(1.5, x), -2.5), x), x), 1.0);
    if (x < 2.0) return __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(x, -5.0), x), 8.0), x), -4.0), -0.5);
    return 0.0;
}

// precompute_coeffs + normalize_coeffs_8bpc for one output position xx: bounds (xmin, n) and n integer weights
__device__ void rs_coeffs(int in_size, int out_size, int xx, int* bounds, int* kk) {
    const double scale = __ddiv_rn((double)in_size, (double)out_size);
    const double filterscale = scale < 1.0 ? 1.0 : scale;
    const double support = __dmul_rn(2.0, filterscale);
    const double ss = __ddiv_rn(1.0, filterscale);
    const double center = __dmul_rn(__dadd_rn((double)xx, 0.5), scale);
    int xmin = (int)__dadd_rn(__dadd_rn(center, -support), 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)__dadd_rn(__dadd_rn(center, support), 0.5);
    if (xmax > in_size) xmax = in_size;
    const int n = xmax - xmin;
    double ww = 0.0;
    for (int x = 0; x < n; ++x)
        ww = __dadd_rn(ww, rs_bicubic(__dmul_rn(__dadd_rn(__dadd_rn((double)(x + xmin), -center), 0.5), ss)));
    for (int x = 0; x < n; ++x) {
        double v = rs_bicubic(__dmul_rn(__dadd_rn(__dadd_rn((double)(x + xmin), -center), 0.5), ss));
        if (ww != 0.0) v = __ddiv_rn(v, ww);
        const double f = __dmul_rn(v, (double)(1 << kRsPrecision));
        kk[x] = v < 0 ? (int)__dadd_rn(-0.5, f) : (int)__dadd_rn(0.5, f);
    }
    bounds[0] = xmin;
    bounds[1] = n;
}

// workspace layout per image: ResizePlan | bh[224][2] | bv[224][2] | kh[224][kRsMaxTaps] | kv[224][kRsMaxTaps] | temp rows
__host__ __device__ inline size_t rs_tables_bytes() {
    return 64 + 2 * kRsCrop * 2 * sizeof(int) + 2 * (size_t)kRsCrop * kRsMaxTaps * sizeof(int);
}
__host__ __device__ inline size_t rs_image_bytes(int max_h) {
    return (rs_tables_bytes() + (size_t)max_h * kRsCrop * 3 + 255) & ~(size_t)255;
}

__global__ void __launch_bounds__(2 * kRsCrop) resize_plan_kernel(const long long* __restrict__ meta, int size, uint8_t* ws, int max_h, int* err) {
    griddep_launch();
    griddep_wait();
    const int b = blockIdx.x, t = threadIdx.x;
    const int h = (int)meta[b * 3 + 1], w = (int)meta[b * 3 + 2];
    uint8_t* base = ws + (size_t)b * rs_image_bytes(max_h);
    ResizePlan* plan = reinterpret_cast<ResizePlan*>(base);
    int* bh = reinterpret_cast<int*>(base + 64);
    int* bv = bh + kRsCrop * 2;
    int* kh = bv + kRsCrop * 2;
    int* kv = kh + kRsCrop * kRsMaxTaps;
    // torchvision _compute_resized_output_size (int(size * long / short)) and center_crop (round half to even)
    const int shrt = w <= h ? w : h, lng = w <= h ? h : w;
    const int new_long = (int)__ddiv_rn((double)((long long)size * lng), (double)shrt);
    const int nw = w <= h ? size : new_long, nh = w <= h ? new_long : size;
    const int dy = nh - kRsCrop, dx = nw - kRsCrop;
    const int top = (dy >> 1) + ((dy & 1) & (dy >> 1)), left = (dx >> 1) + ((dx & 1) & (dx >> 1));
    const int kh_n = (int)ceil(2.0 * fmax((double)w / nw, 1.0)) * 2 + 1, kv_n = (int)ceil(2.0 * fmax((double)h / nh, 1.0)) * 2 + 1;
    if (h < 1 || w < 1 || dy < 0 || dx < 0 || kh_n > kRsMaxTaps || kv_n > kRsMaxTaps || h > max_h) {
        if (t == 0) {
            atomicExch(err, 1 + b);
            plan->r0 = 0;
            plan->rows = 0;           // the two passes skip this frame
        }
        return;
    }
    if (t < kRsCrop) rs_coeffs(w, nw, left + t, bh + t * 2, kh + t * kRsMaxTaps);
    else rs_coeffs(h, nh, top + (t - kRsCrop), bv + (t - kRsCrop) * 2, kv + (t - kRsCrop) * kRsMaxTaps);
    __syncthreads();
    if (t == 0) {
        plan->r0 = bv[0];
        plan->rows = bv[(kRsCrop - 1) * 2] + bv[(kRsCrop - 1) * 2 + 1] - bv[0];
        plan->w = w; plan->h = h; plan->kh_n = kh_n; plan->kv_n = kv_n;
    }
}

__device__ __forceinline__ uint8_t rs_clip8(int v) {
    v >>= kRsPrecision;
    return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
}

// one CTA = one temporary row of one image; thread = crop column
__global__ void __launch_bounds__(kRsCrop) resize_h_kernel(const uint8_t* __restrict__ src, const long long* __restrict__ meta,
                                                           uint8_t* ws, int max_h) {
    griddep_launch();
    griddep_wait();
    const int b = blockIdx.y, xx = threadIdx.x;
    uint8_t* base = ws + (size_t)b * rs_image_bytes(max_h);
    const ResizePlan* plan = reinterpret_cast<const ResizePlan*>(base);
    const int r = blockIdx.x;
    if (r >= plan->rows) return;
    const int* bh = reinterpret_cast<const int*>(base + 64);
    const int* kh = bh + 4 * kRsCrop + xx * kRsMaxTaps;
    const int xmin = bh[xx * 2], n = bh[xx * 2 + 1];
    const uint8_t* row = src + meta[b * 3] + ((size_t)(plan->r0 + r) * plan->w + xmin) * 3;
    int s0 = 1 << (kRsPrecision - 1), s1 = s0, s2 = s0;
    for (int x = 0; x < n; ++x) {
        const int k = kh[x];
        s0 += row[3 * x] * k;
        s1 += row[3 * x + 1] * k;
        s2 += row[3 * x + 2] * k;
    }
    uint8_t* tmp = base + rs_tables_bytes() + ((size_t)r * kRsCrop + xx) * 3;
    tmp[0] = rs_clip8(s0);
    tmp[1] = rs_clip8(s1);
    tmp[2] = rs_clip8(s2);
}

// one CTA = one output row of one image; thread = crop column; planar uint8 output
__global__ void __launch_bounds__(kRsCrop) resize_v_kernel(uint8_t* ws, int max_h, uint8_t* __restrict__ out) {
    griddep_launch();
    griddep_wait();
    const int b = blockIdx.y, yy = blockIdx.x, xx = threadIdx.x;
    const uint8_t* base = ws + (size_t)b * rs_image_bytes(max_h);
    const ResizePlan* plan = reinterpret_cast<const ResizePlan*>(base);
    const int* bv = reinterpret_cast<const int*>(base + 64) + 2 * kRsCrop;
    const int* kv = reinterpret_cast<const int*>(base + 64) + 4 * kRsCrop + kRsCrop * kRsMaxTaps + yy * kRsMaxTaps;
    if (plan->rows == 0) return;
    const int y0 = bv[yy * 2] - plan->r0, n = bv[yy * 2 + 1];
    const uint8_t* tmp = base + rs_tables_bytes() + ((size_t)y0 * kRsCrop + xx) * 3;
    int s0 = 1 << (kRsPrecision - 1), s1 = s0, s2 = s0;
    for (int y = 0; y < n; ++y) {
        const int k = kv[y];
        const uint8_t* px = tmp + (size_t)y * kRsCrop * 3;
        s0 += px[0] * k;
        s1 += px[1] * k;
        s2 += px[2] * k;
    }
    uint8_t* o = out + ((size_t)b * 3 * kRsCrop + yy) * kRsCrop + xx;
    o[0] = rs_clip8(s0);
    o[(size_t)kRsCrop * kRsCrop] = rs_clip8(s1);
    o[(size_t)2 * kRsCrop * kRsCrop] = rs_clip8(s2);
}

}  // namespace rajni

using namespace rajni;

extern "C" size_t rajni_resize_workspace_bytes(int B, int max_h) {
    if (B <= 0 || max_h <= 0) return 0;
    return (size_t)B * rs_image_bytes(max_h) + 256;
}

extern "C" int rajni_resize_center_crop_u8(const void* frames, const long long* meta, int B, int max_h, int size, int crop,
                                           void* out, void* workspace, size_t workspace_bytes, void* stream) {
    RAJNI_REQUIRE(frames && meta && out && workspace, RAJNI_EINVAL, "rajni_resize_center_crop_u8: null pointer");
    RAJNI_REQUIRE(B > 0 && max_h > 0, RAJNI_EINVAL, "rajni_resize_center_crop_u8: B=%d max_h=%d", B, max_h);
    RAJNI_REQUIRE(crop == kRsCrop && size >= crop, RAJNI_EINVAL,
                  "rajni_resize_center_crop_u8: crop must be %d and size >= crop (got size=%d crop=%d)", kRsCrop, size, crop);
    RAJNI_REQUIRE(workspace_bytes >= rajni_resize_workspace_bytes(B, max_h), RAJNI_EINVAL,
                  "rajni_resize_center_crop_u8: workspace of %zu B, need %zu B", workspace_bytes, rajni_resize_workspace_bytes(B, max_h));
    RAJNI_REQUIRE(B <= 65535, RAJNI_EINVAL, "rajni_resize_center_crop_u8: B exceeds the grid limit");
    auto st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    int* err = reinterpret_cast<int*>(ws + (size_t)B * rs_image_bytes(max_h));
    cudaError_t e = cudaMemsetAsync(err, 0, sizeof(int), st);
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "rajni_resize_center_crop_u8: memset: %s", cudaGetErrorString(e));
    if (int rc = launch_checked("resize_plan", resize_plan_kernel, dim3(B), dim3(2 * kRsCrop), 0, st, 1, meta, size, ws, max_h, err))
        return rc;
    if (int rc = launch_checked("resize_h", resize_h_kernel, dim3(max_h, B), dim3(kRsCrop), 0, st, 1,
                                static_cast<const uint8_t*>(frames), meta, ws, max_h))
        return rc;
    return launch_checked("resize_v", resize_v_kernel, dim3(kRsCrop, B), dim3(kRsCrop), 0, st, 1, ws, max_h, static_cast<uint8_t*>(out));
}

/* 0 if every frame of the last call on this workspace was resized; 1 + the index of a frame that was rejected (smaller than
 * the crop after resizing, taller than max_h, or a downscale beyond kRsMaxTaps taps).  Reads device memory: synchronises. */
extern "C" int rajni_resize_status(const void* workspace, int B, int max_h, void* stream) {
    int v = 0;
    const uint8_t* ws = static_cast<const uint8_t*>(workspace);
    cudaError_t e = cudaMemcpyAsync(&v, ws + (size_t)B * rs_image_bytes(max_h), sizeof(int), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
    RAJNI_REQUIRE(e == cudaSuccess, RAJNI_ECUDA, "rajni_resize_status: %s", cudaGetErrorString(e));
    return v;
}
