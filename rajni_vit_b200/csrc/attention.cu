// a4: C-ABI entry of the attention over kept tokens (attention.py:42-54) and its dispatch to the three tcgen05 kernels.
//
//   128 < Np, Np_pad <= 224        : attention_pipe.cu  (role-pipelined: exp / epilogue / MMA / load warps, S multi-buffered in
//                                    TMEM, half rows of S held in registers): 1.2-1.26x the kernel below at 152..197 tokens and
//                                    batch 256, 1.35-1.5x at 16..64 images, dense or gathered; never slower down to 4 images
//   64 < Np <= 128, dense, >= 1 (image, head) item per SM,
//                or gathered, <= 4 items per SM : attention_pipe.cu, one-tile items: whole rows per thread, the two exp warps of
//                                    a scheduler on alternate tiles (dense 87 tokens at batch 256: 43.5 -> 30.8 us; gathered calls
//                                    of the 32..64-image shards 1.05-1.2x; at 20 items per SM the gathered load is the bound and
//                                    the kernel below, with 7 loader warps against 3, wins by 3-8 %)
//   other Np <= 256                : attention_tc.cu    (two score tiles of 256 columns at once; <= 64 tokens - it packs several
//                                    images into a tile -, large gathered one-tile launches, Np_pad > 224).  The two agree bit
//                                    for bit.  (profiles/r2_attention_pipe.md, r2_attention_fullrow_ab.txt)
//   else                           : attention_long.cu  (key blocks of 224, two passes; the 577-token configuration)
//
// RAJNI_ATTN_TC=1 sends every Np <= 256 call to attention_tc.cu, RAJNI_ATTN_PIPE=1 every Np_pad <= 224 call to
// attention_pipe.cu (A/B timing; the tests run both).
#include <cstdlib>

#include "common.cuh"

namespace rajni {
int launch_attention_pipe(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                          int C, int H, float scale, int reverse, cudaStream_t stream);      // attention_pipe.cu
int launch_attention_tc(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                        int C, int H, float scale, int reverse, cudaStream_t stream);        // attention_tc.cu
int launch_attention_long(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np,
                          int C, int H, float scale, int reverse, cudaStream_t stream);      // attention_long.cu
}  // namespace rajni

using namespace rajni;

static int attention_dispatch(const void* qkv, const int32_t* row_map, void* out, int B, int N_src, int Np, int C, int H,
                              float scale, int reverse, int impl, cudaStream_t st) {
    RAJNI_REQUIRE(qkv && out, RAJNI_EINVAL, "rajni_attention_fwd: null pointer");
    RAJNI_REQUIRE(B > 0 && Np > 0 && N_src >= Np && H > 0 && C == H * 64, RAJNI_EINVAL,
                  "rajni_attention_fwd: B=%d N_src=%d Np=%d C=%d H=%d (head dim must be 64)", B, N_src, Np, C, H);
    RAJNI_REQUIRE(row_map || N_src == Np, RAJNI_EINVAL, "rajni_attention_fwd: N_src != Np needs a row_map");
    RAJNI_REQUIRE(impl >= RAJNI_ATTN_AUTO && impl <= RAJNI_ATTN_LONG, RAJNI_EINVAL, "rajni_attention_fwd_ex: impl %d", impl);
    if (impl == RAJNI_ATTN_AUTO) {
        static const bool force_tc = getenv("RAJNI_ATTN_TC") != nullptr, force_pipe = getenv("RAJNI_ATTN_PIPE") != nullptr;
        const int np_pad = (Np + 15) & ~15;
        const int sms = num_sms();
        const long long items = (long long)B * H;
        const bool big = Np > 128;
        const bool one_tile = Np > 64 && Np <= 128 && (row_map == nullptr ? items >= sms : items <= 4LL * sms);
        if (np_pad <= 224 && (force_pipe || (!force_tc && (big || one_tile)))) impl = RAJNI_ATTN_PIPE;
        else impl = Np <= 256 ? RAJNI_ATTN_TC : RAJNI_ATTN_LONG;
    }
    int rc = 0;
    if (impl == RAJNI_ATTN_PIPE) rc = launch_attention_pipe(qkv, row_map, out, B, N_src, Np, C, H, scale, reverse, st);
    else if (impl == RAJNI_ATTN_TC) rc = launch_attention_tc(qkv, row_map, out, B, N_src, Np, C, H, scale, reverse, st);
    else rc = launch_attention_long(qkv, row_map, out, B, N_src, Np, C, H, scale, reverse, st);
    if (rc == 0) {
        set_error("rajni_attention_fwd: kernel %d does not cover Np=%d", impl, Np);
        return RAJNI_EINVAL;
    }
    return rc < 0 ? rc : RAJNI_OK;
}

extern "C" int rajni_attention_fwd(const void* qkv, const int32_t* row_map, void* out,
                                   int B, int N_src, int Np, int C, int H, float scale, int reverse, void* stream) {
    return attention_dispatch(qkv, row_map, out, B, N_src, Np, C, H, scale, reverse, RAJNI_ATTN_AUTO, static_cast<cudaStream_t>(stream));
}

extern "C" int rajni_attention_fwd_ex(const void* qkv, const int32_t* row_map, void* out,
                                      int B, int N_src, int Np, int C, int H, float scale, int reverse, int impl, void* stream) {
    return attention_dispatch(qkv, row_map, out, B, N_src, Np, C, H, scale, reverse, impl, static_cast<cudaStream_t>(stream));
}
