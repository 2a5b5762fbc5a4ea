/*
 * rajni_b200.h — C ABI of the B200-native RAJNI token-pruning forward path.
 *
 * This is the drop-in boundary: everything the reference computes inside
 * RAJNIViTWrapper.forward (rajni/wrapper/model.py:30-69), RAJNIAttention.forward
 * (rajni/wrapper/attention.py:17-60) and compute_importance
 * (rajni/wrapper/importance.py:5-34) is reachable through these entry points.
 * The reference itself has no native layer (it is eager PyTorch); a maintainer
 * binds this library with ctypes as shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - activations and weights are bf16, row-major; bias / LayerNorm affine /
 *     scores are fp32; indices are int32;
 *   - `stream` is a cudaStream_t passed as void*; no call synchronises, allocates
 *     device memory, or touches the host beyond launching kernels;
 *   - return 0 on success, a negative RAJNI_E* code otherwise; the message is
 *     available from rajni_last_error() (thread-local);
 *   - sm_100a only. There is no CPU path and no fallback.
 */
#ifndef RAJNI_B200_H
#define RAJNI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAJNI_ABI_VERSION 10     /* 10: rajni_patch_im2col takes any patch that is a multiple of 8; long-sequence scores */

enum {
    RAJNI_OK = 0,
    RAJNI_EINVAL = -1,   /* bad shape / null pointer / unsupported size          */
    RAJNI_ECUDA = -2,    /* a CUDA runtime or driver call failed                 */
    RAJNI_EARCH = -3,    /* current device is not compute capability 10.x        */
    RAJNI_ERANGE = -4    /* keep > N-1: the reference's topk raises here         */
};

/* epilogue flags for rajni_gemm_bf16 */
enum {
    RAJNI_EPI_BIAS = 1,       /* + bias[n]                                       */
    RAJNI_EPI_GELU = 2,       /* exact erf GELU (timm nn.GELU) after bias        */
    RAJNI_EPI_RESIDUAL = 4,   /* + residual[res_row(m), n] after activation      */
    RAJNI_EPI_OUT_F32 = 8,    /* store fp32 instead of bf16                      */
    RAJNI_EPI_LN_FOLD = 16,   /* A is the UN-normalised x; apply LayerNorm algebraically (see below)  */
    RAJNI_EPI_ROW_STATS = 32, /* also emit per-row partial (sum, sum of squares) of the stored values */
    RAJNI_HINT_REVERSE_M = 64,/* walk the M tiles last-to-first: a consumer that starts where its producer
                                 finished finds those rows still in the 126 MB L2. Results are identical.   */
    RAJNI_HINT_STREAM_K = 128 /* with a workspace: split the leftover tiles of the last wave along K wherever that is
                                 possible, not only where the cost model expects a gain (tests, A/B timing).   */
};

int rajni_abi_version(void);
const char* rajni_last_error(void);
/* 0 if the current CUDA device can run this library (cc 10.x), else RAJNI_EARCH. */
int rajni_device_check(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches). */
uint64_t rajni_launch_count(void);

/* ---- a1: compute_importance (rajni/wrapper/importance.py:5-34) ------------------
 * qkv [B,N,3C] bf16 with the last dim laid out (3,H,D); scores [B,N] fp32.
 * bf16 tiles in, fp32 arithmetic (SURVEY.md section 4.5). D must be 64. */
int rajni_importance(const void* qkv, int B, int N, int C, int H, float eps,
                     float* scores, void* stream);

/* ---- a2: token selection (rajni/wrapper/attention.py:31-39) and score carry (:58)
 * Top-`keep` of scores[:,1:] -> keep_idx [B,keep+1] int32, strictly ascending,
 * keep_idx[:,0]==0. Tie rule: greater score first, then lower index.
 * next_scores [B,keep+1] = scores[keep_idx]. row_map [B*(keep+1)] = b*N+keep_idx
 * (global row of each kept token; nullable). keep > N-1 -> RAJNI_ERANGE. */
int rajni_select(const float* scores, int B, int N, int keep,
                 int32_t* keep_idx, float* next_scores, int32_t* row_map, void* stream);
/* The same with `prefix` (1 or 2) leading tokens that are always kept: CLS, or CLS and a distillation token.
 * Top-`keep` of scores[:,prefix:] -> keep_idx [B,keep+prefix] int32, strictly ascending, keep_idx[:,r]==r for
 * r < prefix; next_scores and row_map [B*(keep+prefix)] as above.  keep > N-prefix -> RAJNI_ERANGE.
 * rajni_select is this call with prefix 1. */
int rajni_select_prefix(const float* scores, int B, int N, int prefix, int keep,
                        int32_t* keep_idx, float* next_scores, int32_t* row_map, void* stream);

/* ---- a1+a2 fused: one pass over the K and V planes, then in-CTA select.
 * scores may be NULL when the caller does not need the full score vector.
 * rajni_importance and rajni_score_select keep one image's CLS logits and value rows in shared memory; shapes for which
 * rajni_score_select_needs_workspace(N, H) is 1 (N > ~720 at 12 heads) return RAJNI_EINVAL there: use the split entry. */
int rajni_score_select(const void* qkv, int B, int N, int C, int H, int keep, float eps,
                       float* scores, int32_t* keep_idx, float* next_scores,
                       int32_t* row_map, void* stream);

/* Same result, bit for bit, in two launches for batches with far fewer images than the GPU has SMs (one CTA per image
 * would leave most SMs idle): the K/V pass is spread over (image, 16-row block) CTAs into `workspace`
 * (rajni_score_select_workspace_bytes(B,N,C,H) bytes, 16-byte aligned, caller-owned), then the per-image kernel finishes.
 * Every N <= 4096 works here at any batch: when rajni_score_select_needs_workspace(N, H) is 1 the per-image kernel reads
 * the logits and value rows from the workspace in place (same arithmetic, same bits).  keep_idx == NULL computes the
 * scores only (a scores-only call of rajni_importance's meaning): then `scores` is required, keep, next_scores and
 * row_map are ignored. */
size_t rajni_score_select_workspace_bytes(int B, int N, int C, int H);
/* Host-side query, no launch: 1 when one image of N tokens and H heads needs the workspace path of
 * rajni_score_select_split (its CLS logits and value rows exceed the per-image kernel's shared memory), else 0. */
int rajni_score_select_needs_workspace(int N, int H);
int rajni_score_select_split(const void* qkv, int B, int N, int C, int H, int keep, float eps,
                             float* scores, int32_t* keep_idx, float* next_scores, int32_t* row_map,
                             void* workspace, size_t workspace_bytes, void* stream);
/* Both of the above with `prefix` (1 or 2) always-kept leading tokens, selection as in rajni_select_prefix.  The scores do
 * not depend on it: the query is row 0 (CLS), every token (a distillation token too) is a key and value and enters the
 * value-norm statistics.  workspace == NULL: rajni_score_select's one-launch kernel; else rajni_score_select_split's two
 * launches (same bits).  keep_idx == NULL computes the scores only.  rajni_score_select and rajni_score_select_split are
 * this call with prefix 1. */
int rajni_score_select_prefix(const void* qkv, int B, int N, int C, int H, int prefix, int keep, float eps,
                              float* scores, int32_t* keep_idx, float* next_scores, int32_t* row_map,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- a3 / a9: row gather-compaction (attention.py:42-43, model.py:55-56)
 * dst[r, :] = src[row_map[r], :], rows of `row_elems` bf16 (multiple of 8). */
int rajni_gather_rows(const void* src, const int32_t* row_map, void* dst,
                      int rows_out, int row_elems, void* stream);

/* ---- LayerNorm over the last dim (model.py:51,59,65), bf16 -> bf16, fp32 math.
 * Row r is read at x + r*in_row_stride elements (lets the final norm touch CLS
 * rows only) and written densely at y + r*C. C multiple of 8, C <= 4096. */
int rajni_layernorm(const void* x, long long in_row_stride, const float* gamma,
                    const float* beta, float eps, void* y, int rows, int C, void* stream);
/* The same with row r written at y + r*out_row_stride (>= C, multiple of 8): two calls with out_row_stride 2C put the
 * normalised CLS and distillation rows of each image side by side, the A operand of a distilled model's head. */
int rajni_layernorm_strided(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                            void* y, long long out_row_stride, int rows, int C, void* stream);
/* The same values stored as fp32 (the features of a headless model, num_classes = 0): y + r*out_row_stride floats,
 * out_row_stride >= C and a multiple of 4.  bf16_rn of each value is what rajni_layernorm_strided stores. */
int rajni_layernorm_strided_f32(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                                float* y, long long out_row_stride, int rows, int C, void* stream);
/* The same over a whole activation matrix, also emitting the rows' LayerNorm partial sums for an LN-folded GEMM
 * (RAJNI_EPI_LN_FOLD) that reads y next: row_stats[s*row_stats_ld + r] = (sum, sum of squares) of the bf16 row r as stored
 * for s = 0, zero for s = 1..stats_slots-1 (the slot layout of RAJNI_EPI_ROW_STATS).  y may be x (in place).  This is the
 * pre-norm stem of CLIP ViTs (timm's norm_pre), applied to the embedded tokens before block 0.  C <= 2048. */
int rajni_layernorm_row_stats(const void* x, long long in_row_stride, const float* gamma, const float* beta, float eps,
                              void* y, long long out_row_stride, int rows, int C,
                              float* row_stats, long long row_stats_ld, int stats_slots, void* stream);

/* ---- average-pooled head (timm global_pool='avg' with fc_norm: MAE fine-tuned ViTs)
 * y[b*out_row_stride + c] = LN(mean_{n = prefix..N-1} x[b*N + n, :])[c] in bf16, x [B*N, C] bf16 dense, gamma / beta fp32
 * [C].  The mean is an fp32 sum of the bf16 rows divided by N - prefix (the patch tokens; prefix 1 or 2), the LayerNorm is
 * fp32 with a centred variance.  The summation order depends on N, prefix and C only, so an image's row is bit-identical
 * in any batch.  C a multiple of 64 up to 2048, B <= 65535. */
int rajni_mean_pool_layernorm(const void* x, int B, int N, int prefix, int C, const float* gamma, const float* beta,
                              float eps, void* y, long long out_row_stride, void* stream);
/* The same values stored as fp32 (the pooled features of a headless model): y + b*out_row_stride floats, out_row_stride
 * >= C and a multiple of 4.  Same summation order; bf16_rn of each value is what rajni_mean_pool_layernorm stores. */
int rajni_mean_pool_layernorm_f32(const void* x, int B, int N, int prefix, int C, const float* gamma, const float* beta,
                                  float eps, float* y, long long out_row_stride, void* stream);

/* ---- dense contractions (attention.py:22,55; timm Mlp fc1/fc2; patch_embed; head)
 * D[orow(m), n] = epi( sum_k A[m,k] * W[n,k] ), A [M,K] bf16, W [N,K] bf16
 * (nn.Linear layout), fp32 accumulation in TMEM (tcgen05.mma, TMA-fed).
 *   orow(m) = out_row_map ? out_row_map[m] : m
 *   res row = res_row_map ? res_row_map[m] : m      (gathered residual, model.py:55-58)
 * K multiple of 8; ldd/ldres are row strides in elements (multiples of 8). */
int rajni_gemm_bf16(const void* A, const void* W, const float* bias, void* D,
                    int M, int N, int K, int flags,
                    const void* residual, long long ldres, const int32_t* res_row_map,
                    long long ldd, const int32_t* out_row_map, void* stream);

/* ---- the same contraction with LayerNorm folded in (model.py:51 norm1 -> qkv, model.py:59 norm2 -> fc1)
 *
 *   LN(x) W^T + b  =  rstd[m] * ( x (W.gamma)^T )[m,n]  -  rstd[m]*mean[m] * wsum[n]  +  ( b + W beta )[n]
 *
 * so the normalised activations never touch HBM.  Producer side (RAJNI_EPI_ROW_STATS, with the
 * bias+residual epilogue): for every stored row r the kernel writes, per slot s of 64 columns (32 when
 * N is not a multiple of 128), row_stats[s*row_stats_ld + r] = (sum, sum of squares) of the bf16 values
 * it stored in that slot; rajni_gemm_row_stats_slots(N) is the slot count for an N-column output (the
 * partition depends on N only, never on the tile shape or M, so results do not depend on the batch).  Consumer side
 * (RAJNI_EPI_LN_FOLD): A = x, W = bf16(W*gamma), bias = b + W beta, ln_wsum[n] = sum_k W'[n,k]; mean and the
 * biased variance of row m come from summing ln_slots partials at ln_stats[s*ln_stats_ld + m]; K is the
 * LayerNorm width.  Both need N % tile == 0 and 32-byte aligned rows (true for every ViT width). */
typedef struct rajni_gemm_args {
    const void* A; const void* W; const float* bias; void* D;
    int M, N, K, flags;
    const void* residual; long long ldres; const int32_t* res_row_map;
    long long ldd; const int32_t* out_row_map;
    const float* ln_stats; long long ln_stats_ld; int ln_slots; const float* ln_wsum; float ln_eps;
    float* row_stats; long long row_stats_ld;
    /* optional stream-K scratch (may be NULL): >= rajni_gemm_workspace_bytes() bytes, 128-byte aligned, its first 4096 bytes
     * ZERO before the first call (the kernels leave them zero).  With it, a CTA-pair GEMM with a long K whose tile count is
     * not a multiple of the SM pairs splits the leftover tiles of the last wave along K over the pairs and reduces the fp32
     * partials through this buffer (deterministic order).  Calls that share one workspace must be ordered on one stream. */
    void* workspace; long long workspace_bytes;
} rajni_gemm_args;
int rajni_gemm_bf16_ex(const rajni_gemm_args* args, void* stream);
size_t rajni_gemm_workspace_bytes(void);
/* Host-side query, no launch: the number of tiles a GEMM of this shape and these flags would split along K when given a
 * workspace (0 = none) and, through sk_pairs (may be NULL), the number of CTA pairs that share the pieces. */
int rajni_gemm_stream_k_plan(int M, int N, int K, int flags, int* sk_pairs);
int rajni_gemm_row_stats_slots(int N);

/* ---- a4: multi-head attention over kept tokens (attention.py:45-54)
 * qkv [B,N_src,3C] bf16; when row_map != NULL token j of image b is read from
 * global row row_map[b*Np+j] (gather fused into the loads), else N_src == Np.
 * out [B,Np,C] bf16 = softmax(q k^T * scale) v, heads concatenated. D must be 64.
 * reverse != 0: process the images last-to-first (L2 reuse hint, see RAJNI_HINT_REVERSE_M).
 * Images are independent for finite inputs.  Np > 64: also for non-finite ones (a NaN/Inf in one image never reaches
 * another's output).  Np <= 64: consecutive images may share a tile and one P V product (masked softmax): a NaN/Inf VALUE row
 * then reaches the images packed with it (0 * NaN); the environment variable RAJNI_ATTN_NOPACK=1 keeps one image per tile. */
int rajni_attention_fwd(const void* qkv, const int32_t* row_map, void* out,
                        int B, int N_src, int Np, int C, int H, float scale, int reverse, void* stream);
/* The same call with the kernel chosen by the caller (tests and A/B timing; results agree within bf16 rounding):
 * AUTO = what rajni_attention_fwd picks; PIPE = role-pipelined kernel (Np_pad <= 224); TC = two-tile kernel (Np <= 256);
 * LONG = key-block kernel (built for Np > 256).  A kernel asked for a shape it does not cover returns RAJNI_EINVAL. */
enum { RAJNI_ATTN_AUTO = 0, RAJNI_ATTN_PIPE = 1, RAJNI_ATTN_TC = 2, RAJNI_ATTN_LONG = 3 };
int rajni_attention_fwd_ex(const void* qkv, const int32_t* row_map, void* out,
                           int B, int N_src, int Np, int C, int H, float scale, int reverse, int impl, void* stream);

/* ---- a8: patch-embed front end (model.py:31-37)
 * im2col: images [B,3,S,S] (image_dtype: RAJNI_IMG_BF16 / _F32 / _U8) -> cols [B*P, 3*p*p] bf16, P = (S/p)^2,
 * in Conv2d weight order (c, ky, kx).  patch: any multiple of 8 that divides S <= 16384 (8, 16, 24, 32, ...; ABI >= 10,
 * 16 only before), so 3*p*p is a multiple of 64.  RAJNI_IMG_U8: raw pixels, normalised here as the reference's
 * loader does in fp32 (run.py:62-70: ToTensor + Normalize): (u/255 - norm[c]) / norm[3+c] with
 * norm = HOST array {mean[3], std[3]} (read at call time); other dtypes ignore norm (may be NULL).
 * Also writes the CLS rows
 * x[b,0,:] = cls_pos0[:] (= cls_token + pos_embed[0], precomputed) into x [B,1+P,C] and, when
 * row_stats != NULL, the LayerNorm partials of those rows (slot 0 = (cls_sum, cls_sumsq), the
 * other `stats_slots-1` slots zero) in the layout RAJNI_EPI_ROW_STATS uses. */
enum { RAJNI_IMG_BF16 = 0, RAJNI_IMG_F32 = 1, RAJNI_IMG_U8 = 2 };
int rajni_patch_im2col(const void* images, int image_dtype, int B, int S, int patch,
                       void* cols, const void* cls_pos0, void* x, int C,
                       float* row_stats, long long row_stats_ld, int stats_slots,
                       float cls_sum, float cls_sumsq, const float* norm, void* stream);
/* The same with `prefix` (1 or 2) rows in front of each image's patches: x is [B,P+prefix,C], and x[b,r,:] =
 * prefix_rows[r,:] for r < prefix (prefix_rows [prefix,C] bf16: cls_token + pos_embed[0], dist_token + pos_embed[1]; the
 * tokens alone for a model that adds positions to the patches only).  With row_stats, prefix_stats_host = HOST array
 * [prefix][2] of each row's (sum, sum of squares), written to slot 0 (read at call time).  The embed GEMM stores patch q
 * of image b at row b*(P+prefix) + prefix + q.  rajni_patch_im2col is this call with prefix 1. */
int rajni_patch_im2col_prefix(const void* images, int image_dtype, int B, int S, int patch,
                              void* cols, const void* prefix_rows, int prefix, void* x, int C,
                              float* row_stats, long long row_stats_ld, int stats_slots,
                              const float* prefix_stats_host, const float* norm, void* stream);

/* ---- f3: the loader's Resize(size, bicubic) + CenterCrop(224) on decoded uint8 RGB frames (run.py:62-66), bit-identical
 * to torchvision on PIL images (Pillow's antialiased two-pass resampler; oracle/resize_oracle.py restates it).
 * frames: device buffer, the B decoded frames (HWC, uint8) back to back; meta: DEVICE int64 [B][3] = (byte offset of the
 * frame in `frames`, height, width); max_h >= every height.  out: uint8 [B,3,224,224] planar - what PILToTensor gives after
 * the two transforms; feed it to rajni_patch_im2col (RAJNI_IMG_U8) for ToTensor + Normalize.
 * workspace: rajni_resize_workspace_bytes(B, max_h) bytes.  A frame that cannot be handled (shorter edge would end up
 * below the crop, height above max_h, downscale beyond ~23x) is skipped and reported by rajni_resize_status (which
 * synchronises the stream): 0 = all frames done, else 1 + index of a rejected frame. */
size_t rajni_resize_workspace_bytes(int B, int max_h);
int rajni_resize_center_crop_u8(const void* frames, const long long* meta, int B, int max_h, int size, int crop,
                                void* out, void* workspace, size_t workspace_bytes, void* stream);
int rajni_resize_status(const void* workspace, int B, int max_h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RAJNI_B200_H */
