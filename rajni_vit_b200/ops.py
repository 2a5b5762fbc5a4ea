"""Tensor-level wrappers over the C ABI: torch supplies device memory and the stream,
librajni_b200.so does the work.  Every function requires CUDA tensors on an sm_100
device and raises otherwise (no CPU path)."""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (EPI_BIAS, EPI_GELU, EPI_LN_FOLD, EPI_OUT_F32, EPI_RESIDUAL, EPI_ROW_STATS,  # noqa: F401  (re-exported)
                   HINT_REVERSE_M)

_checked_devices = set()
_prof = None        # list of (name, work, start_event, end_event) while profile_steps() runs


def _call(name: str, work: float, fn, *args) -> None:
    """Launch one C-ABI kernel; under profile_steps() bracket it with CUDA events on the launch stream."""
    if _prof is None:
        _lib.check(fn(*args))
        return
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    _lib.check(fn(*args))
    end.record()
    _prof.append((name, work, start, end))


def profile_steps(step_fn, steps: int = 3):
    """Run ``step_fn`` ``steps`` times with every kernel launch timed by its own CUDA-event pair.
    Returns {kernel class: {"ms": per-step ms, "work": per-step flops or bytes, "launches": per step}}."""
    global _prof
    step_fn()
    torch.cuda.synchronize()
    _prof = []
    try:
        for _ in range(steps):
            step_fn()
        torch.cuda.synchronize()
        out = {}
        for name, work, s, e in _prof:
            d = out.setdefault(name, {"ms": 0.0, "work": 0.0, "launches": 0})
            d["ms"] += s.elapsed_time(e) / steps
            d["work"] += work / steps
            d["launches"] += 1
        for d in out.values():
            d["launches"] //= steps
        return out
    finally:
        _prof = None


def _stream(t: torch.Tensor) -> int:
    dev = t.device
    if dev.type != "cuda":
        raise RuntimeError("rajni_vit_b200 runs on CUDA (sm_100a) tensors only; there is no CPU path")
    if dev.index not in _checked_devices:
        with torch.cuda.device(dev):
            _lib.check(_lib.load().rajni_device_check())
        _checked_devices.add(dev.index)
    return torch.cuda.current_stream(dev).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _bf16c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.bfloat16 or not t.is_contiguous():
        raise ValueError(f"expected a contiguous bf16 tensor, got {t.dtype} contiguous={t.is_contiguous()}")
    return t


def _check_prefix(prefix: int) -> int:
    if prefix not in (1, 2):
        raise ValueError(f"prefix={prefix}: 1 (CLS) or 2 (CLS + distillation token) leading tokens are supported")
    return prefix


def importance(qkv: torch.Tensor, num_heads: int, eps: float = 1e-6, workspace: Optional[torch.Tensor] = None,
               prefix: int = 1) -> torch.Tensor:
    """qkv [B,N,3C] bf16 -> scores [B,N] fp32.   importance.py:5-34
    Sequences too long for the one-launch kernel (``needs_score_workspace``) take the two-launch path with scratch
    (``workspace`` as in ``score_select``).  ``prefix`` (1 or 2 leading tokens) does not change the scores: the query is
    row 0 and every token, a distillation token too, is a key and value."""
    _check_prefix(prefix)
    _bf16c(qkv)
    B, N, C3 = qkv.shape
    C = C3 // 3
    scores = torch.empty((B, N), device=qkv.device, dtype=torch.float32)
    work = B * (2 * N * C * 2 + C * 2 + 4 * N)
    ws = _checked_score_workspace(qkv.device, B, N, C, num_heads, workspace) if needs_score_workspace(N, num_heads) else None
    _call("score_select", work, _lib.load().rajni_score_select_prefix, qkv.data_ptr(), B, N, C, num_heads, prefix, 0, eps,
          scores.data_ptr(), None, None, None, _ptr(ws), 0 if ws is None else ws.numel(), _stream(qkv))
    return scores


def select(scores: torch.Tensor, keep: int, keep_idx=None, next_scores=None, row_map=None, prefix: int = 1
           ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """scores [B,N] fp32 -> (keep_idx int32 [B,keep+prefix], next_scores fp32, row_map int32 [B*(keep+prefix)]).
    The first ``prefix`` tokens (CLS, or CLS + distillation token) are always kept; the top ``keep`` of the rest follow."""
    if scores.dtype != torch.float32 or not scores.is_contiguous():
        raise ValueError("scores must be contiguous fp32")
    _check_prefix(prefix)
    B, N = scores.shape
    dev = scores.device
    Np = keep + prefix
    keep_idx = torch.empty((B, Np), device=dev, dtype=torch.int32) if keep_idx is None else keep_idx
    next_scores = torch.empty((B, Np), device=dev, dtype=torch.float32) if next_scores is None else next_scores
    row_map = torch.empty((B * Np,), device=dev, dtype=torch.int32) if row_map is None else row_map
    _call("select", B * (4 * N + 12 * Np), _lib.load().rajni_select_prefix, scores.data_ptr(), B, N, prefix, keep,
          keep_idx.data_ptr(), next_scores.data_ptr(), row_map.data_ptr(), _stream(scores))
    return keep_idx, next_scores, row_map


# Up to this many images per launch (about one per SM) the K/V pass is spread over (image, row-block) CTAs: at 197 tokens the
# split path wins up to ~160 images (128: 27.8 vs 30.9 us), at 577 tokens by 12 % at 128 (profiles/r2_score_select.md)
SPLIT_SCORE_MAX_BATCH = 148
_score_ws = {}


def score_workspace_bytes(B: int, N: int, C: int, num_heads: int) -> int:
    """Scratch bytes the split score path needs (rajni_score_select_workspace_bytes)."""
    return int(_lib.load().rajni_score_select_workspace_bytes(B, N, C, num_heads))


def needs_score_workspace(N: int, num_heads: int) -> bool:
    """True when scoring N tokens with this many heads needs the split path's workspace at every batch size (the one-launch
    kernel's shared memory cannot hold the image's logits and value rows).  Host-side query, no launch."""
    return bool(_lib.load().rajni_score_select_needs_workspace(N, num_heads))


def _score_workspace(dev: torch.device, nbytes: int) -> torch.Tensor:
    """Process-wide scratch for callers that do not bring their own (stand-alone ops.score_select calls).  Grow-only and
    NEVER freed: a CUDA graph captured by some other caller may have baked an older buffer's address in, so superseded
    buffers stay alive in the list.  RAJNIViTWrapper owns its scratch (``workspace=``) and does not come here."""
    bufs = _score_ws.setdefault(dev, [])
    if not bufs or bufs[-1].numel() < nbytes:
        bufs.append(torch.empty(nbytes, device=dev, dtype=torch.uint8))
    return bufs[-1]


def _checked_score_workspace(dev: torch.device, B: int, N: int, C: int, num_heads: int,
                             workspace: Optional[torch.Tensor]) -> torch.Tensor:
    nbytes = score_workspace_bytes(B, N, C, num_heads)
    ws = workspace if workspace is not None else _score_workspace(dev, nbytes)
    if ws.numel() * ws.element_size() < nbytes or ws.device != dev:
        raise ValueError(f"score_select: workspace of {ws.numel() * ws.element_size()} B on {ws.device}, need {nbytes} B on {dev}")
    return ws


def score_select(qkv: torch.Tensor, num_heads: int, keep: int, eps: float = 1e-6, want_scores: bool = False,
                 keep_idx=None, next_scores=None, row_map=None, scores=None, split: Optional[bool] = None,
                 workspace: Optional[torch.Tensor] = None, prefix: int = 1):
    """Fused importance + selection on qkv [B,N,3C] bf16.
    Returns (scores or None, keep_idx [B,keep+prefix], next_scores, row_map); ``prefix`` as in ``select``.
    ``workspace``: uint8 scratch of at least ``score_workspace_bytes(B, N, C, H)`` for the split path (small batches, and
    every batch of a sequence for which ``needs_score_workspace``); a caller that replays CUDA graphs must pass one it owns,
    so that the captured address lives as long as the graph."""
    _bf16c(qkv)
    _check_prefix(prefix)
    B, N, C3 = qkv.shape
    dev = qkv.device
    Np = keep + prefix
    if want_scores and scores is None:
        scores = torch.empty((B, N), device=dev, dtype=torch.float32)
    keep_idx = torch.empty((B, Np), device=dev, dtype=torch.int32) if keep_idx is None else keep_idx
    next_scores = torch.empty((B, Np), device=dev, dtype=torch.float32) if next_scores is None else next_scores
    row_map = torch.empty((B * Np,), device=dev, dtype=torch.int32) if row_map is None else row_map
    C = C3 // 3
    lib = _lib.load()
    if split is None:
        split = B <= SPLIT_SCORE_MAX_BATCH or needs_score_workspace(N, num_heads)
    # algorithmic bytes (SURVEY 8d): K and V planes + CLS query in, index + carried score out
    work = B * (2 * N * C * 2 + C * 2 + 8 * Np)
    ws = _checked_score_workspace(dev, B, N, C, num_heads, workspace) if split else None
    _call("score_select", work, lib.rajni_score_select_prefix, qkv.data_ptr(), B, N, C, num_heads, prefix, keep, eps,
          _ptr(scores), keep_idx.data_ptr(), next_scores.data_ptr(), row_map.data_ptr(), _ptr(ws),
          0 if ws is None else ws.numel(), _stream(qkv))
    return scores, keep_idx, next_scores, row_map


def gather_rows(src: torch.Tensor, row_map: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """src [R,E] bf16, row_map int32 [R_out] -> out [R_out,E]."""
    _bf16c(src)
    rows_out, E = row_map.numel(), src.shape[-1]
    out = torch.empty((rows_out, E), device=src.device, dtype=torch.bfloat16) if out is None else out
    _call("gather_rows", rows_out * (4 * E + 4), _lib.load().rajni_gather_rows,
          src.data_ptr(), row_map.data_ptr(), out.data_ptr(), rows_out, E, _stream(src))
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, rows: int, C: int,
              in_row_stride: Optional[int] = None, out: Optional[torch.Tensor] = None, in_offset: int = 0,
              out_row_stride: Optional[int] = None, out_offset: int = 0, row_stats: Optional[torch.Tensor] = None,
              stats_slots: int = 0) -> torch.Tensor:
    """Row LayerNorm, bf16 -> bf16 or fp32 (the dtype of ``out``; bf16 when ``out`` is None); row r read at
    x.data_ptr + in_offset + r*in_row_stride elements and written at out.data_ptr + out_offset + r*out_row_stride elements
    (default C: dense rows).  ``out`` may be ``x`` (in place).  An fp32 ``out`` holds the values that the bf16 output rounds.
    ``row_stats`` fp32 [>= stats_slots, >= rows, 2]: also write the LayerNorm partial sums of the stored rows for an LN-folded
    ``gemm`` (slot 0 = (sum, sum of squares) of row r as stored in bf16, slots 1..stats_slots-1 zero); bf16 ``out`` only."""
    out = torch.empty((rows, C), device=x.device, dtype=torch.bfloat16) if out is None else out
    if out.dtype not in (torch.bfloat16, torch.float32):
        raise ValueError(f"layernorm: out must be bf16 or fp32, got {out.dtype}")
    f32 = out.dtype == torch.float32
    stride = C if in_row_stride is None else in_row_stride
    ostride = C if out_row_stride is None else out_row_stride
    if in_offset + (rows - 1) * stride + C > x.numel() or out_offset + (rows - 1) * ostride + C > out.numel():
        raise ValueError(f"layernorm: {rows} rows (strides {stride} / {ostride}, offsets {in_offset} / {out_offset}) exceed "
                         f"the input ({x.numel()}) or output ({out.numel()} elements)")
    if row_stats is None:
        _call("layernorm_f32" if f32 else "layernorm", rows * C * (6 if f32 else 4),
              _lib.load().rajni_layernorm_strided_f32 if f32 else _lib.load().rajni_layernorm_strided, x.data_ptr() + 2 * in_offset,
              stride, gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr() + out.element_size() * out_offset, ostride, rows, C,
              _stream(x))
        return out
    if f32:
        raise ValueError("layernorm: row_stats are the sums of the stored bf16 rows; out must be bf16")
    if (row_stats.dtype != torch.float32 or not row_stats.is_contiguous() or row_stats.dim() != 3 or row_stats.shape[2] != 2
            or row_stats.shape[0] < stats_slots or row_stats.shape[1] < rows):
        raise ValueError(f"layernorm: row_stats must be contiguous fp32 [>= {stats_slots}, >= {rows}, 2], got "
                         f"{row_stats.dtype} {tuple(row_stats.shape)}")
    _call("layernorm_row_stats", rows * C * 4 + rows * stats_slots * 8, _lib.load().rajni_layernorm_row_stats,
          x.data_ptr() + 2 * in_offset, stride, gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr() + 2 * out_offset, ostride,
          rows, C, row_stats.data_ptr(), row_stats.shape[1], stats_slots, _stream(x))
    return out


def mean_pool_layernorm(x: torch.Tensor, B: int, N: int, C: int, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
                        prefix: int = 1, out: Optional[torch.Tensor] = None, out_row_stride: Optional[int] = None) -> torch.Tensor:
    """timm's average-pooled head input: out[b] = LayerNorm(mean of x[b*N + prefix .. b*N + N-1]) (fc_norm over the patch
    tokens' mean), x [>= B*N, C] bf16 dense; -> bf16 or fp32 rows (the dtype of ``out``; bf16 when ``out`` is None) at
    out.data_ptr + b*out_row_stride elements (default C).  fp32 sums in an order that does not depend on B; an fp32 ``out``
    holds the values that the bf16 output rounds."""
    _check_prefix(prefix)
    if x.dtype != torch.bfloat16 or not x.is_contiguous() or x.numel() < B * N * C:
        raise ValueError(f"mean_pool_layernorm: x must be contiguous bf16 with at least {B}*{N} rows of {C}")
    ostride = C if out_row_stride is None else out_row_stride
    out = torch.empty((B, C), device=x.device, dtype=torch.bfloat16) if out is None else out
    if out.dtype not in (torch.bfloat16, torch.float32) or out.numel() < (B - 1) * ostride + C:
        raise ValueError(f"mean_pool_layernorm: out must be bf16 or fp32 with room for {B} rows at stride {ostride}")
    f32 = out.dtype == torch.float32
    lib = _lib.load()
    _call("mean_pool_layernorm_f32" if f32 else "mean_pool_layernorm", B * ((N - prefix) * C * 2 + C * out.element_size()),
          lib.rajni_mean_pool_layernorm_f32 if f32 else lib.rajni_mean_pool_layernorm, x.data_ptr(), B, N, prefix, C,
          gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(), ostride, _stream(x))
    return out


def row_stats_slots(n_cols: int) -> int:
    """Partial-sum slots per row that a ``row_stats`` GEMM with ``n_cols`` output columns writes (one per 32 columns)."""
    return int(_lib.load().rajni_gemm_row_stats_slots(n_cols))


def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], M: int, N: int, K: int, *,
         gelu: bool = False, residual: Optional[torch.Tensor] = None, ldres: Optional[int] = None,
         res_row_map: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
         ldd: Optional[int] = None, out_row_map: Optional[torch.Tensor] = None, out_f32: bool = False,
         ln: Optional[tuple] = None, row_stats: Optional[torch.Tensor] = None, tag: str = "",
         reverse: bool = False) -> torch.Tensor:
    """out[orow(m), n] = epi(sum_k a[m,k] w[n,k]); a [M,K] bf16, w [N,K] bf16, bias fp32 [N].

    ``ln = (stats, slots, wsum, eps)``: LayerNorm folded in (a is the un-normalised x, w = W*gamma,
    bias = b + W beta, wsum[n] = sum_k w[n,k], stats fp32 [>=slots, rows, 2] partial sums of x's rows).
    ``row_stats`` fp32 [slots, rows, 2]: also emit the partial sums of the rows this GEMM stores.
    ``reverse``: walk the M tiles last-to-first (L2 reuse hint; results identical)."""
    flags = (EPI_BIAS if bias is not None else 0) | (EPI_GELU if gelu else 0) | \
            (EPI_RESIDUAL if residual is not None else 0) | (EPI_OUT_F32 if out_f32 else 0) | \
            (HINT_REVERSE_M if reverse else 0)
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=torch.float32 if out_f32 else torch.bfloat16)
    args = _lib.GemmArgs(a.data_ptr(), w.data_ptr(), _ptr(bias), out.data_ptr(), M, N, K, flags,
                         _ptr(residual), (N if ldres is None else ldres), _ptr(res_row_map),
                         (N if ldd is None else ldd), _ptr(out_row_map))
    if ln is not None:
        stats, slots, wsum, eps = ln
        args.flags |= EPI_LN_FOLD
        args.ln_stats, args.ln_stats_ld, args.ln_slots = stats.data_ptr(), stats.shape[1], slots
        args.ln_wsum, args.ln_eps = wsum.data_ptr(), eps
    if row_stats is not None:
        args.flags |= EPI_ROW_STATS
        args.row_stats, args.row_stats_ld = row_stats.data_ptr(), row_stats.shape[1]
    _call("gemm:" + tag if tag else "gemm", 2.0 * M * N * K, _lib.load().rajni_gemm_bf16_ex, args, _stream(a))
    return out


LONG_SEQ = 256          # above this many kept tokens the key-block kernel runs; it wants its rows compacted first


def attention(qkv: torch.Tensor, row_map: Optional[torch.Tensor], B: int, N_src: int, Np: int, C: int,
              num_heads: int, scale: float, out: Optional[torch.Tensor] = None, reverse: bool = False,
              compact: Optional[torch.Tensor] = None, impl: int = _lib.ATTN_AUTO) -> torch.Tensor:
    """Attention over the Np kept tokens of each image.  -> [B*Np, C] bf16

    ``impl``: _lib.ATTN_AUTO (default) or a specific kernel (tests / A-B timing), see include/rajni_b200.h.
    Np <= 256: the kept-token gather is fused into the kernel's loads (cp.async by row index).
    Np  > 256: the key-block kernel streams K/V blocks with TMA, which needs consecutive rows, so the kept rows are
    compacted once with ``gather_rows`` (HBM-bound, into ``compact`` [B*Np, 3C] if given) and the dense path runs on them:
    per-row cp.async sustains only ~8 B/clk/SM, TMA boxes are not limited that way (profiles/r1_attn_long.txt)."""
    out = torch.empty((B * Np, C), device=qkv.device, dtype=torch.bfloat16) if out is None else out
    if row_map is not None and Np > LONG_SEQ:
        qkv = gather_rows(qkv.view(-1, 3 * C), row_map, out=None if compact is None else compact[: B * Np])
        row_map, N_src = None, Np
    _call("attention", 4.0 * B * Np * Np * C, _lib.load().rajni_attention_fwd_ex,
          qkv.data_ptr(), _ptr(row_map), out.data_ptr(), B, N_src, Np, C, num_heads, scale, int(reverse), int(impl), _stream(qkv))
    return out


_IMG_DTYPES = {torch.bfloat16: 0, torch.float32: 1, torch.uint8: 2}      # RAJNI_IMG_* (include/rajni_b200.h)


def patch_im2col(images: torch.Tensor, patch: int, cols: torch.Tensor, cls_pos0: torch.Tensor,
                 x: torch.Tensor, C: int, row_stats: Optional[torch.Tensor] = None, stats_slots: int = 0,
                 cls_sum=0.0, cls_sumsq=0.0, norm: Optional[tuple] = None, prefix: int = 1) -> None:
    """images [B,3,S,S] fp32|bf16|uint8 -> cols [B*P, 3*p*p] bf16; also writes the CLS rows of x (and their
    LayerNorm partial sums into row_stats fp32 [slots, rows, 2]).  uint8 pixels are normalised in the kernel with
    ``norm = (mean[3], std[3])`` exactly as ToTensor + Normalize do in fp32 (run.py:62-70).
    ``prefix`` = 2 (CLS + distillation token): x is [B, P+2, C], ``cls_pos0`` is the [2, C] block of the two prefix rows
    and ``cls_sum`` / ``cls_sumsq`` are sequences of two, one per row."""
    if images.dtype not in _IMG_DTYPES or not images.is_contiguous():
        raise ValueError("images must be contiguous fp32, bf16 or uint8")
    norm_arr = None
    if images.dtype == torch.uint8:
        if norm is None or len(norm[0]) != 3 or len(norm[1]) != 3:
            raise ValueError("uint8 images need norm=(mean[3], std[3])")
        norm_arr = (ctypes.c_float * 6)(*[float(v) for v in norm[0]], *[float(v) for v in norm[1]])
    B, ch, S, S2 = images.shape
    if ch != 3 or S != S2:
        raise ValueError(f"images must be [B,3,S,S], got {tuple(images.shape)}")
    _check_prefix(prefix)
    if cls_pos0.dtype != torch.bfloat16 or not cls_pos0.is_contiguous() or cls_pos0.numel() != prefix * C:
        raise ValueError(f"cls_pos0 must be {prefix} contiguous bf16 row(s) of {C}")
    sums = [float(v) for v in (cls_sum if prefix > 1 else [cls_sum])]
    sqs = [float(v) for v in (cls_sumsq if prefix > 1 else [cls_sumsq])]
    if len(sums) != prefix or len(sqs) != prefix:
        raise ValueError(f"cls_sum and cls_sumsq need one value per prefix row ({prefix})")
    stats_arr = (ctypes.c_float * (2 * prefix))(*[v for pair in zip(sums, sqs) for v in pair])
    _call("patch_im2col", images.numel() * images.element_size() + images.numel() * 2 + B * prefix * C * 2,
          _lib.load().rajni_patch_im2col_prefix, images.data_ptr(), _IMG_DTYPES[images.dtype], B, S, patch,
          cols.data_ptr(), cls_pos0.data_ptr(), prefix, x.data_ptr(), C, _ptr(row_stats),
          0 if row_stats is None else row_stats.shape[1], stats_slots, stats_arr, norm_arr, _stream(images))


def resize_center_crop(frames: torch.Tensor, meta: torch.Tensor, max_h: int, size: int = 256, crop: int = 224,
                       out: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None,
                       check: bool = True) -> torch.Tensor:
    """Resize(size, bicubic) + CenterCrop(crop) of B decoded uint8 RGB frames (run.py:62-66), bit-identical to torchvision
    on PIL images.  ``frames``: 1-D uint8 CUDA tensor holding the frames (HWC) back to back; ``meta``: int64 CUDA tensor
    [B,3] = (byte offset, height, width).  -> uint8 [B,3,crop,crop] (planar, what PILToTensor yields).
    ``check``: read the status word back (synchronises) and raise for frames the kernel had to skip."""
    if frames.dtype != torch.uint8 or frames.dim() != 1 or not frames.is_contiguous():
        raise ValueError("frames must be a contiguous 1-D uint8 tensor")
    if meta.dtype != torch.int64 or meta.dim() != 2 or meta.shape[1] != 3 or not meta.is_contiguous() or meta.device != frames.device:
        raise ValueError("meta must be a contiguous int64 [B,3] tensor on the frames' device")
    B = meta.shape[0]
    lib = _lib.load()
    nbytes = int(lib.rajni_resize_workspace_bytes(B, max_h))
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty(nbytes, device=frames.device, dtype=torch.uint8)
    out = torch.empty((B, 3, crop, crop), device=frames.device, dtype=torch.uint8) if out is None else out
    stream = _stream(frames)
    src_bytes = frames.numel()
    _call("resize_center_crop", src_bytes + out.numel(), lib.rajni_resize_center_crop_u8, frames.data_ptr(), meta.data_ptr(),
          B, max_h, size, crop, out.data_ptr(), workspace.data_ptr(), workspace.numel(), stream)
    if check:
        bad = int(lib.rajni_resize_status(workspace.data_ptr(), B, max_h, stream))
        if bad < 0:
            _lib.check(bad)
        if bad:
            raise ValueError(f"frame {bad - 1} cannot be resized on the GPU (too small for the crop, taller than max_h={max_h}, "
                             "or a downscale beyond 23x)")
    return out
