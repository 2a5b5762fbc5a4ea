"""Per-kernel timing on one B200 (CUDA events, L2 flushed between iterations).
Prints achieved TFLOP/s or GB/s against MEASURED_PEAKS.json for the shapes of BASELINE config 2."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rajni_vit_b200 import ops  # noqa: E402

PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
try:
    PEAKS.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
except Exception:
    pass

flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")


def timeit(fn, iters=10, warm=3, inner=1):
    """Median over `iters` of the time of `inner` back-to-back calls (L2 flushed before each group).  The event timer on
    these boxes ticks in ~4 us steps, so kernels shorter than ~100 us should be timed with inner > 1."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / inner)
    ts.sort()
    return ts[len(ts) // 2] * 1e-3


def gemm_case(name, M, N, K, **kw):
    a = torch.randn(M, K, device="cuda").bfloat16()
    w = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
    bias = torch.randn(N, device="cuda")
    res = torch.randn(M, N, device="cuda").bfloat16() if kw.pop("res", False) else None
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    t = timeit(lambda: ops.gemm(a, w, bias, M, N, K, residual=res, out=out, **kw))
    tf = 2.0 * M * N * K / t / 1e12
    t2 = timeit(lambda: torch.nn.functional.linear(a, w))
    print(f"{name:28s} M={M:6d} N={N:5d} K={K:5d}  {t*1e6:8.1f} us  {tf:7.1f} TF/s  "
          f"({tf/PEAKS['bf16_tflops']*100:5.1f}% of measured burst)   cuBLAS {2.0*M*N*K/t2/1e12:7.1f} TF/s")


def main():
    B = 256
    only = set(sys.argv[1:])

    def want(k):
        return not only or k in only

    for N in (197, 173, 87) if want("gemm") else ():
        M = B * N
        gemm_case(f"qkv N={N}", M, 2304, 768)
        gemm_case(f"proj+res N={N}", M, 768, 768, res=True)
        gemm_case(f"fc1+gelu N={N}", M, 3072, 768, gelu=True)
        gemm_case(f"fc2+res N={N}", M, 768, 3072, res=True)
    if want("gemm"):
        gemm_case("patch-embed", B * 196, 768, 768)
    # score+select
    for N, keep in ((197, 172), (173, 151), (152, 120), (121, 86)) if want("score") else ():
        qkv = torch.randn(B, N, 2304, device="cuda").bfloat16()
        t = timeit(lambda: ops.score_select(qkv, 12, keep), inner=8)
        nbytes = B * (2 * N * 768 * 2 + 768 * 2 + 8 * (keep + 1))
        print(f"score_select N={N:3d}            {t*1e6:8.1f} us  {nbytes/t/1e9:7.1f} GB/s ({nbytes/t/1e9/PEAKS['hbm_gbs']*100:5.1f}% of measured HBM)")
    # the long-sequence score path (ViT-B/8, 785 tokens: logits and value rows through the workspace); K/V-plane bytes
    if want("score_long"):
        N, keep = 785, 690
        qkv = torch.randn(B, N, 2304, device="cuda").bfloat16()
        t = timeit(lambda: ops.score_select(qkv, 12, keep), inner=4)
        kv = B * 2 * N * 768 * 2
        print(f"score_select N={N} (workspace)  {t*1e6:8.1f} us  {kv/t/1e9:7.1f} GB/s of K/V planes ({kv/t/1e9/PEAKS['hbm_gbs']*100:5.1f}% of measured HBM)")
        del qkv
    # attention
    for N, Np in ((197, 197), (197, 173), (173, 152), (152, 121), (121, 87), (87, 87)) if want("attn") else ():
        qkv = torch.randn(B * N, 2304, device="cuda").bfloat16()
        rmap = None
        if Np < N:
            idx = torch.stack([torch.sort(torch.randperm(N, device="cuda")[:Np]).values for _ in range(B)])
            rmap = (idx + torch.arange(B, device="cuda")[:, None] * N).int().flatten()
        out = torch.empty(B * Np, 768, device="cuda", dtype=torch.bfloat16)
        t = timeit(lambda: ops.attention(qkv, rmap, B, N, Np, 768, 12, 0.125, out=out), inner=8)
        fl = 4.0 * B * Np * Np * 768
        print(f"attention N={N:3d} Np={Np:3d}        {t*1e6:8.1f} us  {fl/t/1e12:7.1f} TF/s")
    if not want("rows"):
        return
    # layernorm
    M = B * 197
    x = torch.randn(M, 768, device="cuda").bfloat16()
    g = torch.ones(768, device="cuda")
    out = torch.empty_like(x)
    t = timeit(lambda: ops.layernorm(x, g, g, 1e-6, M, 768, out=out))
    print(f"layernorm {M}x768            {t*1e6:8.1f} us  {2*M*768*2/t/1e9:7.1f} GB/s")
    # im2col
    img = torch.randn(B, 3, 224, 224, device="cuda")
    cols = torch.empty(B * 196, 768, device="cuda", dtype=torch.bfloat16)
    xx = torch.empty(B * 197, 768, device="cuda", dtype=torch.bfloat16)
    c0 = torch.zeros(768, device="cuda", dtype=torch.bfloat16)
    t = timeit(lambda: ops.patch_im2col(img, 16, cols, c0, xx, 768))
    print(f"im2col                       {t*1e6:8.1f} us  {(img.numel()*4+cols.numel()*2)/t/1e9:7.1f} GB/s")
    # im2col at 8/16/32-pixel patches, fp32 and uint8 pixels: the same bytes at every patch size (3*224*224 pixels in, as
    # many bf16 out per image)
    img8 = torch.randint(0, 256, (B, 3, 224, 224), device="cuda", dtype=torch.uint8)
    norm = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    for p in (8, 16, 32):
        P = (224 // p) ** 2
        cp = torch.empty(B * P, 3 * p * p, device="cuda", dtype=torch.bfloat16)
        xp = torch.empty(B * (P + 1), 768, device="cuda", dtype=torch.bfloat16)
        for im in (img, img8):
            t = timeit(lambda: ops.patch_im2col(im, p, cp, c0, xp, 768, norm=norm if im.dtype == torch.uint8 else None), inner=4)
            nb = im.numel() * im.element_size() + cp.numel() * 2
            print(f"im2col p={p:2d} {str(im.dtype)[6:]:7s}          {t*1e6:8.1f} us  {nb/t/1e9:7.1f} GB/s")


if __name__ == "__main__":
    main()
