"""Long-sequence attention (Np > 256): the tcgen05 key-block kernel.  usage: python tools/attn_long_bench.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rajni_vit_b200 import ops  # noqa: E402
from tools.kbench import timeit  # noqa: E402

for B, N, Np in ((16, 577, 577), (128, 577, 577), (128, 577, 507), (128, 507, 446), (128, 446, 357), (128, 357, 257), (128, 257, 257)):
    qkv = torch.randn(B * N, 2304, device="cuda").bfloat16()
    rmap = None
    if Np < N:
        idx = torch.stack([torch.sort(torch.randperm(N, device="cuda")[:Np]).values for _ in range(B)])
        rmap = (idx + torch.arange(B, device="cuda")[:, None] * N).int().flatten()
    out = torch.empty(B * Np, 768, device="cuda", dtype=torch.bfloat16)
    t = timeit(lambda: ops.attention(qkv, rmap, B, N, Np, 768, 12, 0.125, out=out))
    print(f"tcgen05 key-block  B={B:3d} N={N} Np={Np}: {t*1e6:7.1f} us  {4.0*B*Np*Np*768/t/1e12:6.1f} TF/s", flush=True)
