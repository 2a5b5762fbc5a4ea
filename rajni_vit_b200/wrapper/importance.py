"""compute_importance — drop-in for rajni/wrapper/importance.py:5-34."""
from __future__ import annotations

import torch

from .. import ops


@torch.no_grad()
def compute_importance(qkv: torch.Tensor, num_heads: int, eps: float = 1e-6, prefix: int = 1) -> torch.Tensor:
    """qkv [B, N, 3*C] -> importance [B, N] in qkv's dtype.

    Same signature and meaning as the reference.  The tile is consumed as bf16 and
    every reduction is done in fp32 by the fused sm_100a scoring kernel (the
    reference computes in the tensor's own dtype; bf16-computed scores reorder the
    top-k, SURVEY.md section 4.5).  Head dim must be 64.  ``prefix`` (1, or 2 for a distilled DeiT's CLS +
    distillation token) leaves the scores as they are: the query is row 0 and every token is a key and value.
    """
    if qkv.dim() != 3 or qkv.shape[-1] % 3:
        raise ValueError(f"qkv must be [B, N, 3*C], got {tuple(qkv.shape)}")
    tile = qkv.detach().to(torch.bfloat16).contiguous()
    return ops.importance(tile, num_heads, eps, prefix=prefix).to(qkv.dtype)
