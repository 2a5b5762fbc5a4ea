"""RAJNIAttention — drop-in for rajni/wrapper/attention.py:5-60 on sm_100a kernels."""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from .. import ops
from ..packing import PackCache


def keep_count(num_tokens: int, keep_ratio: float, prefix: int = 1) -> int:
    """Patches kept out of ``num_tokens - prefix``: Python double multiply, truncation, floor of 1
    (rajni/wrapper/attention.py:31-32).  ``prefix``: the leading tokens that are always kept (1: CLS; 2: CLS and the
    distillation token of a distilled DeiT)."""
    return max(1, int(keep_ratio * (num_tokens - prefix)))


class RAJNIAttention(nn.Module):
    """Importance -> top-k -> gather -> attention over kept tokens -> proj.

    Same constructor, attributes and return contract as the reference:
    ``forward(x[B,N,C], prev_scores=None) -> (out[B,Np,C], keep_idx[B,Np] int64, next_scores[B,Np])``.
    Shares (does not copy) the wrapped attention's ``qkv`` / ``proj`` modules
    (attention.py:10-11).  ``num_prefix_tokens`` (set by RAJNIViTWrapper from its base model) leading tokens are always
    kept: Np = keep + num_prefix_tokens.
    """

    def __init__(self, attn: nn.Module, keep_ratio: float, update: bool):
        super().__init__()
        self.num_heads = attn.num_heads
        self.scale = attn.scale
        self.qkv = attn.qkv
        self.proj = attn.proj
        self.proj_drop = attn.proj_drop
        self.keep_ratio = keep_ratio
        self.update = update
        self.num_prefix_tokens = 1
        for name in ("q_norm", "k_norm"):
            sub = getattr(attn, name, None)
            if sub is not None and not isinstance(sub, nn.Identity):
                raise NotImplementedError(f"attention.{name} = {type(sub).__name__} is not supported by the B200 path")
        self._packs = PackCache()

    def _apply(self, fn, *a, **kw):
        self._packs.clear()
        return super()._apply(fn, *a, **kw)

    def _check_eval(self):
        d = self.proj_drop
        if isinstance(d, nn.Dropout) and d.p > 0 and self.training:
            raise NotImplementedError("proj_drop with p > 0 in training mode is not supported (inference path)")

    def forward_packed(self, xn: torch.Tensor, prev_scores: Optional[torch.Tensor], B: int, N: int,
                       want_scores: bool = False):
        """xn [B*N, C] bf16 (already LayerNorm'd) ->
        (out [B*Np, C] bf16 pre-residual, keep_idx i32 [B,Np], next_scores f32 [B,Np], row_map i32, scores|None)."""
        self._check_eval()
        C = xn.shape[-1]
        H = self.num_heads
        qw, qb = self._packs.linear(self.qkv)
        pw, pb = self._packs.linear(self.proj)
        qkv = ops.gemm(xn, qw, qb, B * N, 3 * C, C)                                   # attention.py:22
        P0 = self.num_prefix_tokens
        keep = keep_count(N, self.keep_ratio, P0)
        if keep > N - P0:
            raise RuntimeError("selected index k out of range")                       # torch.topk's error, attention.py:35
        scores = None
        if self.update or prev_scores is None:                                        # attention.py:25-28
            scores, keep_idx, next_scores, row_map = ops.score_select(
                qkv.view(B, N, 3 * C), H, keep, want_scores=want_scores, prefix=P0)
        else:
            scores = prev_scores.detach().to(torch.float32).contiguous()
            keep_idx, next_scores, row_map = ops.select(scores, keep, prefix=P0)
        att = ops.attention(qkv, row_map, B, N, keep + P0, C, H, float(self.scale))   # attention.py:42-54
        out = ops.gemm(att, pw, pb, B * (keep + P0), C, C)                            # attention.py:55
        return out, keep_idx, next_scores, row_map, scores

    @torch.no_grad()
    def forward(self, x: torch.Tensor, prev_scores: Optional[torch.Tensor] = None):
        B, N, C = x.shape
        xn = x.detach().to(torch.bfloat16).contiguous().view(B * N, C)
        out, keep_idx, next_scores, _, _ = self.forward_packed(xn, prev_scores, B, N)
        return (out.view(B, -1, C).to(x.dtype), keep_idx.to(torch.int64), next_scores.to(x.dtype))
