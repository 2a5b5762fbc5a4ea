"""Kernel-ready views of a timm-style ViT's parameters.

bf16 row-major weights ([out, in], the nn.Linear layout the GEMM consumes as-is),
fp32 biases and LayerNorm affines.  Packs are cached per module and rebuilt when a
parameter's storage, version, dtype or device changes, so ``.to()``, ``.bfloat16()``
and ``load_state_dict`` are honoured.  If a parameter already is contiguous bf16 the
pack aliases it (no copy).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn


def _sig(*tensors: Optional[torch.Tensor]):
    return tuple(None if t is None else (t.data_ptr(), t._version, t.dtype, t.device) for t in tensors)


class PackCache:
    def __init__(self):
        self._store: Dict[int, Tuple[tuple, tuple]] = {}

    def clear(self):
        self._store.clear()

    def linear(self, m: nn.Module) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """(weight bf16 [N,K] contiguous, bias fp32 [N] or None) for Linear / Conv2d(k=stride)."""
        w, b = m.weight, getattr(m, "bias", None)
        sig = _sig(w, b)
        hit = self._store.get(id(m))
        if hit is not None and hit[0] == sig:
            return hit[1]
        wd = w.detach()
        if wd.dim() > 2:
            wd = wd.reshape(wd.shape[0], -1)
        packed = (wd.to(torch.bfloat16).contiguous(),
                  None if b is None else b.detach().to(torch.float32).contiguous())
        self._store[id(m)] = (sig, packed)
        return packed

    def linear_ln(self, lin: nn.Module, norm: nn.LayerNorm):
        """LayerNorm folded into the Linear that follows it (model.py:51 -> attention.py:22, model.py:59 -> fc1):
        (W' = bf16(W*gamma) [N,K], b' = b + W beta fp32 [N], wsum[n] = sum_k W'[n,k] fp32, eps)."""
        sig = _sig(lin.weight, getattr(lin, "bias", None), norm.weight, norm.bias)
        key = (id(lin), "ln")
        hit = self._store.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        w = lin.weight.detach().to(torch.float32)
        gamma = norm.weight.detach().to(torch.float32)
        beta = norm.bias.detach().to(torch.float32)
        wg = (w * gamma[None, :]).to(torch.bfloat16).contiguous()
        bias = w @ beta
        if getattr(lin, "bias", None) is not None:
            bias = bias + lin.bias.detach().to(torch.float32)
        packed = (wg, bias.contiguous(), wg.to(torch.float32).sum(dim=1).contiguous(), float(norm.eps))
        self._store[key] = (sig, packed)
        return packed

    def linear_ls(self, lin: nn.Module, ls: nn.Module) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
        """LayerScale folded into the Linear that feeds the residual (DeiT-III's ls1 after proj, ls2 after fc2):
        x + gamma*(W a + b) = x + (gamma[:,None]*W) a + gamma*b  ->  (bf16(gamma[:,None]*W) [N,K], fp32 gamma*b [N] or None).
        The product is rounded to bf16 once; bf16 keeps its relative precision down to ~1e-38, so a gamma of 1e-6 costs no
        more than the weights' own rounding."""
        sig = _sig(lin.weight, getattr(lin, "bias", None), ls.gamma)
        key = (id(lin), "ls")
        hit = self._store.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        gamma = ls.gamma.detach().to(torch.float32)
        w = lin.weight.detach().to(torch.float32)
        b = getattr(lin, "bias", None)
        packed = ((w * gamma[:, None]).to(torch.bfloat16).contiguous(),
                  None if b is None else (b.detach().to(torch.float32) * gamma).contiguous())
        self._store[key] = (sig, packed)
        return packed

    def norm(self, m: nn.LayerNorm) -> Tuple[torch.Tensor, torch.Tensor, float]:
        sig = _sig(m.weight, m.bias)
        hit = self._store.get(id(m))
        if hit is not None and hit[0] == sig:
            return hit[1]
        packed = (m.weight.detach().to(torch.float32).contiguous(),
                  m.bias.detach().to(torch.float32).contiguous(), float(m.eps))
        self._store[id(m)] = (sig, packed)
        return packed

    def tensors(self, key, srcs, build):
        """Generic cached derivation from a tuple of source tensors."""
        sig = _sig(*srcs)
        hit = self._store.get(key)
        if hit is not None and hit[0] == sig:
            return hit[1]
        packed = build()
        self._store[key] = (sig, packed)
        return packed
