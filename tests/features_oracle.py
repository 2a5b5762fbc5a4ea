"""CPU reference for token-level features of pruned ViTs (``forward_features`` / ``forward_intermediates``) — TEST
INFRASTRUCTURE ONLY, built on ``tests/headless_oracle.py`` and ``tests/pool_prenorm_oracle.py``.

The rule: a token pruned by block k keeps the features it had when it was dropped, which is its row in the input of
block k (the output of block k-1, the last block that kept it); a token never pruned has its row in the output of the
last block run.  Rows stay at their original positions (prefix tokens first, then the patches in raster order).  This
module assembles that map from a ``trace`` of ``porc.forward`` (per-block ``x_in``, ``x_out`` and ``keep_idx``), with
selection teacher-forced through ``forced_keep`` as in the other references, and applies the final ``norm`` (Identity for
an average-pooled model, whose params carry no ``norm_w``).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from tests import headless_oracle as horc
from tests import pool_prenorm_oracle as porc

Tensor = torch.Tensor
extract_params = horc.extract_params


def token_map(trace: List[Dict], depth: int) -> Tuple[Tensor, Tensor]:
    """The map after the first ``depth`` blocks of ``trace`` -> (rows [B, N0, C], depth int64 [B, N0])."""
    x0 = trace[0]["x_in"]
    B, N0, C = x0.shape
    out = torch.empty_like(x0)
    dep = torch.empty((B, N0), dtype=torch.long)
    pos = torch.arange(N0).expand(B, N0)                 # original position of each row of the current stage
    for rec in trace[:depth]:
        if rec["pruned"]:
            out.scatter_(1, pos[..., None].expand(-1, -1, C), rec["x_in"])
            dep.scatter_(1, pos, rec["block"])
            pos = torch.gather(pos, 1, rec["keep_idx"])
    out.scatter_(1, pos[..., None].expand(-1, -1, C), trace[depth - 1]["x_out"])
    dep.scatter_(1, pos, depth)
    return out, dep


def final_norm(params: Dict, x: Tensor) -> Tensor:
    """The model's final ``norm`` on every row: LayerNorm, or Identity for an average-pooled model."""
    if "norm_w" not in params:
        return x
    return F.layer_norm(x, (x.shape[-1],), params["norm_w"], params["norm_b"], params["norm_eps"])


@torch.no_grad()
def forward_features(params: Dict, images: Tensor, schedule: Dict,
                     forced_keep: Optional[List[Optional[Tensor]]] = None) -> Tuple[Tensor, Tensor, List[Dict], Dict]:
    """-> (norm of the token map after the last block [B, N0, C], depth map [B, N0], trace, stats)."""
    trace = []
    _, stats = porc.forward(params, images, schedule, trace=trace, forced_keep=forced_keep)
    x, dep = token_map(trace, len(trace))
    return final_norm(params, x), dep, trace, stats
