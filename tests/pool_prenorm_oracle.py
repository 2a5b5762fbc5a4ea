"""CPU reference for average-pooled heads and the pre-norm stem — TEST INFRASTRUCTURE ONLY, built on
``tests/deit_oracle.py`` (itself built on ``oracle/rajni_oracle.py``).

It adds to the DeiT reference, in plain torch on CPU (fp32 or fp64), what the two timm ViT variants add:
  * ``norm_pre`` (CLIP fine-tunes): a LayerNorm over the embedded tokens before block 0;
  * a patch embedding without bias (``pe_b`` None; the oracle's conv already takes that);
  * ``global_pool='avg'`` with ``fc_norm`` (MAE fine-tunes): the logits are ``head(fc_norm(mean of x[:, prefix:]))``
    over the tokens the last block kept, and ``norm`` is not applied (timm's ``forward_head``).
Blocks, selection and teacher forcing are the DeiT reference's own functions.  With neither feature on ``forward`` computes
what ``deit_oracle.forward`` computes (``tests/test_host_pool_prenorm.py`` checks the bits).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import rajni_oracle as orc
from tests import deit_oracle as dorc

Tensor = torch.Tensor


def _ln(m) -> Optional[Tuple[Tensor, Tensor, float]]:
    return (m.weight.detach(), m.bias.detach(), m.eps) if isinstance(m, nn.LayerNorm) else None


def extract_params(model) -> Dict:
    """``dorc.extract_params`` plus ``norm_pre`` and the pooling (``avg_pool``, ``fc_norm`` as (weight, bias, eps) or
    None).  A pooled model has no ``norm``: its final-norm fields are left out."""
    norm = model.norm
    if not isinstance(norm, nn.LayerNorm):              # orc.extract_params reads norm.weight: hand it a stand-in
        model.norm = nn.LayerNorm(model.embed_dim)
    try:
        out = dorc.extract_params(model)
    finally:
        model.norm = norm
    if not isinstance(norm, nn.LayerNorm):
        for k in ("norm_w", "norm_b", "norm_eps"):
            del out[k]
    out["norm_pre"] = _ln(getattr(model, "norm_pre", None))
    out["avg_pool"] = getattr(model, "global_pool", "token") == "avg"
    out["fc_norm"] = _ln(getattr(model, "fc_norm", None))
    return out


def head(params: Dict, x: Tensor) -> Tensor:
    """Logits from the last block's output: fc_norm of the patch tokens' mean, or dorc's class-token head."""
    C = x.shape[-1]
    if params.get("avg_pool"):
        w, b, eps = params["fc_norm"]
        pooled = F.layer_norm(x[:, params.get("prefix", 1):].mean(dim=1), (C,), w, b, eps)
        return F.linear(pooled, params["head_w"], params["head_b"])
    cls = F.layer_norm(x[:, 0], (C,), params["norm_w"], params["norm_b"], params["norm_eps"])
    logits = F.linear(cls, params["head_w"], params["head_b"])
    if params.get("head_dist_w") is not None:                   # distilled: the eval-mode average of the two heads
        dist = F.layer_norm(x[:, 1], (C,), params["norm_w"], params["norm_b"], params["norm_eps"])
        logits = (logits + F.linear(dist, params["head_dist_w"], params["head_dist_b"])) / 2
    return logits


@torch.no_grad()
def forward(params: Dict, images: Tensor, schedule: Dict, trace: Optional[List] = None,
            forced_keep: Optional[List[Optional[Tensor]]] = None) -> Tuple[Tensor, Dict]:
    """dorc.forward with ``norm_pre`` after the embedding and the pooled head: same return values, ``trace`` records and
    ``forced_keep`` teacher forcing."""
    sched = orc.normalise_schedule(schedule)
    prefix = params.get("prefix", 1)
    x = dorc.embed(params, images)
    if params.get("norm_pre") is not None:
        w, b, eps = params["norm_pre"]
        x = F.layer_norm(x, (x.shape[-1],), w, b, eps)
    scores = None
    counts = []
    for i, blk in enumerate(params["blocks"]):
        counts.append(x.shape[1])
        rec = {"block": i, "x_in": x} if trace is not None else None
        if i in sched:
            ratio, update = sched[i]
            prev = scores
            forced = forced_keep[i] if forced_keep is not None else None
            x, keep_idx, scores, full = dorc.pruned_block(x, scores, blk, ratio, update, forced, prefix)
            if rec is not None:
                rec.update(pruned=True, keep_idx=keep_idx, scores=full, prev_scores=prev, next_scores=scores)
        else:
            x = dorc.dense_block(x, blk)
            scores = None
            if rec is not None:
                rec.update(pruned=False)
        if rec is not None:
            rec["x_out"] = x
            trace.append(rec)
    return head(params, x), {"token_counts": counts}
