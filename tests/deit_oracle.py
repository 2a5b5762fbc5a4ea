"""CPU reference for the two DeiT families — TEST INFRASTRUCTURE ONLY, built on ``oracle/rajni_oracle.py``.

The reference the oracle restates runs ViTs with one class token and no LayerScale.  This module extends that
functional restatement (plain torch on CPU, fp32 or fp64) to what the DeiT families add, reusing the oracle's own
``importance``, ``mha``, ``mlp`` and schedule handling unchanged:
  * LayerScale (DeiT-III): ``x += ls(out)`` after attention and MLP, in pruned and dense blocks alike, as the
    reference's own blocks do (model.py:45-59);
  * ``prefix`` leading tokens (distilled DeiT: CLS and a distillation token) that selection always keeps; the top-k runs
    over the tokens after them, ``keep = max(1, int(ratio * (N - prefix)))``, and the output averages the two heads;
  * ``no_embed_class`` (DeiT-III): pos_embed has one row per patch, added to the patches before the class token is
    prepended.  The reference would fail on such a pos_embed (``pos_embed[:, :N]`` with P rows, model.py:37); this
    follows timm's ``_pos_embed`` there.
With one prefix token, no LayerScale and class-token positions every function computes what the oracle computes
(``tests/test_host_deit.py`` checks it on the golden cases).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from oracle import rajni_oracle as orc

Tensor = torch.Tensor
importance = orc.importance


def keep_count(num_tokens: int, keep_ratio: float, prefix: int = 1) -> int:
    """Patches kept (the ``prefix`` leading tokens excluded): Python double multiply then truncation, floor of 1."""
    return max(1, int(keep_ratio * (num_tokens - prefix)))


def select(scores: Tensor, keep: int, prefix: int = 1) -> Tensor:
    """Prefix-preserving ascending kept-token index, [B,N] -> int64 [B,keep+prefix]: tokens 0..prefix-1, then the top
    ``keep`` of scores[:,prefix:] (greater score first, then lower index, as ``orc.select``)."""
    B, N = scores.shape
    if keep > N - prefix:
        raise RuntimeError("selected index k out of range")       # what topk raises, attention.py:35
    order = torch.sort(scores[:, prefix:], dim=1, descending=True, stable=True).indices[:, :keep]
    idx = torch.sort(order, dim=1).values + prefix
    return torch.cat([torch.arange(prefix, dtype=torch.long).expand(B, prefix), idx], dim=1)


def tie_straddles_cut(scores: Tensor, keep: int, prefix: int = 1) -> Tensor:
    """bool [B]: the keep-th and (keep+1)-th largest scores after the prefix tokens are equal."""
    patch = scores[:, prefix:]
    if keep >= patch.shape[1]:
        return torch.zeros(scores.shape[0], dtype=torch.bool)
    s = torch.sort(patch, dim=1, descending=True).values
    return s[:, keep - 1] == s[:, keep]


def extract_params(model) -> Dict:
    """``orc.extract_params`` plus the DeiT fields: per-block LayerScale gammas (None where the block has none), the
    prefix count, ``no_embed_class`` and, for a distilled model, the distillation token and ``head_dist``."""
    out = orc.extract_params(model)
    for p, blk in zip(out["blocks"], model.blocks):
        for name in ("ls1", "ls2"):
            g = getattr(getattr(blk, name, None), "gamma", None)
            p[name] = None if g is None else g.detach()
    out["prefix"] = int(getattr(model, "num_prefix_tokens", 1))
    out["no_embed_class"] = bool(getattr(model, "no_embed_class", False))
    if getattr(model, "dist_token", None) is not None:
        out["dist"] = model.dist_token.detach()
        out["head_dist_w"] = model.head_dist.weight.detach()
        out["head_dist_b"] = None if model.head_dist.bias is None else model.head_dist.bias.detach()
    return out


def embed(params: Dict, images: Tensor) -> Tensor:
    """Patch-embed + CLS (+ distillation token) + position (timm ``_pos_embed``)."""
    p = params["patch"]
    x = F.conv2d(images, params["pe_w"], params["pe_b"], stride=p).flatten(2).transpose(1, 2)
    tokens = [params["cls"].expand(x.shape[0], -1, -1)]
    if params.get("dist") is not None:
        tokens.append(params["dist"].expand(x.shape[0], -1, -1))
    if params.get("no_embed_class", False):
        return torch.cat(tokens + [x + params["pos"][:, : x.shape[1]]], dim=1)
    x = torch.cat(tokens + [x], dim=1)
    return x + params["pos"][:, : x.shape[1]]


def _ls(out: Tensor, gamma: Optional[Tensor]) -> Tensor:
    return out if gamma is None else out * gamma


def dense_block(x: Tensor, blk: Dict) -> Tensor:
    """Un-pruned timm block with optional LayerScale."""
    C = x.shape[-1]
    H = blk["num_heads"]
    h = F.layer_norm(x, (C,), blk["n1_w"], blk["n1_b"], blk["n1_eps"])
    qkv = F.linear(h, blk["qkv_w"], blk["qkv_b"])
    x = x + _ls(F.linear(orc.mha(qkv, H, (C // H) ** -0.5), blk["proj_w"], blk["proj_b"]), blk.get("ls1"))
    return x + _ls(orc.mlp(x, blk), blk.get("ls2"))


def pruned_block(x: Tensor, scores: Optional[Tensor], blk: Dict, keep_ratio: float, update: bool,
                 forced_idx: Optional[Tensor] = None, prefix: int = 1):
    """orc.pruned_block with ``prefix`` always-kept tokens and optional LayerScale."""
    B, N, C = x.shape
    H = blk["num_heads"]
    h = F.layer_norm(x, (C,), blk["n1_w"], blk["n1_b"], blk["n1_eps"])
    qkv = F.linear(h, blk["qkv_w"], blk["qkv_b"])
    full = importance(qkv, H) if update or scores is None else scores
    keep = keep_count(N, keep_ratio, prefix)
    keep_idx = select(full, keep, prefix) if forced_idx is None else forced_idx.to(torch.long)
    assert keep_idx.shape == (B, keep + prefix)
    kept = torch.gather(qkv, 1, keep_idx[:, :, None].expand(-1, -1, 3 * C))
    out = F.linear(orc.mha(kept, H, (C // H) ** -0.5), blk["proj_w"], blk["proj_b"])
    x = torch.gather(x, 1, keep_idx[:, :, None].expand(-1, -1, C)) + _ls(out, blk.get("ls1"))
    x = x + _ls(orc.mlp(x, blk), blk.get("ls2"))
    return x, keep_idx, torch.gather(full, 1, keep_idx), full


@torch.no_grad()
def forward(params: Dict, images: Tensor, schedule: Dict, trace: Optional[List] = None,
            forced_keep: Optional[List[Optional[Tensor]]] = None) -> Tuple[Tensor, Dict]:
    """orc.forward for the DeiT families: same return values, ``trace`` records and ``forced_keep`` teacher forcing."""
    sched = orc.normalise_schedule(schedule)
    prefix = params.get("prefix", 1)
    x = embed(params, images)
    scores = None
    counts = []
    for i, blk in enumerate(params["blocks"]):
        counts.append(x.shape[1])
        rec = {"block": i, "x_in": x} if trace is not None else None
        if i in sched:
            ratio, update = sched[i]
            prev = scores
            forced = forced_keep[i] if forced_keep is not None else None
            x, keep_idx, scores, full = pruned_block(x, scores, blk, ratio, update, forced, prefix)
            if rec is not None:
                rec.update(pruned=True, keep_idx=keep_idx, scores=full, prev_scores=prev, next_scores=scores)
        else:
            x = dense_block(x, blk)
            scores = None
            if rec is not None:
                rec.update(pruned=False)
        if rec is not None:
            rec["x_out"] = x
            trace.append(rec)
    C = x.shape[-1]
    cls = F.layer_norm(x[:, 0], (C,), params["norm_w"], params["norm_b"], params["norm_eps"])
    logits = F.linear(cls, params["head_w"], params["head_b"])
    if params.get("head_dist_w") is not None:                   # distilled: the eval-mode average of the two heads
        dist = F.layer_norm(x[:, 1], (C,), params["norm_w"], params["norm_b"], params["norm_eps"])
        logits = (logits + F.linear(dist, params["head_dist_w"], params["head_dist_b"])) / 2
    return logits, {"token_counts": counts}
