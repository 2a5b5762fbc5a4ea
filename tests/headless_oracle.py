"""CPU reference for headless ViTs (``head`` = Identity, timm's ``num_classes=0``) — TEST INFRASTRUCTURE ONLY, built on
``tests/pool_prenorm_oracle.py``.

A headless model's output is what its head would read: ``norm(x)[:, 0]`` with class-token pooling, or
``fc_norm(mean of x[:, prefix:])`` with ``global_pool='avg'``, over the tokens the last block kept, with or without
``norm_pre``.  Blocks, selection and teacher forcing are the pooled / pre-norm reference's own functions; only the head is
left out.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import pool_prenorm_oracle as porc

Tensor = torch.Tensor


def extract_params(model) -> Dict:
    """``porc.extract_params`` with ``headless`` set.  ``orc.extract_params`` reads ``head.weight``: a headless model is
    handed a stand-in head for the call, and its head fields are a zero row the reference's head may multiply."""
    head = model.head
    if isinstance(head, nn.Linear):
        return dict(porc.extract_params(model), headless=False)
    model.head = nn.Linear(model.embed_dim, 1, device="meta")
    try:
        out = porc.extract_params(model)
    finally:
        model.head = head
    out.update(headless=True, head_w=torch.zeros(1, model.embed_dim, dtype=model.cls_token.dtype), head_b=None)
    return out


def features(params: Dict, x: Tensor) -> Tensor:
    """The head's input from the last block's output [B, N, C]: fc_norm of the patch tokens' mean, or the normalised
    class token."""
    C = x.shape[-1]
    if params.get("avg_pool"):
        w, b, eps = params["fc_norm"]
        return F.layer_norm(x[:, params.get("prefix", 1):].mean(dim=1), (C,), w, b, eps)
    return F.layer_norm(x[:, 0], (C,), params["norm_w"], params["norm_b"], params["norm_eps"])


@torch.no_grad()
def forward(params: Dict, images: Tensor, schedule: Dict, trace: Optional[List] = None,
            forced_keep: Optional[List[Optional[Tensor]]] = None) -> Tuple[Tensor, Dict]:
    """porc.forward returning the features [B, C] instead of logits; same ``trace`` records and ``forced_keep``."""
    trace = [] if trace is None else trace
    _, stats = porc.forward(params, images, schedule, trace=trace, forced_keep=forced_keep)
    return features(params, trace[-1]["x_out"]), stats
