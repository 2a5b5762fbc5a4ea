"""Real-weights path: load a timm-named ViT checkpoint into a model the wrapper can take.

The reference runs pretrained timm weights (``rajni/run.py:89-92,126-129``:
``timm.create_model(args.model, pretrained=True)``); timm and its hub are not available
here, so ``load_checkpoint`` takes the state dict itself — a ``.safetensors`` file, a
``torch.save``d ``.pt``/``.pth``/``.bin`` file, or a dict already in memory — and returns a
timm-attribute-compatible model (``rajni_vit_b200.vit.VisionTransformer``) carrying those
weights:

    base = load_checkpoint("vit_base_patch16_224.augreg_in21k_ft_in1k.safetensors")
    model = RAJNIViTWrapper(base, schedule).cuda().eval()

Accepted key families (SURVEY.md section 5):
  * timm's own:            ``cls_token``, ``pos_embed``, ``patch_embed.proj.*``, ``blocks.{i}.*``, ``norm.*``, ``head.*``
  * a saved RAJNI wrapper: the same keys under ``m.`` plus the aliased ``blocks.{i}.*`` duplicates
    (``RAJNIViTWrapper.blocks`` IS ``base_model.blocks``, ``model.py:9-10``) — duplicates must agree
  * wrappers around either: ``module.`` (DataParallel), ``model.``, and ``{"state_dict": ...}`` / ``{"model": ...}`` nesting

The architecture is inferred from the tensors' shapes (width from ``cls_token``, depth from
the block indices, image size from ``pos_embed``, classes from ``head.weight``, none without ``head.*``: timm's
``num_classes=0``, whose output is the pooled features); heads =
width / 64, the only head dimension the kernels (and every BASELINE config) use.  The two DeiT families load too:
  * DeiT-III: ``blocks.{i}.ls1.gamma`` / ``ls2.gamma`` (LayerScale, accepted only when every block has both), and a
    ``pos_embed`` with one row per patch (a square length: no position for the class token, timm's ``no_embed_class``);
  * distilled DeiT: ``dist_token`` together with ``head_dist.*``, ``pos_embed`` of patches + 2.
So do the two head / stem variants:
  * average pooling (MAE fine-tunes): ``fc_norm.weight`` and ``fc_norm.bias`` and no ``norm.*`` (timm
    ``global_pool='avg'``: the head reads fc_norm of the patch tokens' mean);
  * a pre-norm stem (CLIP fine-tunes): ``norm_pre.weight`` and ``norm_pre.bias``.  A checkpoint does not record LayerNorm
    eps; timm's CLIP ViTs, the models with this stem, use 1e-5 everywhere, so that is what a pre-norm model gets (1e-6
    otherwise);
  * a patch embedding without bias (CLIP): no ``patch_embed.proj.bias``.
Checkpoints outside the wrapper's contract — partial LayerScale, a partial ``norm_pre`` or ``fc_norm``, ``fc_norm`` next
to ``norm``, register tokens, a distillation token without its head, qk-norm — raise ``NotImplementedError`` naming the
offending keys: never a silent partial load.
"""
from __future__ import annotations

import json
import os
import re
import struct
from typing import Dict, Mapping, Optional, Union

import torch

from .vit import VisionTransformer

_SAFETENSORS_DTYPES = {"F32": torch.float32, "F16": torch.float16, "BF16": torch.bfloat16, "F64": torch.float64,
                       "I64": torch.int64, "I32": torch.int32, "U8": torch.uint8, "BOOL": torch.bool}

_UNSUPPORTED = (r"\.ls[12]\.(?!gamma$)", r"^norm_pre\.(?!(weight|bias)$)", r"^fc_norm\.(?!(weight|bias)$)", r"^reg_token$",
                r"\.attn\.[qk]_norm\.", r"^patch_embed\.norm\.", r"\.mlp\.norm\.", r"rel_pos", r"^pre_logits\.")


def read_safetensors(path: str) -> Dict[str, torch.Tensor]:
    """Minimal reader of the safetensors container (8-byte little-endian header length, JSON header, raw tensors)."""
    with open(path, "rb") as f:
        (n,) = struct.unpack("<Q", f.read(8))
        header = json.loads(f.read(n).decode("utf-8"))
        blob = f.read()
    out = {}
    for name, meta in header.items():
        if name == "__metadata__":
            continue
        dtype = _SAFETENSORS_DTYPES.get(meta["dtype"])
        if dtype is None:
            raise NotImplementedError(f"{path}: tensor {name!r} has unsupported dtype {meta['dtype']}")
        lo, hi = meta["data_offsets"]
        t = torch.frombuffer(bytearray(blob[lo:hi]), dtype=dtype) if hi > lo else torch.empty(0, dtype=dtype)
        out[name] = t.reshape(meta["shape"])
    return out


def write_safetensors(path: str, tensors: Mapping[str, torch.Tensor]) -> None:
    """The matching writer (tests, and exporting a model for the reference side)."""
    rev = {v: k for k, v in _SAFETENSORS_DTYPES.items()}
    header, chunks, off = {}, [], 0
    for name, t in tensors.items():
        t = t.detach().cpu().contiguous()
        raw = t.view(torch.uint8).numpy().tobytes() if t.numel() else b""
        header[name] = {"dtype": rev[t.dtype], "shape": list(t.shape), "data_offsets": [off, off + len(raw)]}
        chunks.append(raw)
        off += len(raw)
    hj = json.dumps(header, separators=(",", ":")).encode("utf-8")
    hj += b" " * (-len(hj) % 8)
    with open(path, "wb") as f:
        f.write(struct.pack("<Q", len(hj)))
        f.write(hj)
        for c in chunks:
            f.write(c)


def _read(path: str) -> Dict[str, torch.Tensor]:
    if path.endswith(".safetensors"):
        return read_safetensors(path)
    obj = torch.load(path, map_location="cpu", weights_only=True)
    if not isinstance(obj, Mapping):
        raise TypeError(f"{path}: expected a state dict, got {type(obj).__name__}")
    return dict(obj)


def normalise_keys(sd: Mapping[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """Strip container / wrapper prefixes and merge the wrapper's duplicated ``m.blocks.*`` / ``blocks.*`` families."""
    for nest in ("state_dict", "model", "model_state_dict"):
        if nest in sd and isinstance(sd[nest], Mapping) and not isinstance(sd[nest], torch.Tensor):
            sd = sd[nest]
    out: Dict[str, torch.Tensor] = {}
    for k, v in sd.items():
        if not isinstance(v, torch.Tensor):
            continue
        key = k
        changed = True
        while changed:                                         # module.m.blocks.0... -> blocks.0...
            changed = False
            for prefix in ("module.", "model.", "m."):
                if key.startswith(prefix):
                    key, changed = key[len(prefix):], True
        if key in out:
            if out[key].shape != v.shape or not torch.equal(out[key], v):
                raise ValueError(f"checkpoint holds two different tensors for {key!r} (the wrapper's m.blocks.* and blocks.* "
                                 "families alias one module and must agree)")
            continue
        out[key] = v
    return out


def infer_config(sd: Mapping[str, torch.Tensor]) -> Dict[str, int]:
    for k in ("cls_token", "pos_embed", "patch_embed.proj.weight"):
        if k not in sd:
            raise KeyError(f"checkpoint has no {k!r}: not a timm-named ViT state dict (keys start with {sorted(sd)[:4]})")
    # no head.* at all: a headless backbone (num_classes=0: DINO, MAE pretraining, in21k backbones)
    headless = "head.weight" not in sd
    if headless and "head.bias" in sd:
        raise KeyError("checkpoint has 'head.bias' but no 'head.weight'")
    if headless and ("dist_token" in sd or any(k.startswith("head_dist.") for k in sd)):
        raise NotImplementedError("a distillation token ('dist_token' / 'head_dist.*') without 'head.weight' is not supported: "
                                  "distilled models need their classifier heads")
    bad = sorted(k for k in sd if any(re.search(p, k) for p in _UNSUPPORTED))
    if bad:
        raise NotImplementedError(f"checkpoint uses features outside the RAJNI wrapper's contract: {bad[:6]}"
                                  f"{' ...' if len(bad) > 6 else ''}")
    # the final LayerNorm: `norm` before class-token pooling, or `fc_norm` after average pooling - never both, never partial
    fam = {name: sorted(k for k in sd if k.startswith(name + ".")) for name in ("norm", "fc_norm", "norm_pre")}
    for name, keys in fam.items():
        if keys and keys != [f"{name}.bias", f"{name}.weight"]:
            raise NotImplementedError(f"{name} must be a LayerNorm with weight and bias: the checkpoint has {keys}")
    if fam["fc_norm"] and fam["norm"]:
        raise NotImplementedError(f"fc_norm next to norm is not supported (average pooling has norm = Identity): {fam['fc_norm']} "
                                  f"and {fam['norm']}")
    if not fam["fc_norm"] and not fam["norm"]:
        raise KeyError("checkpoint has neither 'norm.weight' nor 'fc_norm.weight': not a timm-named ViT state dict")
    avg_pool, pre_norm = bool(fam["fc_norm"]), bool(fam["norm_pre"])
    if avg_pool and "dist_token" in sd:
        raise NotImplementedError("fc_norm (global_pool='avg') with a distillation token is not supported")
    C = sd["cls_token"].shape[-1]
    pw = sd["patch_embed.proj.weight"]
    if pw.dim() != 4 or pw.shape[1] != 3 or pw.shape[2] != pw.shape[3]:
        raise NotImplementedError(f"patch_embed.proj.weight has shape {tuple(pw.shape)}; expected [C, 3, p, p]")
    patch = pw.shape[2]
    blocks = {int(m.group(1)) for k in sd for m in [re.match(r"blocks\.(\d+)\.", k)] if m}
    if not blocks or blocks != set(range(len(blocks))):
        raise KeyError(f"block indices {sorted(blocks)} are not 0..depth-1")
    # LayerScale (DeiT-III): both gammas in every block, or none at all
    ls = sorted(k for k in sd if re.match(r"blocks\.\d+\.ls[12]\.gamma$", k))
    if ls and len(ls) != 2 * len(blocks):
        have = set(ls)
        odd = sorted(k for i in blocks for k in (f"blocks.{i}.ls1.gamma", f"blocks.{i}.ls2.gamma") if k not in have) or ls
        raise NotImplementedError(f"LayerScale must be in every block (ls1 and ls2): the checkpoint has {ls[:4]}"
                                  f"{' ...' if len(ls) > 4 else ''} but not {odd[:4]}")
    # distillation token (distilled DeiT): only together with its head
    dist = "dist_token" in sd
    head_dist = sorted(k for k in sd if k.startswith("head_dist."))
    if dist != bool(head_dist) or (dist and "head_dist.weight" not in sd):
        raise NotImplementedError("a distillation token needs its head and the head needs the token: checkpoint has "
                                  f"{['dist_token'] if dist else []} {head_dist}")
    # pos_embed layout from its length: patches (square, no position for the class token), + 1 (class token), + 2 (distilled)
    n_tok = sd["pos_embed"].shape[1]
    prefix = 2 if dist else 1
    grid = int(round(max(n_tok - prefix, 0) ** 0.5))
    no_embed_class = False
    if grid * grid != n_tok - prefix:
        grid = int(round(n_tok ** 0.5))
        no_embed_class = True
        if grid * grid != n_tok:
            raise NotImplementedError(f"pos_embed has {n_tok} positions: not a square grid of patches, plus {prefix} "
                                      f"({'class and distillation tokens' if dist else 'class token'}) or plus none")
    if C % 64:
        raise NotImplementedError(f"width {C} is not a multiple of the head dimension 64")
    hidden = sd["blocks.0.mlp.fc1.weight"].shape[0]
    return dict(embed_dim=C, depth=len(blocks), num_heads=C // 64, img_size=grid * patch, patch_size=patch,
                num_classes=0 if headless else sd["head.weight"].shape[0], mlp_ratio=hidden / C, init_values=1.0 if ls else None,
                no_embed_class=no_embed_class, distilled=dist, global_pool="avg" if avg_pool else "token", fc_norm=avg_pool,
                pre_norm=pre_norm, patch_bias="patch_embed.proj.bias" in sd, norm_eps=1e-5 if pre_norm else 1e-6)


def load_checkpoint(source: Union[str, os.PathLike, Mapping[str, torch.Tensor]], model: Optional[torch.nn.Module] = None,
                    strict: bool = True) -> torch.nn.Module:
    """Load timm-named ViT weights; returns ``model`` (or a new stand-in ViT built from the checkpoint's shapes), eval mode.

    ``strict``: every parameter of the model must be present and every checkpoint tensor must be used (buffers such as
    ``num_batches_tracked`` do not exist in a ViT; anything left over is an error, not a warning)."""
    sd = normalise_keys(_read(os.fspath(source)) if isinstance(source, (str, os.PathLike)) else source)
    cfg = infer_config(sd)
    if model is None:
        model = VisionTransformer(**cfg)
    target = model.m if hasattr(model, "pruning_schedule") and hasattr(model, "m") else model      # a RAJNIViTWrapper: its base
    want = target.state_dict()
    missing = sorted(k for k in want if k not in sd)
    unexpected = sorted(k for k in sd if k not in want)
    shape_bad = sorted(k for k in want if k in sd and tuple(sd[k].shape) != tuple(want[k].shape))
    if shape_bad:
        k = shape_bad[0]
        raise ValueError(f"shape mismatch for {k!r}: checkpoint {tuple(sd[k].shape)} vs model {tuple(want[k].shape)}"
                         f" ({len(shape_bad)} tensors)")
    if strict and (missing or unexpected):
        raise KeyError(f"checkpoint does not match the model: missing {missing[:5]}, unexpected {unexpected[:5]}")
    with torch.no_grad():
        for k, p in want.items():
            if k in sd:
                p.copy_(sd[k].to(p.dtype))
    return model.eval()
