"""A timm-attribute-compatible ViT used as the base model in tests and benches.

The reference drives a ``timm`` VisionTransformer (``/root/reference/rajni/run.py:89-92``)
but only ever touches a small duck-typed surface of it
(``/root/reference/rajni/wrapper/model.py:10,34-37,45-66`` and
``/root/reference/rajni/wrapper/attention.py:8-12``).  timm is not installed in
this image and there is no network, so this module provides a model with exactly
those attribute names and timm's ViT semantics:

    patch_embed.proj : Conv2d(3, C, k=p, s=p)  -> flatten(2).transpose(1, 2)   (p = 16, or 8 / 32, see VIT_PATCH)
    cls_token [1,1,C], pos_embed [1,1+P,C], pos_drop
    blocks[i] : norm1, attn{num_heads, scale, qkv, proj, proj_drop}, norm2,
                mlp{fc1, act=GELU(erf), fc2}, ls1/ls2/drop_path1/drop_path2 = Identity
    norm, head

(and timm's ``norm_pre``, ``fc_norm`` = Identity), and the two DeiT families (extra fields in VIT_VARIANT):

    DeiT-III (``deit3_*``): ls1/ls2 = LayerScale (``gamma`` [C]), and no position for the class token
        (timm's ``no_embed_class``: pos_embed [1,P,C] is added to the patches before the class token is prepended);
    distilled DeiT (``deit_*_distilled_*``): a distillation token after the class token (``dist_token``,
        ``num_prefix_tokens = 2``, pos_embed [1,2+P,C]) and a second head ``head_dist`` on it; in eval mode the output is
        ``(head(x[:,0]) + head_dist(x[:,1])) / 2``;

and two head / stem variants (extra fields in VIT_POOL_PRENORM):

    average pooling (MAE fine-tunes, ``*_mae``): ``global_pool='avg'``, ``norm`` = Identity and ``fc_norm`` = LayerNorm,
        the output is ``head(fc_norm(x[:, 1:].mean(1)))`` (timm's ``forward_head``);
    a pre-norm stem (CLIP, ``*_clip_*``): a patch embedding without bias, ``norm_pre`` = LayerNorm applied to the embedded
        tokens before block 0, and LayerNorm eps 1e-5 everywhere.

Any of them built with ``num_classes=0`` is headless, as in timm: ``head`` = Identity and the output is the pooled,
normalised features [B, C].  The DINO backbones (``*_dino``, extra fields in VIT_HEADLESS) are built that way.

It is a plain eager PyTorch module.  It is NOT on the accelerated path: the
B200 wrapper reads its leaf parameters and runs its own kernels.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

# name -> (embed_dim, depth, heads, img_size); the patch size is in VIT_PATCH (callers unpack these four fields)
VIT_CONFIGS = {
    "vit_tiny_patch16_224": (192, 12, 3, 224),
    "vit_small_patch16_224": (384, 12, 6, 224),
    "vit_base_patch16_224": (768, 12, 12, 224),
    "vit_large_patch16_224": (1024, 24, 16, 224),
    "deit_base_patch16_384": (768, 12, 12, 384),
    "vit_small_patch32_224": (384, 12, 6, 224),
    "vit_base_patch32_224": (768, 12, 12, 224),
    "vit_small_patch8_224": (384, 12, 6, 224),
    "vit_base_patch8_224": (768, 12, 12, 224),
    # 4-block models small enough for golden fixtures and oracle runs: 17 tokens, 82 tokens (72 px is not a multiple of 16)
    # and 17 tokens again at patch 32
    "vit_micro_patch16_64": (128, 4, 2, 64),
    "vit_micro_patch8_72": (128, 4, 2, 72),
    "vit_micro_patch32_128": (128, 4, 2, 128),
    # DeiT-III (LayerScale, class token without a position) and distilled DeiT (class + distillation token, two heads)
    "deit3_small_patch16_224": (384, 12, 6, 224),
    "deit3_medium_patch16_224": (512, 12, 8, 224),
    "deit3_base_patch16_224": (768, 12, 12, 224),
    "deit3_large_patch16_224": (1024, 24, 16, 224),
    "deit3_base_patch16_384": (768, 12, 12, 384),
    "deit_tiny_distilled_patch16_224": (192, 12, 3, 224),
    "deit_small_distilled_patch16_224": (384, 12, 6, 224),
    "deit_base_distilled_patch16_224": (768, 12, 12, 224),
    "deit_base_distilled_patch16_384": (768, 12, 12, 384),
    # 4-block test models of the two families: 16 + 1 and 16 + 2 tokens
    "deit3_micro_patch16_64": (128, 4, 2, 64),
    "deit_micro_distilled_patch16_64": (128, 4, 2, 64),
    # average pooling with fc_norm (MAE fine-tunes) and a pre-norm stem (CLIP fine-tunes), and a 4-block test model of each
    "vit_base_patch16_224_mae": (768, 12, 12, 224),
    "vit_large_patch16_224_mae": (1024, 24, 16, 224),
    "vit_base_patch16_clip_224": (768, 12, 12, 224),
    "vit_base_patch32_clip_224": (768, 12, 12, 224),
    "vit_base_patch16_clip_384": (768, 12, 12, 384),
    "vit_micro_patch16_64_mae": (128, 4, 2, 64),
    "vit_micro_patch16_64_clip": (128, 4, 2, 64),
    # headless self-supervised backbones (DINO: num_classes=0, the output is the normalised class token), and a 4-block test
    # model
    "vit_small_patch16_224_dino": (384, 12, 6, 224),
    "vit_base_patch16_224_dino": (768, 12, 12, 224),
    "vit_small_patch8_224_dino": (384, 12, 6, 224),
    "vit_base_patch8_224_dino": (768, 12, 12, 224),
    "vit_micro_patch16_64_dino": (128, 4, 2, 64),
}
# name -> patch size (pixels per side of a patch; 50 tokens at 224 px for 32, 785 for 8)
VIT_PATCH = {name: 16 for name in VIT_CONFIGS}
VIT_PATCH.update({"vit_small_patch32_224": 32, "vit_base_patch32_224": 32, "vit_micro_patch32_128": 32, "vit_base_patch32_clip_224": 32,
                  "vit_small_patch8_224": 8, "vit_base_patch8_224": 8, "vit_micro_patch8_72": 8,
                  "vit_small_patch8_224_dino": 8, "vit_base_patch8_224_dino": 8})
# name -> extra VisionTransformer arguments of the DeiT families (timm's deit3_* use init_values=1e-6 and no_embed_class;
# create_model spreads the LayerScale gammas, see spread_layer_scale)
_DEIT3 = dict(init_values=1e-6, no_embed_class=True)
VIT_VARIANT = {name: dict(_DEIT3) for name in VIT_CONFIGS if name.startswith("deit3_")}
VIT_VARIANT.update({name: dict(distilled=True) for name in VIT_CONFIGS if "_distilled_" in name})
# name -> extra VisionTransformer arguments of the pooled and pre-norm families (timm's *_mae fine-tunes: global_pool='avg',
# fc_norm; *_clip_*: pre_norm, no patch-embed bias, LayerNorm eps 1e-5)
VIT_POOL_PRENORM = {name: dict(global_pool="avg", fc_norm=True) for name in VIT_CONFIGS if name.endswith("_mae")}
VIT_POOL_PRENORM.update({name: dict(pre_norm=True, patch_bias=False, norm_eps=1e-5) for name in VIT_CONFIGS if "_clip" in name})
# name -> extra VisionTransformer arguments of the headless models (timm's *.dino weights: num_classes=0, head = Identity)
VIT_HEADLESS = {name: dict(num_classes=0) for name in VIT_CONFIGS if name.endswith("_dino")}


class PatchEmbed(nn.Module):
    def __init__(self, img_size, patch, in_chans, dim, bias=True):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch, patch)
        self.grid_size = (img_size // patch, img_size // patch)
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, dim, kernel_size=patch, stride=patch, bias=bias)
        self.norm = nn.Identity()

    def forward(self, x):
        return self.norm(self.proj(x).flatten(2).transpose(1, 2))


class Attention(nn.Module):
    fused_attn = True

    def __init__(self, dim, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.q_norm = nn.Identity()
        self.k_norm = nn.Identity()
        self.attn_drop = nn.Dropout(0.0)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(0.0)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        x = F.scaled_dot_product_attention(q, k, v)
        x = x.transpose(1, 2).reshape(B, N, C)
        return self.proj_drop(self.proj(x))


class Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.drop1 = nn.Dropout(0.0)
        self.norm = nn.Identity()
        self.fc2 = nn.Linear(hidden, dim)
        self.drop2 = nn.Dropout(0.0)

    def forward(self, x):
        return self.drop2(self.fc2(self.norm(self.drop1(self.act(self.fc1(x))))))


class LayerScale(nn.Module):
    """timm's LayerScale: x * gamma, gamma [C] learnt per channel (DeiT-III, CaiT)."""

    def __init__(self, dim, init_values=1e-5):
        super().__init__()
        self.gamma = nn.Parameter(init_values * torch.ones(dim))

    def forward(self, x):
        return x * self.gamma


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, init_values=None, norm_eps=1e-6):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=norm_eps)
        self.attn = Attention(dim, num_heads)
        self.ls1 = LayerScale(dim, init_values) if init_values else nn.Identity()
        self.drop_path1 = nn.Identity()
        self.norm2 = nn.LayerNorm(dim, eps=norm_eps)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))
        self.ls2 = LayerScale(dim, init_values) if init_values else nn.Identity()
        self.drop_path2 = nn.Identity()

    def forward(self, x):
        x = x + self.drop_path1(self.ls1(self.attn(self.norm1(x))))
        x = x + self.drop_path2(self.ls2(self.mlp(self.norm2(x))))
        return x


class VisionTransformer(nn.Module):
    """``init_values``: LayerScale after attention and MLP (None: Identity).  ``no_embed_class``: pos_embed covers the patches
    only.  ``distilled``: a distillation token and ``head_dist`` (timm's VisionTransformerDistilled, eval-mode output).
    ``global_pool``: 'token' (class token) or 'avg' (mean of the tokens after the prefix); ``fc_norm``: the final LayerNorm
    after pooling instead of before it (None: timm's default, on for 'avg').  ``pre_norm``: ``norm_pre`` LayerNorm after the
    embedding.  ``patch_bias``: the patch projection has a bias.  ``norm_eps``: eps of every LayerNorm.  ``num_classes=0``:
    ``head`` (and ``head_dist``) = Identity, timm's headless model."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000,
                 embed_dim=768, depth=12, num_heads=12, mlp_ratio=4.0, init_values=None, no_embed_class=False,
                 distilled=False, global_pool="token", fc_norm=None, pre_norm=False, patch_bias=True, norm_eps=1e-6):
        super().__init__()
        use_fc_norm = global_pool == "avg" if fc_norm is None else fc_norm
        self.num_classes = num_classes
        self.embed_dim = self.num_features = embed_dim
        self.global_pool = global_pool
        self.num_prefix_tokens = 2 if distilled else 1
        self.no_embed_class = no_embed_class
        self.patch_embed = PatchEmbed(img_size, patch_size, in_chans, embed_dim, bias=patch_bias)
        n_tok = self.patch_embed.num_patches + (0 if no_embed_class else self.num_prefix_tokens)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.dist_token = nn.Parameter(torch.zeros(1, 1, embed_dim)) if distilled else None
        self.pos_embed = nn.Parameter(torch.zeros(1, n_tok, embed_dim))
        self.pos_drop = nn.Dropout(0.0)
        self.patch_drop = nn.Identity()
        self.norm_pre = nn.LayerNorm(embed_dim, eps=norm_eps) if pre_norm else nn.Identity()
        self.blocks = nn.Sequential(*[Block(embed_dim, num_heads, mlp_ratio, init_values, norm_eps) for _ in range(depth)])
        self.norm = nn.Identity() if use_fc_norm else nn.LayerNorm(embed_dim, eps=norm_eps)
        self.fc_norm = nn.LayerNorm(embed_dim, eps=norm_eps) if use_fc_norm else nn.Identity()
        self.head_drop = nn.Dropout(0.0)
        self.head = nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        self.head_dist = (nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()) if distilled else None
        nn.init.normal_(self.cls_token, std=0.02)
        nn.init.normal_(self.pos_embed, std=0.02)
        if distilled:
            nn.init.normal_(self.dist_token, std=0.02)

    def _pos_embed(self, x):
        prefix = [self.cls_token.expand(x.shape[0], -1, -1)]
        if self.dist_token is not None:
            prefix.append(self.dist_token.expand(x.shape[0], -1, -1))
        if self.no_embed_class:                                 # timm: positions for the patches only, tokens prepended after
            return self.pos_drop(torch.cat(prefix + [x + self.pos_embed], dim=1))
        return self.pos_drop(torch.cat(prefix + [x], dim=1) + self.pos_embed)

    def forward_features(self, x):
        x = self._pos_embed(self.patch_embed(x))
        x = self.blocks(self.norm_pre(self.patch_drop(x)))
        return self.norm(x)

    def forward(self, x):
        x = self.forward_features(x)
        if self.head_dist is not None:                          # timm VisionTransformerDistilled, eval mode
            return (self.head(self.head_drop(x[:, 0])) + self.head_dist(self.head_drop(x[:, 1]))) / 2
        x = x[:, self.num_prefix_tokens:].mean(dim=1) if self.global_pool == "avg" else x[:, 0]     # timm forward_head
        return self.head(self.head_drop(self.fc_norm(x)))


def create_model(name: str, seed: int | None = 0, bf16_round: bool = True,
                 num_classes: int | None = None) -> VisionTransformer:
    """Random-init stand-in for ``timm.create_model(name)`` (no pretrained weights exist here).

    seed: torch CPU RNG seed for the init (SURVEY.md section 8d: manual_seed(0)).
    bf16_round: round every parameter to a bf16-representable fp32 value so that the
        fp32 oracle and the bf16 kernel path share bit-identical weights.
    num_classes: None = the model's own (1000, or 0 for the headless models of VIT_HEADLESS); 0 = headless.
    """
    dim, depth, heads, img = VIT_CONFIGS[name]
    if seed is not None:
        gen_state = torch.random.get_rng_state()
        torch.manual_seed(seed)
    variant = {"num_classes": 1000, **VIT_VARIANT.get(name, {}), **VIT_POOL_PRENORM.get(name, {}), **VIT_HEADLESS.get(name, {})}
    if num_classes is not None:
        variant["num_classes"] = num_classes
    model = VisionTransformer(img_size=img, patch_size=VIT_PATCH[name], embed_dim=dim, depth=depth, num_heads=heads, **variant)
    if seed is not None:
        torch.random.set_rng_state(gen_state)
    if variant.get("init_values"):
        spread_layer_scale(model, seed=0 if seed is None else seed, bf16_round=False)
    if bf16_round:
        with torch.no_grad():
            for p in model.parameters():
                p.copy_(p.to(torch.bfloat16).to(torch.float32))
    return model.eval()


def spread_layer_scale(model: VisionTransformer, seed: int = 0, lo: float = 1e-6, hi: float = 1.0,
                       bf16_round: bool = True) -> VisionTransformer:
    """Give every LayerScale gamma values spread log-uniformly over [lo, hi] (DeiT-III's trained gammas range from its
    1e-6 init to O(1)); a constant gamma would leave the per-channel fold untested.  Own generator: the other parameters
    are not touched."""
    g = torch.Generator().manual_seed(1000 + seed)
    lo_, hi_ = torch.log(torch.tensor(lo)), torch.log(torch.tensor(hi))
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith(".gamma"):
                p.copy_(torch.exp(lo_ + (hi_ - lo_) * torch.rand(p.shape, generator=g)))
                if bf16_round:
                    p.copy_(p.to(torch.bfloat16).to(torch.float32))
    return model


def randomize_trained_like(model: VisionTransformer, seed: int = 0, outlier_channels: int = 4, outlier_scale: float = 20.0,
                           bf16_round: bool = True) -> VisionTransformer:
    """Give a random-init stand-in the parameter STATISTICS of a trained ViT (no pretrained weights exist offline):
    LayerNorm gains spread over [0.3, 2.5] and non-zero shifts, biases of O(0.5), and a few "massive activation"
    channels - residual-stream channels that every block's fc2 / proj pushes far from zero, with the matching large
    LayerNorm gains trained models show there.  Exercises the folded-LayerNorm path (W*gamma, b + W beta, E[x^2]-mean^2
    statistics at large |mean|/sigma) that gamma = 1, beta = 0 never touches."""
    g = torch.Generator().manual_seed(seed)
    C = model.embed_dim
    hot = torch.randperm(C, generator=g)[:outlier_channels]
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("norm1.weight") or name.endswith("norm2.weight") or name in ("norm.weight", "fc_norm.weight",
                                                                                        "norm_pre.weight"):
                p.copy_(0.3 + 2.2 * torch.rand(p.shape, generator=g))
            elif name.endswith("norm1.bias") or name.endswith("norm2.bias") or name in ("norm.bias", "fc_norm.bias", "norm_pre.bias"):
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
            elif name.endswith(".bias"):
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
        for blk in model.blocks:
            blk.mlp.fc2.bias[hot] += outlier_scale * (0.5 + torch.rand(outlier_channels, generator=g))
            blk.attn.proj.bias[hot] -= 0.25 * outlier_scale * torch.rand(outlier_channels, generator=g)
            for nrm in (blk.norm1, blk.norm2):
                nrm.weight[hot] *= 0.1                      # trained models damp their massive channels at the next norm
        model.pos_embed[..., hot] += outlier_scale
        if bf16_round:
            for p in model.parameters():
                p.copy_(p.to(torch.bfloat16).to(torch.float32))
    return model
