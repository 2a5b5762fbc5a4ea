"""CPU-side tests of headless ViTs (head = Identity, timm's num_classes=0: DINO and other backbones): the stand-ins and the
reference (tests/headless_oracle.py) against timm's forward semantics, what the wrapper accepts and refuses, checkpoint
loading, the schedule tools' feature quality and the CLI's refusal."""
import json
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import headless_oracle as horc
from tests import pool_prenorm_oracle as porc
from rajni_vit_b200 import schedule as S
from rajni_vit_b200.checkpoint import load_checkpoint, write_safetensors
from rajni_vit_b200.vit import (VIT_CONFIGS, VIT_HEADLESS, VIT_PATCH, VIT_POOL_PRENORM, VIT_VARIANT, VisionTransformer,
                                create_model, randomize_trained_like)
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images

DINO = ["vit_small_patch16_224_dino", "vit_base_patch16_224_dino", "vit_small_patch8_224_dino", "vit_base_patch8_224_dino",
        "vit_micro_patch16_64_dino"]


def _micro(name, seed=3, num_classes=None):
    return randomize_trained_like(create_model(name, seed=seed, num_classes=num_classes), seed=seed + 1)


# ------------------------------------------------------------------ stand-ins and the reference
def test_stand_in_layouts():
    assert set(VIT_HEADLESS) == set(DINO)
    assert not set(VIT_HEADLESS) & (set(VIT_POOL_PRENORM) | set(VIT_VARIANT))
    for name in DINO:
        m = create_model(name, seed=None)
        dim, depth, heads, img = VIT_CONFIGS[name]
        assert isinstance(m.head, nn.Identity) and m.num_classes == 0 and m.global_pool == "token"
        assert isinstance(m.norm, nn.LayerNorm) and isinstance(m.fc_norm, nn.Identity) and isinstance(m.norm_pre, nn.Identity)
        assert all(n.eps == 1e-6 for n in m.modules() if isinstance(n, nn.LayerNorm))
        assert m.patch_embed.proj.kernel_size == (VIT_PATCH[name],) * 2 and m.embed_dim == dim and len(m.blocks) == depth
        assert not any(k.startswith("head") for k in m.state_dict())
    assert VIT_PATCH["vit_base_patch8_224_dino"] == 8 and VIT_PATCH["vit_small_patch16_224_dino"] == 16


def test_num_classes():
    """An explicit num_classes wins, and num_classes=0 gives any stand-in timm's Identity head."""
    m = create_model("vit_micro_patch16_64_dino", num_classes=10)
    assert isinstance(m.head, nn.Linear) and m.head.out_features == 10
    a, b = create_model("vit_micro_patch16_64"), create_model("vit_micro_patch16_64", num_classes=0)
    assert a.head.out_features == 1000 and isinstance(b.head, nn.Identity)
    assert set(a.state_dict()) - set(b.state_dict()) == {"head.weight", "head.bias"}
    m = create_model("deit_micro_distilled_patch16_64", num_classes=0)
    assert isinstance(m.head, nn.Identity) and isinstance(m.head_dist, nn.Identity)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip"])
def test_headless_forward_is_the_classifiers_head_input(name):
    """timm's semantics: with head = Identity the output is what a Linear head reads (norm(x)[:, 0], or fc_norm of the
    patch tokens' mean)."""
    base = _micro(name, num_classes=0)
    images = make_images(3, 64, 6)
    feats = base(images)
    assert feats.shape == (3, 128)
    base.head = nn.Linear(128, 128)
    with torch.no_grad():
        base.head.weight.copy_(torch.eye(128))
        base.head.bias.zero_()
    torch.testing.assert_close(base(images), feats, rtol=1e-6, atol=1e-6)
    x = base.forward_features(images)
    want = base.fc_norm(x[:, 1:].mean(1)) if "mae" in name else x[:, 0]
    assert torch.equal(feats, want)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip",
                                  "vit_small_patch16_224_dino"])
def test_reference_equals_the_stand_in_forward(name):
    """fp64: the headless reference is the stand-ins' own forward."""
    base = (_micro(name, num_classes=0) if "micro" in name else create_model(name, seed=1)).double()
    images = make_images(2, base.patch_embed.img_size[0], 7).double()
    params = horc.extract_params(base)
    assert params["headless"] and isinstance(base.head, nn.Identity)
    got, stats = horc.forward(params, images, {})
    torch.testing.assert_close(got, base(images), rtol=1e-10, atol=1e-10)
    assert stats["token_counts"] == [base.patch_embed.num_patches + 1] * len(base.blocks)


def test_reference_features_are_the_pooled_reference_head_input():
    """With pruning: the headless reference runs the same blocks as the pooled / pre-norm reference; a classifier with an
    identity head gives the same numbers."""
    for name in ("vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae"):
        base = _micro(name, num_classes=0).double()
        images = make_images(3, 64, 2).double()
        feats, stats = horc.forward(horc.extract_params(base), images, MICRO_SCHEDULE)
        assert stats["token_counts"] == [17, 17, 13, 8] and feats.shape == (3, 128)
        base.head = nn.Linear(128, 128).double()
        with torch.no_grad():
            base.head.weight.copy_(torch.eye(128))
            base.head.bias.zero_()
        params = horc.extract_params(base)
        assert not params["headless"]
        logits, _ = porc.forward(params, images, MICRO_SCHEDULE)
        torch.testing.assert_close(logits, feats, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------ wrapper construction (host side)
def test_wrapper_accepts_headless_models():
    w = RAJNIViTWrapper(_micro("vit_micro_patch16_64_dino"), MICRO_SCHEDULE)
    assert w.headless and not w.avg_pool and not w.pre_norm
    w = RAJNIViTWrapper(_micro("vit_micro_patch16_64_mae", num_classes=0), MICRO_SCHEDULE)
    assert w.headless and w.avg_pool
    w = RAJNIViTWrapper(_micro("vit_micro_patch16_64_clip", num_classes=0), MICRO_SCHEDULE)
    assert w.headless and w.pre_norm
    base = _micro("vit_micro_patch16_64")
    base.head = nn.Dropout(0.0)                                   # an identity too
    assert RAJNIViTWrapper(base, {}).headless
    for name in DINO[:4]:
        assert RAJNIViTWrapper(create_model(name, seed=None), README_SCHEDULE).headless
    assert not RAJNIViTWrapper(create_model("vit_micro_patch16_64"), {}).headless


def test_wrapper_rejections():
    base = create_model("deit_micro_distilled_patch16_64", num_classes=0)        # distilled, both heads Identity
    with pytest.raises(NotImplementedError, match="dist_token with head = Identity"):
        RAJNIViTWrapper(base, {})
    base = create_model("deit_micro_distilled_patch16_64")
    base.head = nn.Identity()                                                      # distilled, head Identity, head_dist Linear
    with pytest.raises(NotImplementedError, match="headless"):
        RAJNIViTWrapper(base, {})
    base = create_model("vit_micro_patch16_64_dino")
    base.head = nn.Sequential(nn.Linear(128, 64), nn.ReLU(), nn.Linear(64, 10))   # neither Linear nor Identity
    with pytest.raises(NotImplementedError, match="head = Sequential"):
        RAJNIViTWrapper(base, {})
    base.head = nn.Dropout(0.1)
    with pytest.raises(NotImplementedError, match="head = Dropout"):
        RAJNIViTWrapper(base, {})


# ------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("fmt", ["dict", "safetensors", "pt"])
@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip"])
def test_load_checkpoint_round_trip(tmp_path, fmt, name):
    src = _micro(name, num_classes=0)
    sd = src.state_dict()
    assert not any(k.startswith("head") for k in sd)
    if fmt == "dict":
        got = load_checkpoint({"model": sd})
    else:
        path = str(tmp_path / f"w.{fmt}")
        write_safetensors(path, sd) if fmt == "safetensors" else torch.save(sd, path)
        got = load_checkpoint(path)
    assert isinstance(got.head, nn.Identity) and got.num_classes == 0
    assert got.global_pool == src.global_pool and type(got.norm_pre) is type(src.norm_pre)
    assert list(got.state_dict()) == list(sd)
    for k, v in sd.items():
        assert torch.equal(got.state_dict()[k], v), k
    images = make_images(2, 64, 4)
    assert torch.equal(got(images), src(images))
    assert RAJNIViTWrapper(got, MICRO_SCHEDULE).headless


def test_load_checkpoint_rejections():
    vit = create_model("vit_micro_patch16_64").state_dict()
    headless = {k: v for k, v in vit.items() if not k.startswith("head.")}
    with pytest.raises(KeyError, match="'head.bias'"):
        load_checkpoint({**headless, "head.bias": vit["head.bias"]})
    dd = create_model("deit_micro_distilled_patch16_64").state_dict()
    with pytest.raises(NotImplementedError, match="dist_token"):                  # distilled without any head
        load_checkpoint({k: v for k, v in dd.items() if not k.startswith("head")})
    with pytest.raises(NotImplementedError, match="dist_token"):                  # head_dist but no head
        load_checkpoint({k: v for k, v in dd.items() if not k.startswith("head.")})
    with pytest.raises(NotImplementedError, match="head_dist"):                   # no dist_token, head_dist only
        load_checkpoint({**headless, "head_dist.weight": vit["head.weight"], "head_dist.bias": vit["head.bias"]})
    with pytest.raises(KeyError, match="not a timm-named"):
        load_checkpoint({"encoder.layer.0.weight": torch.ones(2)})
    for k in ("cls_token", "pos_embed", "patch_embed.proj.weight"):                 # the other required keys stay required
        with pytest.raises(KeyError, match=re.escape(repr(k))):
            load_checkpoint({q: v for q, v in headless.items() if q != k})


# ------------------------------------------------------------------ schedule tools and the CLI
def test_flops_per_image_without_a_head():
    counts = S.token_counts(README_SCHEDULE, 12, 197)
    with_head = S.flops_per_image(counts, 768, 3072, 196)
    assert with_head - S.flops_per_image(counts, 768, 3072, 196, classes=0) == 2.0 * 768 * 1000


def test_cosine_agreement_arithmetic():
    g = torch.Generator().manual_seed(0)
    dense = [torch.randn(4, 16, generator=g), torch.randn(3, 16, generator=g)]
    assert S.cosine_agreement(dense, dense) == pytest.approx(100.0, abs=1e-12)
    assert S.cosine_agreement([2.5 * d for d in dense], dense) == pytest.approx(100.0, abs=1e-12)     # scale-free
    assert S.cosine_agreement([-d for d in dense], dense) == pytest.approx(-100.0, abs=1e-12)
    got = [d + 0.5 * torch.randn(d.shape, generator=g) for d in dense]
    want = 100.0 * torch.cat([F.cosine_similarity(a.double(), b.double(), dim=1) for a, b in zip(got, dense)]).mean().item()
    assert S.cosine_agreement(got, dense) == pytest.approx(want, rel=1e-12)
    # a mean over images, not over batches
    one = F.cosine_similarity(got[1].double(), dense[1].double(), dim=1)
    assert S.cosine_agreement(got[1:], dense[1:]) == pytest.approx(100.0 * one.mean().item(), rel=1e-12)
    with pytest.raises(ValueError):
        S.cosine_agreement(got, dense[:1])


def test_run_refuses_a_headless_model(tmp_path):
    from rajni_vit_b200 import run
    sched = tmp_path / "s.json"
    sched.write_text(json.dumps({"1": {"keep_ratio": 0.5}}))
    with pytest.raises(ValueError, match="headless"):
        run.main(["--synthetic", "1", "--batch_size", "2", "--model", "vit_micro_patch16_64_dino", "--schedule", str(sched),
                  "--device", "cpu"])
    path = str(tmp_path / "dino.safetensors")
    write_safetensors(path, create_model("vit_micro_patch16_64_dino").state_dict())
    with pytest.raises(ValueError, match="headless"):
        run.main(["--synthetic", "1", "--batch_size", "2", "--ckpt", path, "--schedule", str(sched), "--device", "cpu"])
