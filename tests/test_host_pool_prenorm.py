"""CPU-side tests of average-pooled heads (global_pool='avg' with fc_norm, MAE fine-tunes) and the pre-norm stem
(norm_pre, a bias-free patch embedding, LayerNorm eps 1e-5: CLIP fine-tunes): the reference (tests/pool_prenorm_oracle.py)
against the stand-ins' own forward and against the DeiT reference with neither feature, what the wrapper accepts and still
refuses, and checkpoint loading."""
import pytest
import torch
import torch.nn as nn

from tests import deit_oracle as dorc
from tests import pool_prenorm_oracle as porc
from rajni_vit_b200.checkpoint import load_checkpoint, write_safetensors
from rajni_vit_b200.vit import VIT_CONFIGS, VIT_PATCH, VIT_POOL_PRENORM, create_model, randomize_trained_like
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images

POOLED = ["vit_base_patch16_224_mae", "vit_large_patch16_224_mae", "vit_micro_patch16_64_mae"]
PRENORM = ["vit_base_patch16_clip_224", "vit_base_patch32_clip_224", "vit_base_patch16_clip_384", "vit_micro_patch16_64_clip"]


def _micro(name, seed=3):
    return randomize_trained_like(create_model(name, seed=seed), seed=seed + 1)


def test_stand_in_layouts():
    assert set(VIT_POOL_PRENORM) == set(POOLED) | set(PRENORM)
    for name in POOLED:
        m = create_model(name, seed=None)
        assert m.global_pool == "avg" and isinstance(m.fc_norm, nn.LayerNorm) and isinstance(m.norm, nn.Identity)
        assert isinstance(m.norm_pre, nn.Identity) and m.patch_embed.proj.bias is not None and m.fc_norm.eps == 1e-6
    for name in PRENORM:
        m = create_model(name, seed=None)
        assert m.global_pool == "token" and isinstance(m.norm, nn.LayerNorm) and isinstance(m.fc_norm, nn.Identity)
        assert isinstance(m.norm_pre, nn.LayerNorm) and m.patch_embed.proj.bias is None
        assert all(n.eps == 1e-5 for n in m.modules() if isinstance(n, nn.LayerNorm))
        assert m.patch_embed.proj.kernel_size == (VIT_PATCH[name],) * 2 and m.patch_embed.img_size[0] == VIT_CONFIGS[name][3]
    for name, cfg in VIT_CONFIGS.items():
        assert len(cfg) == 4, name                   # bench.py unpacks four fields


def test_trained_like_spreads_the_new_norms():
    for name, mod in (("vit_micro_patch16_64_mae", "fc_norm"), ("vit_micro_patch16_64_clip", "norm_pre")):
        ln = getattr(_micro(name), mod)
        assert ln.weight.min() >= 0.3 and ln.weight.std() > 0.3 and ln.bias.abs().max() > 0.1


@pytest.mark.parametrize("name", POOLED[2:] + PRENORM[3:] + ["vit_base_patch32_clip_224"])
def test_dense_reference_equals_the_stand_in_forward(name):
    """fp64: the reference's norm_pre, bias-free embedding and pooled head are timm's."""
    base = (_micro(name) if "micro" in name else create_model(name, seed=1)).double()
    images = make_images(2, base.patch_embed.img_size[0], 7).double()
    ref = base(images)
    got, stats = porc.forward(porc.extract_params(base), images, {})
    torch.testing.assert_close(got, ref, rtol=1e-10, atol=1e-10)
    assert stats["token_counts"] == [base.patch_embed.num_patches + 1] * len(base.blocks)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64", "deit_micro_distilled_patch16_64", "deit3_micro_patch16_64"])
def test_reference_without_the_features_is_the_deit_reference(name):
    base = _micro(name)
    params = porc.extract_params(base)
    assert params["norm_pre"] is None and not params["avg_pool"] and params["fc_norm"] is None
    images = make_images(3, 64, 5)
    trace, ref_trace = [], []
    got, stats = porc.forward(params, images, MICRO_SCHEDULE, trace=trace)
    ref, ref_stats = dorc.forward(dorc.extract_params(base), images, MICRO_SCHEDULE, trace=ref_trace)
    assert stats == ref_stats and torch.equal(got, ref)
    for rec, rrec in zip(trace, ref_trace):
        assert torch.equal(rec["x_out"], rrec["x_out"])


def test_pooled_reference_averages_the_kept_patch_tokens():
    base = _micro("vit_micro_patch16_64_mae").double()
    params = porc.extract_params(base)
    trace = []
    logits, stats = porc.forward(params, make_images(3, 64, 2).double(), MICRO_SCHEDULE, trace=trace)
    assert stats["token_counts"] == [17, 17, 13, 8]
    x = trace[-1]["x_out"]
    assert x.shape[1] == 1 + int(0.5 * 7)
    w, b, eps = params["fc_norm"]
    want = torch.nn.functional.linear(torch.nn.functional.layer_norm(x[:, 1:].mean(1), (128,), w, b, eps),
                                      params["head_w"], params["head_b"])
    assert torch.equal(logits, want)


# ------------------------------------------------------------------ wrapper construction (host side)
def test_wrapper_accepts_both_families():
    w = RAJNIViTWrapper(_micro("vit_micro_patch16_64_mae"), MICRO_SCHEDULE)
    assert w.avg_pool and not w.pre_norm and w.prefix == 1
    w = RAJNIViTWrapper(_micro("vit_micro_patch16_64_clip"), MICRO_SCHEDULE)
    assert w.pre_norm and not w.avg_pool
    for name in POOLED[:2] + PRENORM[:3]:
        RAJNIViTWrapper(create_model(name, seed=None), README_SCHEDULE if "large" not in name else {})
    w = RAJNIViTWrapper(create_model("vit_micro_patch16_64"), {})
    assert not w.avg_pool and not w.pre_norm


def _refused(base, match):
    with pytest.raises(NotImplementedError, match=match):
        RAJNIViTWrapper(base, {})


def test_wrapper_rejections():
    mae = "vit_micro_patch16_64_mae"
    base = create_model("deit_micro_distilled_patch16_64")       # avg pooling with a distillation token
    base.global_pool, base.fc_norm, base.norm = "avg", nn.LayerNorm(128), nn.Identity()
    _refused(base, "global_pool")
    base = create_model("vit_micro_patch16_64")                  # fc_norm with token pooling
    base.fc_norm, base.norm = nn.LayerNorm(128), nn.Identity()
    _refused(base, "fc_norm")
    base = create_model(mae)                                     # fc_norm together with norm
    base.norm = nn.LayerNorm(128)
    _refused(base, "fc_norm")
    base = create_model(mae)                                     # avg pooling without fc_norm (timm fc_norm=False)
    base.fc_norm, base.norm = nn.Identity(), nn.LayerNorm(128)
    _refused(base, "without fc_norm")
    base = create_model(mae)
    base.fc_norm = nn.LayerNorm(128, elementwise_affine=False)
    _refused(base, "fc_norm")
    for pool in ("avgmax", "max", "map"):
        base = create_model(mae)
        base.global_pool = pool
        _refused(base, f"global_pool='{pool}'")
    base = create_model("vit_micro_patch16_64_clip")
    base.norm_pre = nn.LayerNorm(64)
    _refused(base, "norm_pre")
    base = create_model(mae)                                     # register tokens
    base.reg_token, base.num_prefix_tokens = nn.Parameter(torch.zeros(1, 4, 128)), 5
    _refused(base, "register")
    base = create_model(mae)                                     # no class token (timm *_gap_*)
    base.cls_token = None
    _refused(base, "class token")

    class QuickGELU(nn.Module):                                  # OpenAI CLIP's activation
        def forward(self, x):
            return x * torch.sigmoid(1.702 * x)

    base = create_model("vit_micro_patch16_64_clip")
    base.blocks[1].mlp.act = QuickGELU()
    _refused(base, "QuickGELU")
    base = create_model("vit_micro_patch16_64_clip")             # patch 14
    base.patch_embed.proj = nn.Conv2d(3, 128, 14, 14, bias=False)
    _refused(base, r"kernel=\(14, 14\)")


# ------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("fmt", ["dict", "safetensors", "pt"])
@pytest.mark.parametrize("name", ["vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip", "vit_base_patch32_clip_224"])
def test_load_checkpoint_round_trip(tmp_path, fmt, name):
    src = _micro(name) if "micro" in name else create_model(name, seed=2)
    sd = src.state_dict()
    if "mae" in name:
        assert {"fc_norm.weight", "fc_norm.bias"} <= set(sd) and not any(k.startswith("norm.") for k in sd)
    else:
        assert {"norm_pre.weight", "norm_pre.bias"} <= set(sd) and "patch_embed.proj.bias" not in sd
    if fmt == "dict":
        got = load_checkpoint({"model": sd} if "mae" in name else sd)        # MAE releases nest the weights under "model"
    else:
        path = str(tmp_path / f"w.{fmt}")
        write_safetensors(path, sd) if fmt == "safetensors" else torch.save(sd, path)
        got = load_checkpoint(path)
    assert got.global_pool == src.global_pool and type(got.norm_pre) is type(src.norm_pre)
    assert got.patch_embed.img_size == src.patch_embed.img_size and got.patch_embed.patch_size == src.patch_embed.patch_size
    assert [n.eps for n in got.modules() if isinstance(n, nn.LayerNorm)] == \
           [n.eps for n in src.modules() if isinstance(n, nn.LayerNorm)]
    assert list(got.state_dict()) == list(sd)
    for k, v in sd.items():
        assert torch.equal(got.state_dict()[k], v), k
    if "micro" in name:
        images = make_images(1, 64, 4)
        assert torch.equal(got(images), src(images))
    w = RAJNIViTWrapper(got, README_SCHEDULE if len(got.blocks) == 12 else MICRO_SCHEDULE)
    assert w.avg_pool == ("mae" in name) and w.pre_norm == ("clip" in name)


def test_load_checkpoint_rejections():
    vit = create_model("vit_micro_patch16_64").state_dict()
    mae = _micro("vit_micro_patch16_64_mae").state_dict()
    clip = _micro("vit_micro_patch16_64_clip").state_dict()
    with pytest.raises(NotImplementedError, match="fc_norm"):                 # fc_norm next to norm
        load_checkpoint({**vit, "fc_norm.weight": torch.ones(128), "fc_norm.bias": torch.zeros(128)})
    with pytest.raises(NotImplementedError, match="fc_norm"):                 # fc_norm without its bias
        load_checkpoint({k: v for k, v in mae.items() if k != "fc_norm.bias"})
    with pytest.raises(NotImplementedError, match="norm_pre"):                # norm_pre without its bias
        load_checkpoint({k: v for k, v in clip.items() if k != "norm_pre.bias"})
    with pytest.raises(NotImplementedError, match="norm_pre"):                # norm_pre with more than an affine LayerNorm
        load_checkpoint({**clip, "norm_pre.running_mean": torch.zeros(128)})
    dd = _micro("deit_micro_distilled_patch16_64").state_dict()
    pooled_dist = {k: v for k, v in dd.items() if not k.startswith("norm.")}
    with pytest.raises(NotImplementedError, match="fc_norm"):                 # average pooling with a distillation token
        load_checkpoint({**pooled_dist, "fc_norm.weight": torch.ones(128), "fc_norm.bias": torch.zeros(128)})
    with pytest.raises(KeyError, match="norm"):                               # no final norm at all
        load_checkpoint({k: v for k, v in vit.items() if not k.startswith("norm.")})
