"""Token-level features on the B200 (``forward_features`` / ``forward_intermediates``): every family against the stand-ins'
own ``forward_features`` with an empty schedule, pruned models against the reference (tests/features_oracle.py) with
selection teacher-forced, full-size DINO backbones, bit-exact cross-checks against ``forward`` and between the methods,
graph replay, uint8 input, batch independence and launch counts."""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests import features_oracle as forc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images
from tests.test_gpu_deit import MEAN, STD

pytestmark = pytest.mark.gpu

FAMILIES = ["vit_micro_patch16_64", "deit3_micro_patch16_64", "deit_micro_distilled_patch16_64", "vit_micro_patch16_64_mae",
            "vit_micro_patch16_64_clip", "vit_micro_patch16_64_dino", "vit_micro_patch8_72", "vit_micro_patch32_128"]


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def _base(name, **kw):
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    return randomize_trained_like(create_model(name, seed=0, **kw), seed=1)


def _close(got, ref, what=""):
    """Rows against the reference: max |d| under 0.1 times the reference's std, and every row's cosine similarity above
    0.999 (a row gathered from the wrong place or the wrong depth fails that by far).  The headless tests allow 0.05 std
    on a pooled [B, C] output; here the max runs over B·N0·C values, so its tail reaches further (measured on a B200 at
    1000 W: up to 0.059 std on the micro models, 0.080 on DINO ViT-B/16 at batch 64; row cosines >= 0.99995)."""
    got = got.float().cpu()
    assert got.shape == ref.shape and torch.isfinite(got).all()
    err, std = (got - ref).abs().max().item(), ref.std().item()
    cos = F.cosine_similarity(got.double().reshape(-1, got.shape[-1]), ref.double().reshape(-1, ref.shape[-1]), dim=1)
    print(f"{what}: max |d| {err:.4f} ({err / std:.4f} std), min row cosine {cos.min().item():.6f}")
    assert err < 0.1 * std and cos.min().item() > 0.999


def _keep(model):
    return [None if k is None else k.cpu().long() for k in model._last_keep_idx]


# ------------------------------------------------------------------ against the stand-ins and the reference
@pytest.mark.parametrize("name", FAMILIES)
def test_empty_schedule_matches_the_stand_in(pkg, name):
    base = _base(name)
    size = base.patch_embed.img_size[0]
    images = make_images(4, size, 11)
    model = pkg.RAJNIViTWrapper(copy.deepcopy(base), {}).cuda().eval()
    feats = model.forward_features(images.cuda())
    N0 = base.patch_embed.num_patches + base.num_prefix_tokens
    assert feats.dtype == torch.float32 and feats.shape == (4, N0, base.embed_dim)
    _close(feats, base.forward_features(images), name)
    depth = model.get_last_token_depth()
    assert depth.dtype == torch.int32 and depth.shape == (4, N0) and (depth == len(base.blocks)).all()


@pytest.mark.parametrize("name", FAMILIES[:6])
def test_pruned_teacher_forced(pkg, name):
    """With the GPU's own keep sets: the final features and the map after every block (with and without the final norm)
    against the reference, the depth map exact."""
    base = _base(name)
    images = make_images(4, 64, 12)
    params = forc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(copy.deepcopy(base), MICRO_SCHEDULE).cuda().eval()
    x = images.cuda()
    feats = model.forward_features(x)
    depth = model.get_last_token_depth().cpu()
    ours = _keep(model)
    ref, ref_depth, trace, stats = forc.forward_features(params, images, MICRO_SCHEDULE, forced_keep=ours)
    assert model.get_last_stats() == stats
    assert torch.equal(depth.long(), ref_depth)
    _close(feats, ref, f"{name} features")
    P0 = params["prefix"]
    for norm in (False, True):
        final, maps = model.forward_intermediates(x, norm=norm, output_fmt="NLC", return_prefix_tokens=True)
        assert all((a is None) == (b is None) and (a is None or torch.equal(a, b)) for a, b in zip(_keep(model), ours))
        assert torch.equal(final, feats) and len(maps) == len(base.blocks)
        for d, (patches, prefix) in enumerate(maps, start=1):
            want, _ = forc.token_map(trace, d)
            want = forc.final_norm(params, want) if norm else want
            assert prefix.shape[1] == P0
            _close(torch.cat([prefix, patches], 1), want, f"{name} block {d - 1} norm={norm}")


@pytest.mark.parametrize("name,batch", [("vit_base_patch16_224_dino", 64), ("vit_base_patch8_224_dino", 2)])
def test_full_size_vs_oracle(pkg, name, batch):
    """README schedule, teacher-forced.  ViT-B/8 has 785 tokens: its scores take the workspace path and its attention the
    long-sequence kernel."""
    from rajni_vit_b200 import schedule as S
    from rajni_vit_b200.vit import create_model
    base = create_model(name, seed=0)
    images = make_images(batch, 224, 1234)
    params = forc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, README_SCHEDULE).cuda().eval()
    feats = model.forward_features(images.cuda())
    depth = model.get_last_token_depth().cpu()
    ref, ref_depth, _, stats = forc.forward_features(params, images, README_SCHEDULE, forced_keep=_keep(model))
    N0 = feats.shape[1]
    assert model.get_last_stats() == stats and stats["token_counts"] == S.token_counts(README_SCHEDULE, 12, N0)
    assert torch.equal(depth.long(), ref_depth)
    _close(feats, ref, name)


# ------------------------------------------------------------------ bit-exact cross-checks
@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_clip", "vit_base_patch16_224_dino"])
def test_token_pooled_class_row_is_forward(pkg, name):
    """A token-pooled headless model: forward is norm(x)[:, 0] of the same rows with the same fp32 LayerNorm instance."""
    base = _base(name, num_classes=0)
    size = base.patch_embed.img_size[0]
    for sched in ({}, MICRO_SCHEDULE if "micro" in name else README_SCHEDULE):
        model = pkg.RAJNIViTWrapper(copy.deepcopy(base), sched).cuda().eval()
        x = make_images(8, size, 13).cuda()
        y = model(x)
        assert torch.equal(model.forward_features(x)[:, 0], y)
        assert torch.equal(model.forward_features(x.bfloat16())[:, 0], model(x.bfloat16()))


@pytest.mark.parametrize("name", ["vit_micro_patch16_64", "deit_micro_distilled_patch16_64", "vit_micro_patch16_64_mae",
                                  "vit_micro_patch16_64_dino"])
@pytest.mark.parametrize("graph", [False, True])
def test_methods_agree_and_leave_forward_alone(pkg, name, graph):
    """forward_intermediates(indices=[-1], norm=True) is forward_features split as timm splits it; forward's logits are
    the same before, between and after feature calls; eager equals graph replay; the outputs are the caller's."""
    base = _base(name)
    model = pkg.RAJNIViTWrapper(copy.deepcopy(base), MICRO_SCHEDULE).cuda().eval()
    model.use_cuda_graph = False
    x, x2 = make_images(4, 64, 14).cuda(), make_images(4, 64, 15).cuda()
    ref_logits, ref_feats = model(x).clone(), model.forward_features(x).clone()
    ref_depth = model.get_last_token_depth().clone()
    ref_maps = model.forward_intermediates(x, indices=[1, -1], norm=True, output_fmt="NCHW", intermediates_only=True)
    model.use_cuda_graph = graph
    P0, G = model.prefix, 4
    for _ in range(2):                                  # with graphs: capture, then replay
        assert torch.equal(model(x), ref_logits)
        feats = model.forward_features(x)
        assert torch.equal(feats, ref_feats) and torch.equal(model.get_last_token_depth(), ref_depth)
        assert torch.equal(model(x), ref_logits)
        final, maps = model.forward_intermediates(x, indices=[-1], norm=True, output_fmt="NLC", return_prefix_tokens=True)
        assert torch.equal(final, ref_feats) and len(maps) == 1
        assert torch.equal(maps[0][0], ref_feats[:, P0:]) and torch.equal(maps[0][1], ref_feats[:, :P0])
        grids = model.forward_intermediates(x, indices=[1, -1], norm=True, output_fmt="NCHW", intermediates_only=True)
        assert [g.shape for g in grids] == [(4, base.embed_dim, G, G)] * 2
        assert all(torch.equal(a, b) for a, b in zip(grids, ref_maps))
        assert torch.equal(grids[1].permute(0, 2, 3, 1).reshape(4, G * G, -1), ref_feats[:, P0:])
        assert torch.equal(model(x), ref_logits)
        other = model.forward_features(x2)              # another input through the same graph
        assert not torch.equal(other, feats)
        feats.fill_(0)                                  # a returned tensor is the caller's: the next call is unaffected
        assert torch.equal(model.forward_features(x), ref_feats)
    if graph:
        assert len(model._graphs) == 3                  # one per method


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae"])
def test_batch_independence_uint8_and_dtypes(pkg, name):
    model = pkg.RAJNIViTWrapper(_base(name), MICRO_SCHEDULE).cuda().eval()
    model.use_cuda_graph = False
    x = make_images(4, 64, 16).cuda()
    ref = model.forward_features(x).clone()
    depth = model.get_last_token_depth().clone()
    assert torch.equal(model.forward_features(x[2:3].contiguous()), ref[2:3])
    assert torch.equal(model.get_last_token_depth(), depth[2:3])
    both = model.forward_features(torch.cat([x, x[:2]]))
    assert torch.equal(both, torch.cat([ref, ref[:2]]))
    # bf16 input: bf16 rows, the fp32 rows rounded
    assert torch.equal(model.forward_features(x.bfloat16()).float(), model.forward_features(x.bfloat16().float()).bfloat16().float())
    g = torch.Generator().manual_seed(3)
    u8 = torch.randint(0, 256, (4, 3, 64, 64), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    want = model.forward_features(xf.cuda()).clone()
    model.set_input_normalization(MEAN, STD)
    got = model.forward_features(u8.cuda())
    assert got.dtype == torch.float32 and torch.equal(got, want)
    model.use_cuda_graph = True
    assert torch.equal(model.forward_features(u8.cuda()), want)
    model.train()
    model.m.blocks[0].mlp.drop1.p = 0.1
    with pytest.raises(NotImplementedError, match="training"):
        model.forward_features(x)


@pytest.mark.parametrize("name,num_classes,fwd,feat,norm_launch", [
    ("vit_base_patch16_224", None, 68, 68, 1),          # classification: final LN + head -> gather + LN
    ("vit_base_patch16_224_dino", None, 67, 68, 1),     # token-pooled headless: LN -> gather + LN
    ("vit_base_patch16_224_mae", 0, 67, 67, 0),         # Identity norm: the pooling kernel -> the gather only
])
def test_launches_per_step(pkg, name, num_classes, fwd, feat, norm_launch):
    """C2 (README schedule, 160 images: eager, each score/select one launch).  Each intermediate adds one gather, and one
    LayerNorm with norm=True where the model has a final LayerNorm."""
    from rajni_vit_b200 import _lib
    from rajni_vit_b200.vit import create_model
    model = pkg.RAJNIViTWrapper(create_model(name, seed=0, num_classes=num_classes), README_SCHEDULE).cuda().eval()
    model.use_cuda_graph = False
    x = make_images(160, 224, 1).cuda()

    def count(fn):
        fn()
        torch.cuda.synchronize()
        before = _lib.launch_count()
        fn()
        torch.cuda.synchronize()
        return _lib.launch_count() - before

    assert count(lambda: model(x)) == fwd
    assert "stages" not in next(iter(model._ws.values()))         # forward alone allocates no stage rows
    assert count(lambda: model.forward_features(x)) == feat
    assert count(lambda: model.forward_intermediates(x, indices=4)) == feat + 4
    assert count(lambda: model.forward_intermediates(x, indices=4, norm=True)) == feat + 4 * (1 + norm_launch)
    assert count(lambda: model.forward_intermediates(x, indices=[2, 5], intermediates_only=True)) == feat - 1 - norm_launch + 2
    assert count(lambda: model(x)) == fwd
