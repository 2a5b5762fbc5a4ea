"""CPU-side tests of the 8- and 32-pixel patch models: schedules and work per image, checkpoint loading into a model the
wrapper accepts, the patch sizes it still refuses, and the library's long-sequence score query."""
import pytest
import torch

from rajni_vit_b200 import ops
from rajni_vit_b200 import schedule as S
from rajni_vit_b200.checkpoint import load_checkpoint
from rajni_vit_b200.vit import VIT_CONFIGS, VIT_PATCH, VisionTransformer, create_model
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper
from tests.cases import README_SCHEDULE


@pytest.mark.parametrize("name,tokens,pruned,dense_gflop,pruned_gflop", [
    ("vit_base_patch8_224", 785, [785, 785, 785, 785, 690, 607, 607, 607, 485, 349, 349, 349], 156.297, 110.041),
    ("vit_base_patch32_224", 50, [50, 50, 50, 50, 44, 38, 38, 38, 30, 21, 21, 21], 8.818, 6.360),
    ("vit_base_patch16_224", 197, [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87], 35.128, 25.332),
])
def test_token_counts_and_flops_of_the_patch_variants(name, tokens, pruned, dense_gflop, pruned_gflop):
    dim, depth, heads, img = VIT_CONFIGS[name]
    p = VIT_PATCH[name]
    assert (img // p) ** 2 + 1 == tokens
    assert S.token_counts(README_SCHEDULE, depth, tokens) == pruned
    fl = lambda counts: S.flops_per_image(counts, dim, 4 * dim, tokens - 1, patch_dim=3 * p * p) / 1e9   # noqa: E731
    assert abs(fl([tokens] * depth) - dense_gflop) < 5e-3
    assert abs(fl(pruned) - pruned_gflop) < 5e-3


def test_stand_ins_have_their_patch_size():
    for name, (dim, depth, heads, img) in VIT_CONFIGS.items():
        p = VIT_PATCH[name]
        assert f"patch{p}_" in name and img % p == 0
    m = create_model("vit_micro_patch8_72")
    assert m.patch_embed.proj.kernel_size == (8, 8) and m.pos_embed.shape[1] == 82
    m = create_model("vit_micro_patch32_128")
    assert m.patch_embed.proj.kernel_size == (32, 32) and m.pos_embed.shape[1] == 17


def test_patch16_stand_ins_are_unchanged():
    """The patch-16 names build the same parameters as before the patch size became a field (same RNG order)."""
    a = create_model("vit_micro_patch16_64", seed=0)
    torch.manual_seed(0)
    b = VisionTransformer(img_size=64, embed_dim=128, depth=4, num_heads=2)
    with torch.no_grad():
        for q in b.parameters():
            q.copy_(q.to(torch.bfloat16).to(torch.float32))
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb), ka


@pytest.mark.parametrize("name", ["vit_micro_patch32_128", "vit_micro_patch8_72"])
def test_load_checkpoint_of_other_patch_sizes_builds_an_accepted_model(name):
    sd = create_model(name, seed=5).state_dict()
    base = load_checkpoint(sd)
    p = VIT_PATCH[name]
    assert base.patch_embed.proj.kernel_size == (p, p) and base.patch_embed.img_size[0] == VIT_CONFIGS[name][3]
    for k, v in sd.items():
        assert torch.equal(base.state_dict()[k], v), k
    w = RAJNIViTWrapper(base, {1: {"keep_ratio": 0.5}})
    assert w.patch == p


@pytest.mark.parametrize("p", [14, 12, 4])
def test_wrapper_rejects_patch_sizes_that_are_not_multiples_of_8(p):
    base = VisionTransformer(img_size=p * 4, patch_size=p, embed_dim=128, depth=1, num_heads=2)
    with pytest.raises(NotImplementedError, match=f"kernel=\\({p}, {p}\\)"):
        RAJNIViTWrapper(base, {})


def test_score_workspace_query():
    """Host-side query of the long-sequence score path: the one-launch kernel holds 785 tokens at no head count of a ViT with
    head dim 64 (H = 6 / 12 / 16: 232 960 / 251 800 / 264 360 B of shared memory against 232 448 B), 723 at 12 heads."""
    for H in (6, 12, 16):
        assert ops.needs_score_workspace(785, H)
        assert ops.needs_score_workspace(4096, H)
        assert not ops.needs_score_workspace(577, H)
        assert not ops.needs_score_workspace(197, H)
    assert not ops.needs_score_workspace(723, 12) and ops.needs_score_workspace(724, 12)
