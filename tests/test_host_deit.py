"""CPU-side tests of the two DeiT families (DeiT-III: LayerScale and a class token without a position; distilled DeiT: a
distillation token kept through pruning and two heads): the DeiT reference (tests/deit_oracle.py) against the stand-ins'
own forward and against the oracle at one prefix token, prefix-aware
token counts, checkpoint loading and what is still refused, and the library's new entry points."""
import copy
import os
import re

import numpy as np
import pytest
import torch

from oracle import rajni_oracle as orc
from tests import deit_oracle as dorc
from rajni_vit_b200 import _lib
from rajni_vit_b200 import schedule as S
from rajni_vit_b200.checkpoint import load_checkpoint, write_safetensors
from rajni_vit_b200.packing import PackCache
from rajni_vit_b200.vit import (VIT_CONFIGS, VIT_VARIANT, LayerScale, VisionTransformer, create_model,
                                randomize_trained_like, spread_layer_scale)
from rajni_vit_b200.wrapper.attention import keep_count
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper
from tests.cases import E2E_CASES, MICRO_SCHEDULE, README_SCHEDULE, make_images, npz
from tests.conftest import GOLDEN, ROOT

DEIT3 = ["deit3_small_patch16_224", "deit3_medium_patch16_224", "deit3_base_patch16_224", "deit3_large_patch16_224",
         "deit3_base_patch16_384", "deit3_micro_patch16_64"]
DISTILLED = ["deit_tiny_distilled_patch16_224", "deit_small_distilled_patch16_224", "deit_base_distilled_patch16_224",
             "deit_base_distilled_patch16_384", "deit_micro_distilled_patch16_64"]


def _micro(name, seed=3):
    return randomize_trained_like(create_model(name, seed=seed), seed=seed + 1)


# ------------------------------------------------------------------ stand-ins and the DeiT reference
def test_stand_in_shapes():
    for name in DEIT3:
        m = create_model(name, seed=None)
        dim, depth, heads, img = VIT_CONFIGS[name]
        P = (img // 16) ** 2
        assert m.no_embed_class and m.num_prefix_tokens == 1 and m.pos_embed.shape[1] == P
        assert all(isinstance(b.ls1, LayerScale) and b.ls1.gamma.shape == (dim,) for b in m.blocks)
        g = torch.cat([torch.cat([b.ls1.gamma, b.ls2.gamma]) for b in m.blocks])
        assert g.min() >= 1e-6 * 0.99 and g.max() <= 1.0 and g.min() < 1e-5 and g.max() > 0.1      # spread, not constant
    for name in DISTILLED:
        m = create_model(name, seed=None)
        P = (VIT_CONFIGS[name][3] // 16) ** 2
        assert m.num_prefix_tokens == 2 and m.pos_embed.shape[1] == P + 2 and m.dist_token.shape == (1, 1, m.embed_dim)
        assert m.head_dist.weight.shape == m.head.weight.shape and not m.no_embed_class
    assert set(VIT_VARIANT) == set(DEIT3) | set(DISTILLED)
    for name, cfg in VIT_CONFIGS.items():
        assert len(cfg) == 4, name                   # bench.py unpacks four fields


def test_spread_layer_scale_is_log_uniform_and_leaves_the_rest_alone():
    a = create_model("deit3_micro_patch16_64", seed=0)
    b = copy.deepcopy(a)
    spread_layer_scale(b, seed=5)
    for (k, va), (_, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(va, vb) == (not k.endswith(".gamma")), k
    g = torch.cat([p.flatten() for k, p in b.named_parameters() if k.endswith(".gamma")]).log10()
    assert -6.01 <= g.min() and g.max() <= 0 and abs(g.mean().item() + 3) < 0.3     # 1024 draws of U(-6, 0)


@pytest.mark.parametrize("name", ["deit3_micro_patch16_64", "deit_micro_distilled_patch16_64",
                                  "deit3_small_patch16_224", "deit_tiny_distilled_patch16_224"])
def test_dense_oracle_equals_the_stand_in_forward(name):
    """fp64: the oracle's embedding (no_embed_class / distillation token), LayerScale and two-head average are timm's."""
    base = _micro(name) if "micro" in name else create_model(name, seed=1)
    base = base.double()
    images = make_images(2, base.patch_embed.img_size[0], 7).double()
    ref = base(images)
    got, stats = dorc.forward(dorc.extract_params(base), images, {})
    torch.testing.assert_close(got, ref, rtol=1e-10, atol=1e-10)
    P = base.patch_embed.num_patches
    assert stats["token_counts"] == [P + base.num_prefix_tokens] * len(base.blocks)


def test_deit_reference_with_one_prefix_token_is_the_oracle():
    """With one prefix token, no LayerScale and class-token positions the DeiT reference computes what the oracle computes:
    the same bits on the golden cases (and so the golden vectors the oracle is pinned to)."""
    for name, (model_name, sched, batch, seed) in E2E_CASES.items():
        g = npz(os.path.join(GOLDEN, f"e2e_{name}.npz"))
        base = create_model(model_name, seed=0)
        params = dorc.extract_params(base)
        assert params["prefix"] == 1 and not params["no_embed_class"] and "head_dist_w" not in params
        assert all(b["ls1"] is None and b["ls2"] is None for b in params["blocks"])
        images = make_images(batch, base.patch_embed.img_size[0], seed)
        trace, ref_trace = [], []
        logits, stats = dorc.forward(params, images, sched, trace=trace)
        ref, ref_stats = orc.forward(orc.extract_params(base), images, sched, trace=ref_trace)
        assert stats == ref_stats and torch.equal(logits, ref)
        assert stats["token_counts"] == g["token_counts"].tolist()
        np.testing.assert_allclose(logits.numpy(), g["logits"], atol=2e-5, rtol=1e-4)
        for rec, rrec in zip(trace, ref_trace):
            assert torch.equal(rec["x_out"], rrec["x_out"])
            if rec["pruned"]:
                assert torch.equal(rec["keep_idx"], rrec["keep_idx"]) and torch.equal(rec["next_scores"], rrec["next_scores"])
                np.testing.assert_array_equal(rec["keep_idx"].numpy(), g[f"b{rec['block']}_keep_idx"])
    s = torch.rand(3, 40, generator=torch.Generator().manual_seed(1))
    assert torch.equal(dorc.select(s, 20, prefix=1), orc.select(s, 20))
    assert torch.equal(dorc.tie_straddles_cut(s, 20), orc.tie_straddles_cut(s, 20))
    assert all(dorc.keep_count(n, r) == orc.keep_count(n, r) for n in (5, 121, 197, 577) for r in (0.01, 0.72, 0.88, 1.0))


def test_prefix_selection_rule():
    s = torch.tensor([[0.0, -5.0, 1.0, 2.0, 2.0, 2.0, 0.5, 2.0]])
    # tokens 0 and 1 always kept, whatever their scores; then the greatest, ties to the lower index
    assert dorc.select(s, 2, prefix=2).tolist() == [[0, 1, 3, 4]]
    assert dorc.select(s, 6, prefix=2).tolist() == [[0, 1, 2, 3, 4, 5, 6, 7]]
    assert bool(dorc.tie_straddles_cut(s, 2, prefix=2)[0]) and not bool(dorc.tie_straddles_cut(s, 5, prefix=2)[0])
    with pytest.raises(RuntimeError, match="out of range"):
        dorc.select(s, 7, prefix=2)
    # keep = max(1, int(r * (N - prefix))): Python double multiply and truncation, as for one prefix token
    assert dorc.keep_count(198, 0.88, 2) == keep_count(198, 0.88, 2) == int(0.88 * 196) == 172
    assert keep_count(122, 0.72, 2) == 86 and keep_count(5, 0.01, 2) == 1 and keep_count(197, 0.88) == keep_count(197, 0.88, 1)


@pytest.mark.parametrize("name,tokens,expect", [
    ("deit_base_distilled_patch16_224", 198, [198, 198, 198, 198, 174, 153, 153, 153, 122, 88, 88, 88]),
    ("deit3_base_patch16_224", 197, [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]),
    ("deit_base_distilled_patch16_384", 578, None),
    ("deit3_base_patch16_384", 577, None),
])
def test_token_count_trajectories(name, tokens, expect):
    prefix = 2 if "distilled" in name else 1
    img = VIT_CONFIGS[name][3]
    assert (img // 16) ** 2 + prefix == tokens
    counts = S.token_counts(README_SCHEDULE, 12, tokens, prefix=prefix)
    n, ref = tokens, []
    for i in range(12):
        ref.append(n)
        if i in README_SCHEDULE:
            n = dorc.keep_count(n, README_SCHEDULE[i]["keep_ratio"], prefix) + prefix
    assert counts == ref
    if expect is not None:
        assert counts == expect
    if prefix == 1:
        assert counts == S.token_counts(README_SCHEDULE, 12, tokens)


def test_oracle_pruned_forward_keeps_both_prefix_tokens():
    base = _micro("deit_micro_distilled_patch16_64").double()
    trace = []
    _, stats = dorc.forward(dorc.extract_params(base), make_images(3, 64, 2).double(), MICRO_SCHEDULE, trace=trace)
    assert stats["token_counts"] == [18, 18, 14, 9]                 # 16 patches + 2; keep int(.75*16), int(.6*12), int(.5*7)
    for rec in trace:
        if rec["pruned"]:
            k = rec["keep_idx"]
            assert (k[:, :2] == torch.tensor([0, 1])).all() and (k[:, 1:] > k[:, :-1]).all()
            assert torch.equal(rec["next_scores"], torch.gather(rec["scores"], 1, k))


# ------------------------------------------------------------------ LayerScale fold
def test_layer_scale_pack_folds_gamma_into_weight_and_bias():
    base = _micro("deit3_micro_patch16_64")
    blk = base.blocks[1]
    w, b = PackCache().linear_ls(blk.mlp.fc2, blk.ls2)
    g = blk.ls2.gamma.detach()
    assert w.dtype == torch.bfloat16 and b.dtype == torch.float32
    assert torch.equal(w, (blk.mlp.fc2.weight.detach() * g[:, None]).to(torch.bfloat16))
    assert torch.equal(b, blk.mlp.fc2.bias.detach() * g)
    # one bf16 rounding of the product: relative error <= 2^-8 even where gamma is 1e-6
    exact = blk.mlp.fc2.weight.detach().double() * g.double()[:, None]
    nz = exact != 0
    assert ((w.double() - exact).abs()[nz] / exact.abs()[nz]).max() <= 2.0 ** -8


# ------------------------------------------------------------------ wrapper construction (host side)
def test_wrapper_accepts_both_families_and_sets_the_prefix():
    w = RAJNIViTWrapper(_micro("deit_micro_distilled_patch16_64"), MICRO_SCHEDULE)
    assert w.prefix == 2 and not w.no_embed_class
    assert all(blk.attn.num_prefix_tokens == 2 for blk in w.blocks if blk.has_pruner)
    w = RAJNIViTWrapper(_micro("deit3_micro_patch16_64"), MICRO_SCHEDULE)
    assert w.prefix == 1 and w.no_embed_class
    w = RAJNIViTWrapper(create_model("vit_micro_patch16_64"), MICRO_SCHEDULE)
    assert w.prefix == 1 and not w.no_embed_class


def test_wrapper_rejections():
    class NotLayerScale(torch.nn.Module):            # right parameter, wrong module
        def __init__(self):
            super().__init__()
            self.gamma = torch.nn.Parameter(torch.ones(128))

    class LayerScale(torch.nn.Module):               # the name alone is not enough: a second parameter
        def __init__(self):
            super().__init__()
            self.gamma = torch.nn.Parameter(torch.ones(128))
            self.beta = torch.nn.Parameter(torch.zeros(128))

    for bad in (torch.nn.Linear(128, 128), NotLayerScale(), LayerScale(), torch.nn.LayerNorm(128)):
        base = create_model("deit3_micro_patch16_64")
        base.blocks[2].ls2 = bad
        with pytest.raises(NotImplementedError, match="ls2"):
            RAJNIViTWrapper(base, {})
    base = create_model("deit3_micro_patch16_64")
    base.blocks[0].ls1.gamma = torch.nn.Parameter(torch.ones(64))          # wrong width
    with pytest.raises(NotImplementedError, match="ls1"):
        RAJNIViTWrapper(base, {})
    base = create_model("deit_micro_distilled_patch16_64")
    base.head_dist = None
    with pytest.raises(NotImplementedError, match="head_dist"):
        RAJNIViTWrapper(base, {})
    base = create_model("vit_micro_patch16_64")
    base.reg_token = torch.nn.Parameter(torch.zeros(1, 4, 128))
    base.num_prefix_tokens = 5
    with pytest.raises(NotImplementedError, match="register"):
        RAJNIViTWrapper(base, {})
    base = create_model("vit_micro_patch16_64")
    base.fc_norm = torch.nn.LayerNorm(128)
    with pytest.raises(NotImplementedError, match="fc_norm"):
        RAJNIViTWrapper(base, {})
    base = create_model("deit_micro_distilled_patch16_64")
    base.global_pool = "avg"
    with pytest.raises(NotImplementedError, match="global_pool"):
        RAJNIViTWrapper(base, {})


# ------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("fmt", ["dict", "safetensors", "pt"])
@pytest.mark.parametrize("name", ["deit3_micro_patch16_64", "deit_micro_distilled_patch16_64", "deit3_base_patch16_384"])
def test_load_checkpoint_round_trip(tmp_path, fmt, name):
    src = _micro(name) if "micro" in name else create_model(name, seed=2)
    sd = src.state_dict()
    if "deit3" in name:
        assert "blocks.0.ls1.gamma" in sd and sd["pos_embed"].shape[1] == src.patch_embed.num_patches
    else:
        assert {"dist_token", "head_dist.weight", "head_dist.bias"} <= set(sd)
    if fmt == "dict":
        got = load_checkpoint(sd)
    else:
        path = str(tmp_path / f"w.{fmt}")
        write_safetensors(path, sd) if fmt == "safetensors" else torch.save(sd, path)
        got = load_checkpoint(path)
    assert got.num_prefix_tokens == src.num_prefix_tokens and got.no_embed_class == src.no_embed_class
    assert got.patch_embed.img_size == src.patch_embed.img_size
    assert list(got.state_dict()) == list(sd)
    for k, v in sd.items():
        assert torch.equal(got.state_dict()[k], v), k
    images = make_images(1, src.patch_embed.img_size[0], 4)
    if "micro" in name:
        assert torch.equal(got(images), src(images))
    w = RAJNIViTWrapper(got, README_SCHEDULE if len(got.blocks) == 12 else MICRO_SCHEDULE)
    assert w.prefix == src.num_prefix_tokens


def test_load_checkpoint_rejections():
    d3 = _micro("deit3_micro_patch16_64").state_dict()
    with pytest.raises(NotImplementedError, match="ls2"):                     # one gamma missing
        load_checkpoint({k: v for k, v in d3.items() if k != "blocks.3.ls2.gamma"})
    with pytest.raises(NotImplementedError, match="ls1"):
        load_checkpoint({k: v for k, v in d3.items() if not re.match(r"blocks\.[1-3]\.ls1\.", k)})
    with pytest.raises(NotImplementedError, match="ls1"):                     # LayerScale with more than a gamma
        load_checkpoint({**d3, "blocks.0.ls1.beta": torch.zeros(128)})
    vit = create_model("vit_micro_patch16_64").state_dict()
    with pytest.raises(NotImplementedError, match="ls1"):
        load_checkpoint({**vit, "blocks.0.ls1.gamma": torch.ones(128)})
    dd = _micro("deit_micro_distilled_patch16_64").state_dict()
    with pytest.raises(NotImplementedError, match="head"):                    # dist_token without head_dist
        load_checkpoint({k: v for k, v in dd.items() if not k.startswith("head_dist.")})
    with pytest.raises(NotImplementedError, match="dist"):                    # head_dist without dist_token
        load_checkpoint({k: v for k, v in dd.items() if k != "dist_token"})
    with pytest.raises(NotImplementedError, match="pos_embed"):               # 16 + 2 positions but no distillation token
        load_checkpoint({**vit, "pos_embed": dd["pos_embed"]})
    for extra in ("reg_token", "fc_norm.weight", "norm_pre.weight"):
        with pytest.raises(NotImplementedError, match=extra.split(".")[0]):
            load_checkpoint({**vit, extra: torch.zeros(1, 4, 128) if extra == "reg_token" else torch.ones(128)})


# ------------------------------------------------------------------ the C ABI
def test_new_entry_points_are_declared_and_exported():
    import ctypes
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rajni_b200.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(rajni_[a-z0-9_]+)\s*\(", text))
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in ("rajni_score_select_prefix", "rajni_select_prefix", "rajni_patch_im2col_prefix", "rajni_layernorm_strided"):
        assert n in declared and n in _lib.SIGNATURES and hasattr(lib, n), n
    assert _lib.load().rajni_abi_version() == 10
