"""The oracle (oracle/rajni_oracle.py) against the golden vectors generated from the
unmodified reference (tests/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import rajni_oracle as orc
from rajni_vit_b200.vit import create_model
from tests.cases import (E2E_CASES, IMPORTANCE_CASES, SCHEDULES, SELECT_CASES, checksum,
                         make_images, make_qkv, make_scores, npz)
from tests.conftest import GOLDEN


def test_importance_kat():
    g = npz(os.path.join(GOLDEN, "importance_kat.npz"))
    s = orc.importance(torch.from_numpy(g["qkv"]), 2)
    np.testing.assert_allclose(s.numpy(), g["score"], rtol=1e-12)
    # SURVEY.md section 4.1 literal values
    np.testing.assert_allclose(s.numpy()[0], [0.15003425, 0.44155955, 0.04304628, 0.01046527], rtol=1e-6)


@pytest.mark.parametrize("name", list(IMPORTANCE_CASES))
def test_importance_golden(name):
    B, N, H, D, seed = IMPORTANCE_CASES[name]
    g = npz(os.path.join(GOLDEN, "importance_rand.npz"))
    qkv = make_qkv(B, N, H, D, seed)
    assert checksum(qkv) == pytest.approx(float(g[name + "_sum"]), rel=1e-12)
    np.testing.assert_allclose(orc.importance(qkv.double(), H).numpy(), g[name + "_f64"], rtol=1e-10)
    np.testing.assert_allclose(orc.importance(qkv, H).numpy(), g[name + "_f32"], rtol=2e-5)


@pytest.mark.parametrize("name", list(SELECT_CASES))
def test_select_golden(name):
    B, N, ratio, seed = SELECT_CASES[name]
    g = npz(os.path.join(GOLDEN, "select_cases.npz"))
    scores = make_scores(B, N, seed)
    assert checksum(scores) == pytest.approx(float(g[name + "_sum"]), rel=1e-12)
    idx = orc.select(scores, orc.keep_count(N, ratio))
    assert idx.dtype == torch.int64
    np.testing.assert_array_equal(idx.numpy(), g[name + "_idx"])
    assert (idx[:, 0] == 0).all() and (idx[:, 1:] > idx[:, :-1]).all()


def test_select_tie_rule_and_errors():
    s = torch.tensor([[9.0, 1.0, 2.0, 2.0, 2.0, 0.0, 2.0]])
    # greater first, then lower index: patches (1-based) 2 and 3
    assert orc.select(s, 2).tolist() == [[0, 2, 3]]
    assert bool(orc.tie_straddles_cut(s, 2)[0])
    assert not bool(orc.tie_straddles_cut(s, 4)[0])
    with pytest.raises(RuntimeError):
        orc.select(s, 7)
    assert orc.keep_count(121, 0.72) == 86 and orc.keep_count(101, 0.29) == 28 and orc.keep_count(5, 0.01) == 1


def test_trajectories_shape_only():
    g = json.load(open(os.path.join(GOLDEN, "trajectories.json")))
    for cfg, (model_name, sched) in SCHEDULES.items():
        n = {"deit_base_patch16_384": 577}.get(model_name, 197)
        depth = 24 if "large" in model_name else 12
        counts = []
        for i in range(depth):
            counts.append(n)
            if i in sched:
                n = orc.keep_count(n, sched[i]["keep_ratio"]) + 1
        assert counts == g[cfg], cfg
    assert g["C1_string_keys"] == [197] * 12
    assert g["C2"] == [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]


@pytest.mark.parametrize("name", list(E2E_CASES))
def test_forward_golden(name):
    model_name, sched, batch, seed = E2E_CASES[name]
    g = npz(os.path.join(GOLDEN, f"e2e_{name}.npz"))
    base = create_model(model_name, seed=0)
    assert checksum(torch.cat([p.detach().flatten() for p in base.parameters()])) == \
        pytest.approx(float(g["weight_sum"]), rel=1e-12)
    images = make_images(batch, base.patch_embed.img_size[0], seed)
    assert checksum(images) == pytest.approx(float(g["image_sum"]), rel=1e-12)
    trace = []
    logits, stats = orc.forward(orc.extract_params(base), images, sched, trace=trace)
    assert stats["token_counts"] == g["token_counts"].tolist()
    np.testing.assert_allclose(logits.numpy(), g["logits"], atol=2e-5, rtol=1e-4)
    for rec in trace:
        if rec["pruned"]:
            i = rec["block"]
            np.testing.assert_array_equal(rec["keep_idx"].numpy(), g[f"b{i}_keep_idx"])
            np.testing.assert_allclose(rec["next_scores"].numpy(), g[f"b{i}_next"], rtol=1e-4, atol=1e-9)


def test_string_keys_prune_nothing():
    base = create_model("vit_micro_patch16_64", seed=0)
    images = make_images(2, 64, 5)
    _, stats = orc.forward(orc.extract_params(base), images, {"1": {"keep_ratio": 0.5}})
    assert stats["token_counts"] == [17] * 4


# ------------------------------------------------------------------ loader: Resize(256, bicubic) + CenterCrop(224)  (run.py:62-66)
@pytest.mark.parametrize("h,w", [(375, 500), (500, 375), (256, 256), (224, 224), (300, 257), (257, 256), (333, 999), (480, 640), (227, 1500), (768, 1024)])
def test_resize_oracle_matches_torchvision(h, w):
    """oracle/resize_oracle.py restates Pillow's antialiased bicubic resampler and torchvision's size / crop rules; it must
    reproduce torchvision on PIL images bit for bit (this pins the oracle the CUDA kernel is checked against)."""
    np = pytest.importorskip("numpy")
    Image = pytest.importorskip("PIL.Image")
    T = pytest.importorskip("torchvision.transforms")
    from oracle.resize_oracle import crop_origin, resize_center_crop, resized_size
    rng = np.random.default_rng(h * 1000 + w)
    noise = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    smooth = (np.cumsum(noise.astype(np.int32), axis=1) // 7 % 256).astype(np.uint8)
    tf = T.Compose([T.Resize(256, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(224), T.PILToTensor()])
    for img in (noise, smooth):
        ref = tf(Image.fromarray(img)).numpy()
        assert np.array_equal(resize_center_crop(img), ref)
    nh, nw = resized_size(h, w)
    assert (nw, nh) == T.Resize(256)(Image.fromarray(noise)).size
    assert min(crop_origin(nh, nw)) >= 0
