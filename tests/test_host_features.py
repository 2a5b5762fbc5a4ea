"""CPU-side tests of token-level features (``forward_features`` / ``forward_intermediates``): the retained-token index maps
(``token_maps``) against a brute-force walk, their depth histogram against the schedule's token counts, ``indices``
validation, and the reference (tests/features_oracle.py) against the stand-ins' own ``forward_features``."""
import copy

import pytest
import torch

from rajni_vit_b200 import schedule as S
from rajni_vit_b200.vit import create_model, randomize_trained_like
from rajni_vit_b200.wrapper.attention import keep_count, token_maps
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper, feature_take_indices
from tests import features_oracle as forc
from tests import headless_oracle as horc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images


def _random_keeps(B, N0, prefix, ratios, seed):
    """A keep_log of random keep sets: each pruned block keeps its prefix rows first, then keep_count of the others in a
    random order (token_maps must not rely on any order)."""
    g = torch.Generator().manual_seed(seed)
    log, n = [], N0
    for r in ratios:
        if r is None:
            log.append(None)
            continue
        k = keep_count(n, r, prefix)
        rest = torch.stack([torch.randperm(n - prefix, generator=g)[:k] + prefix for _ in range(B)])
        log.append(torch.cat([torch.arange(prefix).expand(B, prefix), rest], 1).to(torch.int32))
        n = k + prefix
    return log


def _brute_force(log, B, N0):
    """Walk every token through the stages one at a time."""
    rows = torch.zeros(B, N0, dtype=torch.int32)
    depth = torch.zeros(B, N0, dtype=torch.int32)
    stages, ends = [[list(range(N0)) for _ in range(B)]], []
    for i, k in enumerate(log):
        if k is not None:
            ends.append(i)
            stages.append([[stages[-1][b][j] for j in k[b].tolist()] for b in range(B)])
    ends.append(len(log))
    base = 0
    for s, st in enumerate(stages):
        n = len(st[0])
        for b in range(B):
            for j, q in enumerate(st[b]):
                rows[b, q] = base + b * n + j
                depth[b, q] = ends[s]
        base += B * n
    return rows, depth


@pytest.mark.parametrize("prefix", [1, 2])
@pytest.mark.parametrize("seed", range(4))
def test_token_maps_against_brute_force(prefix, seed):
    g = torch.Generator().manual_seed(100 + seed)
    B, N0 = 3, 17 + int(torch.randint(0, 40, (1,), generator=g))
    ratios = [None if torch.rand(1, generator=g) < 0.4 else float(0.3 + 0.7 * torch.rand(1, generator=g)) for _ in range(8)]
    log = _random_keeps(B, N0, prefix, ratios, seed)
    for d in range(len(log) + 1):                         # every depth: the maps forward_intermediates gathers
        rows, depth = token_maps(log[:d], B, N0)
        want_rows, want_depth = _brute_force(log[:d], B, N0)
        assert rows.dtype == torch.int32 and depth.dtype == torch.int32
        assert torch.equal(rows, want_rows) and torch.equal(depth, want_depth), (d, ratios)
        assert (depth[:, :prefix] == d).all()            # prefix tokens go through every block


def test_token_maps_rows_are_distinct_and_inside_the_allocation():
    B, N0 = 4, 197
    log = _random_keeps(B, N0, 1, [README_SCHEDULE[i]["keep_ratio"] if i in README_SCHEDULE else None for i in range(12)], 5)
    rows, _ = token_maps(log, B, N0)
    total = B * sum(S.token_counts(README_SCHEDULE, 12, N0)[i] for i in [0, 4, 5, 8, 9])      # 197 + 173 + 152 + 121 + 87
    assert total == B * 730
    assert len(set(rows.flatten().tolist())) == B * N0 and 0 <= rows.min() and rows.max() < total


def test_depth_histogram_is_the_schedules_token_count_differences():
    """C2 (README schedule, 197 tokens): 24 / 21 / 31 / 34 / 87 tokens per image at depth 3 / 4 / 7 / 8 / 12."""
    B, N0 = 5, 197
    sched = README_SCHEDULE
    log = _random_keeps(B, N0, 1, [sched[i]["keep_ratio"] if i in sched else None for i in range(12)], 9)
    _, depth = token_maps(log, B, N0)
    counts = S.token_counts(sched, 12, N0)                # tokens entering each block; block 11 is dense
    counts = counts + [counts[-1]]
    want = {k: counts[k] - counts[k + 1] for k in sched}
    want[12] = counts[12]
    assert want == {3: 24, 4: 21, 7: 31, 8: 34, 12: 87}
    for b in range(B):
        got = {int(d): int(c) for d, c in zip(*torch.unique(depth[b], return_counts=True))}
        assert got == want


def test_feature_take_indices():
    assert feature_take_indices(12) == tuple(range(12))
    assert feature_take_indices(12, 4) == (8, 9, 10, 11)
    assert feature_take_indices(12, 12) == tuple(range(12))
    assert feature_take_indices(12, [11, -12, 3, 3, -1]) == (0, 3, 11)        # block order, each once (timm returns them so)
    assert feature_take_indices(4, (-1,)) == (3,)
    for bad in (0, 13, -1):
        with pytest.raises(ValueError, match="last-n"):
            feature_take_indices(12, bad)
    for bad in ([12], [-13], [0, 5, 40]):
        with pytest.raises(ValueError, match="out of range"):
            feature_take_indices(12, bad)
    with pytest.raises(ValueError, match="empty"):
        feature_take_indices(12, [])


def test_wrapper_refuses_bad_arguments_before_running():
    w = RAJNIViTWrapper(create_model("vit_micro_patch16_64_dino"), MICRO_SCHEDULE)
    x = make_images(2, 64, 0)
    with pytest.raises(ValueError, match="output_fmt"):
        w.forward_intermediates(x, output_fmt="NHWC")
    with pytest.raises(ValueError, match="out of range"):
        w.forward_intermediates(x, indices=[4])
    with pytest.raises(ValueError, match="last-n"):
        w.forward_intermediates(x, indices=5)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        w.forward_features(x)
    assert w.get_last_token_depth() is None


# ------------------------------------------------------------------ the reference
@pytest.mark.parametrize("name", ["vit_micro_patch16_64", "deit3_micro_patch16_64", "deit_micro_distilled_patch16_64",
                                  "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip", "vit_micro_patch16_64_dino",
                                  "vit_micro_patch8_72", "vit_micro_patch32_128"])
def test_reference_equals_the_stand_in_forward_features(name):
    """fp64, empty schedule: every row is the stand-in's own forward_features, at depth = number of blocks."""
    base = randomize_trained_like(create_model(name, seed=2), seed=3).double()
    images = make_images(2, base.patch_embed.img_size[0], 4).double()
    feats, depth, trace, stats = forc.forward_features(forc.extract_params(copy.deepcopy(base)), images, {})
    torch.testing.assert_close(feats, base.forward_features(images), rtol=1e-10, atol=1e-10)
    assert (depth == len(base.blocks)).all()
    for d in range(1, len(base.blocks) + 1):            # the map after block d-1 is the blocks' own output there
        x, _ = forc.token_map(trace, d)
        assert torch.equal(x, trace[d - 1]["x_out"])


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "deit_micro_distilled_patch16_64", "vit_micro_patch16_64_mae"])
def test_reference_with_pruning(name):
    """The kept tokens' rows are the last block's output, the class row is the headless reference's output, and each pruned
    token's row is the input row of the block that dropped it."""
    base = randomize_trained_like(create_model(name, seed=2), seed=3).double()
    images = make_images(3, 64, 5).double()
    params = forc.extract_params(copy.deepcopy(base))
    feats, depth, trace, stats = forc.forward_features(params, images, MICRO_SCHEDULE)
    P0, counts = params["prefix"], stats["token_counts"]
    counts = counts + [trace[-1]["keep_idx"].shape[1]]                  # tokens entering each block, then leaving the last
    assert counts == ([17, 17, 13, 8, 4] if P0 == 1 else [18, 18, 14, 9, 5])
    x, _ = forc.token_map(trace, len(trace))
    want = {k: counts[k] - counts[k + 1] for k in (1, 2, 3)}
    want[4] = counts[4]
    for b in range(3):
        assert {int(d): int(c) for d, c in zip(*torch.unique(depth[b], return_counts=True))} == want
    assert (depth[:, :P0] == 4).all() and torch.equal(x[:, :P0], trace[-1]["x_out"][:, :P0])
    if "mae" in name:
        assert torch.equal(feats, x)                                     # Identity norm
    elif P0 == 1:
        ref, _ = horc.forward(params, images, MICRO_SCHEDULE)
        torch.testing.assert_close(feats[:, 0], ref, rtol=1e-12, atol=1e-12)
    # a token dropped by block 2 carries its row of block 2's input
    rec = trace[2]
    pos1 = torch.gather(torch.arange(counts[0]).expand(3, -1), 1, trace[1]["keep_idx"])     # original positions, stage 1
    for b in range(3):
        kept = set(rec["keep_idx"][b].tolist())
        for j in range(rec["x_in"].shape[1]):
            if j not in kept:
                q = int(pos1[b, j])
                assert depth[b, q] == 2 and torch.equal(x[b, q], rec["x_in"][b, j])
