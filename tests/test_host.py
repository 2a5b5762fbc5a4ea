"""CPU-side tests (no GPU): host logic of the wrapper, the C-ABI library's exported surface, and the
data-parallel path of evaluate_model under a world_size-2 gloo group.

No compute entry point of librajni_b200.so is called here - there is no CPU path to call.
"""
import copy
import ctypes
import json
import os
import re
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from rajni_vit_b200 import _lib                                     # noqa: E402
from rajni_vit_b200.eval import evaluate_model, shard_bounds         # noqa: E402
from rajni_vit_b200.wrapper.attention import keep_count             # noqa: E402
from rajni_vit_b200.wrapper.model import RAJNIViTWrapper, _normalise_schedule   # noqa: E402
from rajni_vit_b200.vit import create_model                          # noqa: E402


# ------------------------------------------------------------------ host arithmetic
def test_keep_count_matches_python_double_truncation():
    """rajni/wrapper/attention.py:31-32: max(1, int(keep_ratio * (N - 1))) with Python doubles."""
    assert keep_count(121, 0.72) == 86          # 0.72 * 120 = 86.39999...
    assert keep_count(101, 0.29) == 28          # 0.29 * 100 = 28.999999999999996
    assert keep_count(101, 0.57) == 56
    assert keep_count(5, 0.01) == 1             # floor of one patch
    assert keep_count(197, 1.0) == 196


@pytest.mark.parametrize("model,sched,expect", [
    ("C2", {3: .88, 4: .88, 7: .8, 8: .72}, [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]),
    ("C3", {i: .7 for i in range(3, 12)}, [197, 197, 197, 197, 138, 96, 67, 47, 33, 23, 16, 11]),
    ("C5", {3: .88, 4: .88, 7: .8, 8: .72}, [577, 577, 577, 577, 507, 446, 446, 446, 357, 257, 257, 257]),
])
def test_token_count_trajectories(model, sched, expect):
    """SURVEY.md 4.2: token counts are shape-determined, so they can be checked without running a kernel."""
    n = expect[0]
    got = []
    for i in range(12):
        got.append(n)
        if i in sched:
            n = keep_count(n, sched[i]) + 1
    assert got == expect


def test_schedule_normalisation():
    s = _normalise_schedule({"3": {"keep_ratio": 0.5}, 4: {"keep_ratio": 0.9, "update": False}})
    assert s == {3: {"keep_ratio": 0.5}, 4: {"keep_ratio": 0.9, "update": False}}
    with pytest.raises(ValueError):
        _normalise_schedule({"x3": {"keep_ratio": 0.5}})
    with pytest.raises(KeyError):
        _normalise_schedule({3: {"update": True}})


def test_wrapper_construction_mirrors_reference():
    """model.py:7-25: blk.attn swapped on scheduled blocks, has_pruner flags, base model aliased as .m / .blocks."""
    base = create_model("vit_micro_patch16_64", seed=0)
    w = RAJNIViTWrapper(base, {1: {"keep_ratio": 0.75}, 3: {"keep_ratio": 0.5, "update": False}})
    assert w.m is base and w.blocks is base.blocks
    flags = [blk.has_pruner for blk in w.blocks]
    assert flags == [False, True, False, True]
    assert type(w.blocks[1].attn).__name__ == "RAJNIAttention"
    assert w.blocks[3].attn.update is False and w.blocks[3].attn.keep_ratio == 0.5
    assert w.blocks[1].attn.qkv is not None and w.get_last_stats() is None
    with pytest.raises(RuntimeError):
        w(torch.zeros(1, 3, 64, 64))            # CPU tensor: there is no CPU path


def test_shard_bounds_partition():
    for batch in (0, 1, 7, 8, 256, 257):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(batch, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == batch
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


# ------------------------------------------------------------------ the C-ABI library
def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "rajni_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rajni_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    """include/rajni_b200.h is the contract: every function it declares must be exported by the built library
    and bound (with a signature) by the ctypes loader."""
    names = _declared_symbols()
    assert len(names) >= 10
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in the header but not exported by {_lib.LIB_PATH}"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in rajni_vit_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == names


# One entry point per operation (ABI 11); ABI 12 dropped the GEMM's split-K workspace calls.  A name removed from this list
# must not come back with another signature: a caller that binds by name would misbind silently.
C_ABI = sorted("rajni_" + n for n in (
    "abi_version", "last_error", "device_check", "launch_count",
    "select_prefix", "score_select_prefix", "score_select_workspace_bytes", "score_select_needs_workspace",
    "gather_rows",
    "layernorm_strided", "layernorm_strided_f32", "layernorm_row_stats",
    "mean_pool_layernorm", "mean_pool_layernorm_f32",
    "gemm_bf16_ex", "gemm_row_stats_slots",
    "attention_fwd_ex",
    "patch_im2col_prefix",
    "resize_workspace_bytes", "resize_center_crop_u8", "resize_status"))


def test_c_abi_12_is_exactly_the_documented_surface():
    """The header declares exactly these 21 functions (so no superseded sibling is left), the ctypes loader binds exactly
    these, the library exports each, INTEGRATION.md documents each, and both sides report ABI 12."""
    assert len(C_ABI) == 21
    assert _declared_symbols() == C_ABI
    assert sorted(_lib.SIGNATURES) == C_ABI
    lib = ctypes.CDLL(_lib.LIB_PATH)
    integ = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for n in C_ABI:
        assert hasattr(lib, n), f"{n} is not exported by {_lib.LIB_PATH}"
        assert f"`{n}`" in integ, f"{n} is not documented in INTEGRATION.md"
    assert _lib.ABI_VERSION == 12
    assert _lib.load().rajni_abi_version() == 12


def test_library_abi_version_and_error_string():
    lib = _lib.load()
    assert lib.rajni_abi_version() == _lib.ABI_VERSION
    assert isinstance(lib.rajni_last_error(), bytes)
    assert lib.rajni_launch_count() >= 0


def test_library_is_not_linked_against_torch():
    """The boundary is a plain C ABI: no torch / python symbols are needed to load it."""
    import subprocess
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "torch" not in out and "python" not in out and "c10" not in out


# ------------------------------------------------------------------ data-parallel evaluate_model (gloo, world 2)
class _StubModel(torch.nn.Module):
    """Deterministic stand-in for the wrapper: logits depend only on the image, so every sharding of a
    batch must give the same predictions."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.randn(3 * 8 * 8, 10, generator=torch.Generator().manual_seed(3)))

    def forward(self, x):
        return x.flatten(1) @ self.w


def _make_data():
    g = torch.Generator().manual_seed(11)
    return [(torch.randn(7, 3, 8, 8, generator=g), torch.randint(0, 10, (7,), generator=g)) for _ in range(3)]


class _DecodeCounting(torch.utils.data.Dataset):
    """21 images in dataset form; counts how many this process "decoded"."""

    def __init__(self):
        self.batches, self.decoded = _make_data(), 0

    def __len__(self):
        return 21

    def __getitem__(self, i):
        self.decoded += 1
        x, y = self.batches[i // 7]
        return x[i % 7], y[i % 7]


def _dp_worker(rank, world, port, out_path):
    import torch.distributed as dist
    from rajni_vit_b200.data import sharded_loader
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        acc, ips = evaluate_model(_StubModel(), _make_data(), device="cpu", warmup=1, progress=False)
        ds = _DecodeCounting()
        acc2, _ = evaluate_model(_StubModel(), sharded_loader(ds, 7, rank, world), device="cpu", warmup=0, progress=False)
        decoded = torch.tensor([ds.decoded])
        dist.all_reduce(decoded)
        if rank == 0:
            json.dump({"acc": acc, "ips": ips, "acc_sharded_loader": acc2, "decoded_all_ranks": int(decoded)}, open(out_path, "w"))
    finally:
        dist.destroy_process_group()


def test_evaluate_model_data_parallel_gloo(tmp_path):
    """SURVEY.md 8(e): the batch is sharded contiguously by rank and the only collective is the final reduction of
    (correct, total, images) and MAX(time); a 2-rank run must report the single-process accuracy exactly."""
    acc1, _ = evaluate_model(_StubModel(), _make_data(), device="cpu", warmup=1, progress=False)
    out = str(tmp_path / "dp.json")
    for attempt in range(2):                     # (a free port can be taken between the probe and the rendezvous: one retry)
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        try:
            mp.spawn(_dp_worker, args=(2, port, out), nprocs=2, join=True)
            break
        except Exception:
            if attempt:
                raise
    got = json.load(open(out))
    assert got["acc"] == pytest.approx(acc1, abs=1e-9)
    assert got["ips"] > 0
    # the rank-sharded loader gives the same answer with every image decoded exactly once across the ranks
    assert got["acc_sharded_loader"] == pytest.approx(acc1, abs=1e-9)
    assert got["decoded_all_ranks"] == 21


def test_rank_sharded_batch_sampler_matches_slicing():
    """For every global batch the ranks' shards are exactly the slices evaluate_model would cut (same images, same order)."""
    from rajni_vit_b200.data import RankShardedBatchSampler
    from rajni_vit_b200.eval import shard_bounds
    for n, bs, world in ((21, 7, 2), (100, 32, 8), (10, 4, 3), (5, 8, 4), (64, 16, 1)):
        per_rank = [list(RankShardedBatchSampler(n, bs, r, world)) for r in range(world)]
        assert sorted(i for shards in per_rank for b in shards for i in b) == list(range(n))
        for start in range(0, n, bs):
            size = min(bs, n - start)
            for r in range(world):
                lo, hi = shard_bounds(size, r, world)
                want = list(range(start + lo, start + hi))
                if want:
                    assert want in per_rank[r]
        assert [len(RankShardedBatchSampler(n, bs, r, world)) for r in range(world)] == [len(p) for p in per_rank]


def test_cli_flags_match_reference():
    """Same flags and defaults as rajni/run.py:17-43 (plus --synthetic); a schedule is mandatory (run.py:115-116)."""
    from rajni_vit_b200 import run
    a = run.get_args(["--data_path", "/x", "--schedule", "s.json", "--compare_base", "--max_batches", "3"])
    assert (a.batch_size, a.num_workers, a.pin_mem, a.model, a.device, a.warmup) == (256, 8, True, "vit_base_patch16_224", "cuda", 5)
    assert a.compare_base and a.max_batches == 3 and a.schedule == "s.json" and not a.uint8_input
    with pytest.raises(SystemExit):
        run.get_args(["--schedule", "s.json"])                  # neither --data_path nor --synthetic


def test_standin_state_dict_uses_timm_names():
    """A timm checkpoint must load into the stand-in by name (SURVEY 8f item 2): same keys, same shapes."""
    from rajni_vit_b200.vit import create_model
    sd = create_model("vit_tiny_patch16_224", seed=0).state_dict()
    for k, shape in {"cls_token": (1, 1, 192), "pos_embed": (1, 197, 192), "patch_embed.proj.weight": (192, 3, 16, 16),
                     "blocks.0.norm1.weight": (192,), "blocks.0.attn.qkv.weight": (576, 192), "blocks.0.attn.qkv.bias": (576,),
                     "blocks.0.attn.proj.weight": (192, 192), "blocks.11.mlp.fc1.weight": (768, 192),
                     "blocks.11.mlp.fc2.bias": (192,), "norm.weight": (192,), "head.weight": (1000, 192)}.items():
        assert tuple(sd[k].shape) == shape, k


# ------------------------------------------------------------------ real-weights path (run.py:89-92,126-129)
def _ckpt_model():
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    return randomize_trained_like(create_model("vit_micro_patch16_64", seed=3), seed=4)


@pytest.mark.parametrize("fmt", ["pt", "safetensors"])
@pytest.mark.parametrize("family", ["timm", "wrapper", "dataparallel"])
def test_load_checkpoint_key_families(tmp_path, fmt, family):
    """timm keys, a saved wrapper's duplicated m.blocks.* / blocks.* families, and a module.-prefixed copy all load to
    the same model; the architecture is inferred from the shapes."""
    import rajni_vit_b200 as pkg
    from rajni_vit_b200.checkpoint import write_safetensors
    src = _ckpt_model()
    if family == "timm":
        sd = src.state_dict()
    elif family == "wrapper":
        sd = pkg.RAJNIViTWrapper(copy.deepcopy(src), {1: {"keep_ratio": 0.7}}).state_dict()
        assert any(k.startswith("m.blocks.") for k in sd) and any(k.startswith("blocks.") for k in sd)
    else:
        sd = {"state_dict": {"module." + k: v for k, v in src.state_dict().items()}}
    path = str(tmp_path / f"w.{fmt}")
    if fmt == "pt":
        torch.save(sd, path)
    else:
        write_safetensors(path, sd["state_dict"] if "state_dict" in sd else sd)
    got = pkg.load_checkpoint(path)
    assert (got.embed_dim, len(got.blocks), got.blocks[0].attn.num_heads, got.num_classes) == (128, 4, 2, 1000)
    assert got.patch_embed.img_size == (64, 64)
    for (k, a), (_, b) in zip(src.state_dict().items(), got.state_dict().items()):
        assert torch.equal(a, b), k
    # loading into an existing wrapper updates its base model in place
    wrap = pkg.RAJNIViTWrapper(_ckpt_model(), {1: {"keep_ratio": 0.7}})
    with torch.no_grad():
        wrap.m.head.weight.zero_()
    pkg.load_checkpoint(path, model=wrap)
    assert torch.equal(wrap.m.head.weight, src.head.weight)


def test_load_checkpoint_rejects_what_the_wrapper_cannot_run(tmp_path):
    import rajni_vit_b200 as pkg
    sd = _ckpt_model().state_dict()
    with pytest.raises(NotImplementedError, match="ls1"):
        pkg.load_checkpoint({**sd, "blocks.0.ls1.gamma": torch.ones(128)})
    with pytest.raises(KeyError):
        pkg.load_checkpoint({k: v for k, v in sd.items() if k != "blocks.2.mlp.fc1.weight"})
    with pytest.raises(KeyError, match="unexpected"):
        pkg.load_checkpoint({**sd, "blocks.0.attn.extra": torch.ones(1)})
    clash = {**sd, "m.head.bias": sd["head.bias"] + 1}
    with pytest.raises(ValueError, match="two different tensors"):
        pkg.load_checkpoint(clash)
    with pytest.raises(KeyError, match="not a timm-named"):
        pkg.load_checkpoint({"encoder.layer.0.weight": torch.ones(2)})


# ------------------------------------------------------------------ f4: schedule search (host logic)
def test_schedule_token_counts_and_flops_match_the_bench_constants():
    from rajni_vit_b200 import schedule as S
    readme = {3: {"keep_ratio": .88}, 4: {"keep_ratio": .88}, 7: {"keep_ratio": .8}, 8: {"keep_ratio": .72}}
    counts = S.token_counts(readme, 12, 197)
    assert counts == [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]
    assert S.token_counts({}, 12, 197) == [197] * 12
    assert S.token_counts({0: {"keep_ratio": 0.001}}, 2, 50) == [50, 2]          # one patch + CLS survive
    # 25.332 GFLOP/image: the figure bench.py and DESIGN.md quote for C2 (SURVEY 8d formula)
    assert abs(S.flops_per_image(counts, 768, 3072, 196) / 1e9 - 25.332) < 5e-3
    assert S.flops_per_image(counts, 768, 3072, 196) < S.flops_per_image([197] * 12, 768, 3072, 196)


def test_pareto_front_and_candidate_grid():
    from rajni_vit_b200 import schedule as S
    rs = [dict(name="a", img_s=10, accuracy=80.0), dict(name="b", img_s=20, accuracy=79.0), dict(name="c", img_s=15, accuracy=78.0),
          dict(name="d", img_s=30, accuracy=60.0), dict(name="e", img_s=30, accuracy=59.0), dict(name="f", img_s=5, accuracy=80.0)]
    assert [r["name"] for r in S.pareto_front(rs)] == ["d", "b", "a"]
    grid = S.candidate_grid(12)
    assert grid[0] == ("dense", {}) and grid[1][0] == "README"
    assert all(0 <= b < 12 and 0 < v["keep_ratio"] <= 1 for _, s in grid for b, v in s.items())
    assert any(v.get("update") is False for _, s in grid for v in s.values())       # score-carry candidates are in the family
    assert all(name != "README" for name, _ in S.candidate_grid(6))                 # needs blocks 7 and 8


def test_greedy_search_respects_the_floor_and_prefers_cheap_accuracy():
    """Synthetic evaluator: speed grows with the tokens removed (earlier blocks remove more work), accuracy falls by a
    per-block price.  The search must never return a schedule below the floor, must prune the cheap blocks first, and
    its history must be strictly faster at every step."""
    from rajni_vit_b200 import schedule as S
    depth, price = 6, {1: 8.0, 2: 0.5, 3: 0.4, 4: 6.0, 5: 0.2}

    def fake(sched):
        counts = S.token_counts(sched, depth, 101)
        work = sum(counts)
        loss = sum(price[b] * (1.0 - v["keep_ratio"]) * 10 for b, v in sched.items())
        return {"img_s": 1e6 / work, "accuracy": 90.0 - loss}

    sched, hist = S.greedy_search(fake, depth, floor=85.0, blocks=range(1, depth), ratios=(1.0, 0.9, 0.8, 0.7))
    assert hist[0]["schedule"] == {} and len(hist) > 3
    assert all(h["accuracy"] >= 85.0 for h in hist)
    assert all(b["img_s"] > a["img_s"] for a, b in zip(hist, hist[1:]))
    assert sched == hist[-1]["schedule"] and fake(sched)["accuracy"] >= 85.0
    # the expensive blocks (1 and 4) stay dense; block 5 buys no speed in this evaluator (nothing runs after it), so it stays too
    assert set(sched) == {2, 3} and sched[2]["keep_ratio"] == 0.7 and sched[3]["keep_ratio"] == 0.7
    # nothing admissible: the dense model comes back
    sched0, hist0 = S.greedy_search(fake, depth, floor=90.0, blocks=[1, 4])
    assert sched0 == {} and len(hist0) == 1

