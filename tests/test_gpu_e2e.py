"""Whole-path parity on the B200 through the reference-facing API.

Ladder (SURVEY.md 8c): teacher-forced per block against the reference's own dumps
(tests/golden/e2e_micro.npz, written by the unmodified reference), then end-to-end logits
tolerance, top-1 agreement and exact token_counts against the golden files and the oracle.

Tolerances: the path computes in bf16 with fp32 accumulation while the reference dumps are
fp32, so end-to-end logits are compared at atol 0.08 (logit std ~0.56; SURVEY 4.6 measured
0.065-0.089 between the reference's own fp32 and bf16 runs) and top-1 agreement >= 87.5 %.
"""
import copy
import json

import numpy as np
import pytest
import torch

from oracle import rajni_oracle as orc
from tests.cases import E2E_CASES, MICRO_SCHEDULE, README_SCHEDULE, C1_SCHEDULE, C3_SCHEDULE, C4_SCHEDULE, make_images, npz
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def build(pkg, name, sched, seed=0):
    from rajni_vit_b200.vit import create_model
    return pkg.RAJNIViTWrapper(create_model(name, seed=seed), sched).cuda().eval()


def test_compute_importance_api(pkg):
    g = npz(f"{GOLDEN}/importance_kat.npz")       # D=2 KAT is below the kernel's head dim; API check on D=64
    from tests.cases import make_qkv
    qkv = make_qkv(2, 50, 2, 64, 7)
    got = pkg.compute_importance(qkv.cuda(), 2)
    assert got.dtype == torch.float32 and got.shape == (2, 50)
    torch.testing.assert_close(got.cpu(), orc.importance(qkv, 2), rtol=3e-5, atol=1e-10)
    with pytest.raises(RuntimeError):
        pkg.compute_importance(qkv, 2)            # CPU tensor: no fallback
    assert g["score"].shape == (1, 4)


def test_teacher_forced_blocks_micro(pkg):
    """Feed each pruned block the reference's own block input and compare (out, keep_idx, next_scores)."""
    model_name, sched, batch, seed = E2E_CASES["micro"]
    g = npz(f"{GOLDEN}/e2e_micro.npz")
    model = build(pkg, model_name, sched)
    for i, blk in enumerate(model.blocks):
        if not blk.has_pruner:
            continue
        xn = torch.from_numpy(g[f"b{i}_xnorm"]).cuda()
        prev = torch.from_numpy(g[f"b{i}_prev"]).cuda() if f"b{i}_prev" in g else None
        out, keep_idx, nxt = blk.attn(xn, prev)
        assert keep_idx.dtype == torch.int64
        ref_idx = torch.from_numpy(g[f"b{i}_keep_idx"]).long()
        same = (keep_idx.cpu() == ref_idx).all(dim=1)
        print(f"block {i}: kept-index rows equal {int(same.sum())}/{len(same)}")
        assert same.all(), f"block {i} keep_idx differs"
        torch.testing.assert_close(nxt.cpu(), torch.from_numpy(g[f"b{i}_next"]), rtol=2e-2, atol=1e-6)
        ref_out = torch.from_numpy(g[f"b{i}_out"])
        err = (out.cpu() - ref_out).abs().max().item()
        print(f"block {i}: attention-out max abs err {err:.3e} (ref rms {ref_out.pow(2).mean().sqrt():.3e})")
        assert err < 0.02


@pytest.mark.parametrize("name", list(E2E_CASES))
def test_forward_vs_golden(pkg, name):
    model_name, sched, batch, seed = E2E_CASES[name]
    g = npz(f"{GOLDEN}/e2e_{name}.npz")
    model = build(pkg, model_name, sched)
    images = make_images(batch, model.m.patch_embed.img_size[0], seed)
    assert model.get_last_stats() is None
    logits = model(images.cuda())
    assert logits.dtype == torch.float32 and logits.shape == g["logits"].shape
    assert model.get_last_stats() == {"token_counts": g["token_counts"].tolist()}
    ref = torch.from_numpy(g["logits"])
    err = (logits.cpu() - ref).abs().max().item()
    agree = (logits.cpu().argmax(1) == ref.argmax(1)).float().mean().item()
    print(f"{name}: max |dlogit| {err:.4f}, top-1 agreement {agree:.3f}, logit std {ref.std():.3f}")
    assert err < 0.08
    assert agree >= 0.875
    # kept sets per pruned block vs the reference (overlap; exact equality is not expected end to end in bf16)
    for i, kidx in enumerate(model._last_keep_idx):
        if kidx is None:
            continue
        ref_idx = g[f"b{i}_keep_idx"]
        ov = np.mean([len(set(a.tolist()) & set(b.tolist())) / len(b) for a, b in zip(kidx.cpu().numpy(), ref_idx)])
        print(f"  block {i}: kept-set overlap with the reference {ov:.4f}")
        assert ov > 0.85
        k = kidx.cpu().long()
        assert (k[:, 0] == 0).all() and (k[:, 1:] > k[:, :-1]).all()


def test_forward_unpruned_matches_dense_oracle(pkg):
    """Empty schedule = the plain ViT; checks embed / dense blocks / head without any selection noise."""
    from rajni_vit_b200.vit import create_model
    base = create_model("vit_micro_patch16_64", seed=1)
    params = orc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, {}).cuda().eval()
    images = make_images(5, 64, 2)
    logits = model(images.cuda()).cpu()
    ref, stats = orc.forward(params, images, {})
    assert model.get_last_stats() == stats
    err = (logits - ref).abs().max().item()
    print(f"unpruned micro: max |dlogit| {err:.4f}")
    assert err < 0.05


def test_string_keys_are_normalised(pkg):
    """Documented deviation: json.load's string keys prune like int keys (the reference prunes nothing)."""
    sched = json.loads(json.dumps(MICRO_SCHEDULE))
    model = build(pkg, "vit_micro_patch16_64", sched)
    model(make_images(2, 64, 3).cuda())
    assert model.get_last_stats()["token_counts"] == [17, 17, 13, 8]


def test_bf16_model_and_input(pkg):
    model = build(pkg, "vit_micro_patch16_64", MICRO_SCHEDULE).bfloat16()
    x = make_images(3, 64, 4)
    y16 = model(x.cuda().bfloat16())
    assert y16.dtype == torch.bfloat16
    y32 = model(x.to(torch.bfloat16).float().cuda())
    torch.testing.assert_close(y16.float(), y32, rtol=2e-2, atol=2e-2)


def test_errors(pkg):
    from rajni_vit_b200.vit import create_model
    model = build(pkg, "vit_micro_patch16_64", {1: {"keep_ratio": 1.5}})
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        model(make_images(1, 64, 1).cuda())
    with pytest.raises(RuntimeError):
        model(make_images(1, 64, 1))             # CPU tensor
    base = create_model("vit_micro_patch16_64")
    base.blocks[0].ls1 = torch.nn.Linear(128, 128)
    with pytest.raises(NotImplementedError):
        pkg.RAJNIViTWrapper(base, {})


def near_tie_mismatch(ours: torch.Tensor, ref_scores: torch.Tensor, keep: int, rel_gap: float):
    """Compare a kept-index set with the oracle's own scores on the same block input.

    Returns (overlap fraction, worst relative distance to the cut of any token the two sides
    disagree on).  A disagreement is legitimate only if the token sits within ``rel_gap`` of the
    k-th score: bf16 activations perturb the scores by O(1e-2) relative, and random-init scores are
    nearly flat (SURVEY.md 4.5-4.7), so tokens that close to the cut can swap."""
    B = ours.shape[0]
    worst, overlap, in_band, cands = 0.0, 0.0, 0, 0
    for b in range(B):
        s = ref_scores[b, 1:].double()
        cut = torch.sort(s, descending=True).values[keep - 1].item()
        ref_set = set((torch.sort(s, descending=True, stable=True).indices[:keep] + 1).tolist())
        our_set = set(ours[b, 1:].tolist())
        overlap += len(ref_set & our_set) / keep
        for t in ref_set ^ our_set:
            worst = max(worst, abs(s[t - 1].item() - cut) / abs(cut))
        in_band += int(((s - cut).abs() <= rel_gap * abs(cut)).sum())
        cands += s.numel()
    near_tie_mismatch.band_fraction = in_band / max(cands, 1)      # how much of the candidate set the exemption covers
    return overlap / B, worst


@pytest.mark.parametrize("name,sched,batch,size", [("vit_base_patch16_224", README_SCHEDULE, 16, 224),
                                                   ("vit_small_patch16_224", C3_SCHEDULE, 16, 224),
                                                   ("vit_large_patch16_224", C4_SCHEDULE, 4, 224),
                                                   ("deit_base_patch16_384", README_SCHEDULE, 4, 384)])
def test_forward_vs_oracle_full_models(pkg, name, sched, batch, size):
    """BASELINE configs 2, 3, 4 (24 pruned blocks, C=1024) and 5 (577 tokens) at a batch the CPU oracle finishes in seconds.

    End-to-end drift on random-init weights is dominated by selection noise (the reference's own
    fp32-vs-bf16 runs diverge the same way, SURVEY.md 4.6), so the comparison is teacher-forced:
      1. arithmetic: the oracle is run with OUR kept indices forced at every pruned block; logits must
         agree within bf16 tolerance (max |dlogit| < 0.08 at logit std ~0.57; same top-1 wherever the oracle's
         top-2 margin exceeds twice that error);
      2. selection: at every pruned block the oracle's own fp32 scores on that same input must rank
         our kept tokens identically except for tokens within 3 % of the cut score;
      3. token_counts exact.  The free-running comparison is printed for the record."""
    from rajni_vit_b200.vit import create_model
    base = create_model(name, seed=0)
    params = orc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, sched).cuda().eval()
    images = make_images(batch, size, 1234)
    logits = model(images.cuda()).cpu()
    ours = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
    for k in ours:
        if k is not None:
            assert (k[:, 0] == 0).all() and (k[:, 1:] > k[:, :-1]).all()
    trace = []
    ref, stats = orc.forward(params, images, sched, trace=trace, forced_keep=ours)
    assert model.get_last_stats() == stats
    err = (logits - ref).abs().max().item()
    agree = (logits.argmax(1) == ref.argmax(1)).float().mean().item()
    print(f"{name} (selection teacher-forced): max |dlogit| {err:.4f}, top-1 agreement {agree:.3f}, logit std {ref.std():.3f}")
    # top-1 may only differ where the oracle's own top-2 margin is inside the logit error (random-init logits are nearly flat)
    top2 = ref.topk(2, dim=1).values
    decided = (top2[:, 0] - top2[:, 1]) > 2 * err
    assert err < 0.08 and bool((logits.argmax(1) == ref.argmax(1))[decided].all())
    for rec, kidx in zip(trace, ours):
        if kidx is None:
            continue
        keep = kidx.shape[1] - 1
        ov, worst = near_tie_mismatch(kidx, rec["scores"], keep, 0.03)
        print(f"  block {rec['block']}: kept-set overlap {ov:.4f}, worst disagreeing token is {worst:.2e} (relative) from the cut")
        assert worst < 0.03
        # the exemption must stay an exemption: few candidates sit in the band, and almost every kept token agrees
        # (measured on 256 images in bench.py's parity sample: 2.8 % of the candidates in the band, 0.28 % of the kept tokens differ)
        # (with fewer than 64 candidates per image one token is already > 1.5 % of them: only the overlap is bounded there)
        assert ov > 0.97 and (near_tie_mismatch.band_fraction < 0.12 or rec["scores"].shape[1] <= 64), (near_tie_mismatch.band_fraction, ov)
    free, _ = orc.forward(params, images, sched)
    print(f"{name} (free-running): max |dlogit| {(logits - free).abs().max().item():.4f}, "
          f"top-1 agreement {(logits.argmax(1) == free.argmax(1)).float().mean().item():.3f}")


def test_full_batch_properties(pkg):
    """BASELINE config 2 at its full batch (256): size-independent properties instead of the oracle:
    images are independent (a sub-batch reproduces its rows bit for bit) and the run is deterministic."""
    model = build(pkg, "vit_base_patch16_224", README_SCHEDULE)
    images = make_images(256, 224, 1234).cuda()
    y = model(images)
    assert model.get_last_stats()["token_counts"] == [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]
    assert torch.isfinite(y).all()
    y2 = model(images)
    assert torch.equal(y, y2)
    sub = model(images[64:96].contiguous())
    assert torch.equal(sub, y[64:96])


def test_evaluate_model(pkg):
    model = build(pkg, "vit_micro_patch16_64", MICRO_SCHEDULE)
    g = torch.Generator().manual_seed(0)
    data = [(make_images(8, 64, 100 + i), torch.randint(0, 1000, (8,), generator=g)) for i in range(3)]
    acc, ips = pkg.evaluate_model(model, data, device="cuda", max_batches=2, warmup=4, progress=False)
    assert 0.0 <= acc <= 100.0 and ips > 0
    acc2, _ = pkg.evaluate_model(model, data, device=torch.device("cuda"), warmup=1, progress=False)
    params = orc.extract_params(copy.deepcopy(model.m).cpu().float())
    ref_acc, _ = orc.evaluate(params, MICRO_SCHEDULE, data, warmup=0)
    print("acc", acc2, "oracle acc", ref_acc)


def test_evaluate_model_with_a_pinning_dataloader(pkg):
    """A real DataLoader with worker + pin-memory threads (what rajni/run.py:72-76 builds) around the small-batch path, whose
    first forward of each shape captures a CUDA graph: the capture must not mind the pin-memory thread's CUDA calls, and the
    ragged last batch (a new shape) must work."""
    from torch.utils.data import DataLoader, TensorDataset
    model = build(pkg, "vit_micro_patch16_64", MICRO_SCHEDULE)
    g = torch.Generator().manual_seed(3)
    images, labels = make_images(44, 64, 5), torch.randint(0, 1000, (44,), generator=g)
    loader = DataLoader(TensorDataset(images, labels), batch_size=8, shuffle=False, num_workers=2, pin_memory=True)
    acc, ips = pkg.evaluate_model(model, loader, device="cuda", warmup=2, progress=False)
    ref = build(pkg, "vit_micro_patch16_64", MICRO_SCHEDULE)
    ref.use_cuda_graph = False
    correct = sum(int((ref(images[i:i + 8].cuda()).argmax(dim=1).cpu() == labels[i:i + 8]).sum()) for i in range(0, 44, 8))
    assert ips > 0 and abs(acc - 100.0 * correct / 44) < 1e-9


def test_cli_synthetic(pkg, tmp_path, capsys):
    """python -m rajni_vit_b200.run with the reference's flags on synthetic batches: string-key schedule JSON prunes
    (normalised), --compare_base runs the un-pruned model on the same kernels."""
    import json
    from rajni_vit_b200 import run
    sched = tmp_path / "schedule.json"
    sched.write_text(json.dumps({"3": {"keep_ratio": 0.95, "update": False}, "4": {"keep_ratio": 0.95, "update": True},
                                 "5": {"keep_ratio": 0.85, "update": True}}))
    res = run.main(["--synthetic", "3", "--batch_size", "8", "--model", "vit_tiny_patch16_224", "--schedule", str(sched),
                    "--warmup", "1", "--compare_base"])
    out = capsys.readouterr().out
    assert "token_counts [197, 197, 197, 197, 187, 177" in out and "speed-up" in out
    assert res["base"][1] > 0 and res["rajni"][1] > 0


def test_uint8_input_matches_float_pipeline(pkg, tmp_path, capsys):
    """Extension: raw uint8 pixels, ToTensor + Normalize (run.py:62-70) applied inside the patch kernel.  The fp32 loader
    pipeline (u/255, -mean, /std in IEEE fp32) gives the same bf16 patches, so the logits must be bit-identical."""
    from rajni_vit_b200 import run
    model = build(pkg, "vit_tiny_patch16_224", C1_SCHEDULE)
    g = torch.Generator().manual_seed(5)
    u8 = torch.randint(0, 256, (8, 3, 224, 224), generator=g, dtype=torch.uint8)
    u8[0, :, :2] = torch.tensor([0, 255], dtype=torch.uint8)[None, :, None]           # the extremes are in
    mean, std = torch.tensor(run.IMAGENET_MEAN), torch.tensor(run.IMAGENET_STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    ref = model(xf.cuda()).clone()
    with pytest.raises(TypeError):
        model(u8.cuda())                                                              # no normalisation configured
    model.set_input_normalization(run.IMAGENET_MEAN, run.IMAGENET_STD)
    got = model(u8.cuda())
    assert got.dtype == torch.float32 and torch.equal(got, ref)
    assert torch.equal(model(xf.cuda()), ref)                                         # floats still take the float path
    # and through the CLI
    sched = tmp_path / "schedule.json"
    sched.write_text(json.dumps({"3": {"keep_ratio": 0.9}}))
    res = run.main(["--synthetic", "2", "--batch_size", "4", "--model", "vit_tiny_patch16_224", "--schedule", str(sched),
                    "--warmup", "1", "--uint8_input", "--compare_base"])
    assert res["rajni"][1] > 0 and "token_counts [197, 197, 197, 197, 177" in capsys.readouterr().out


def test_cuda_graph_mode_matches_eager(pkg):
    """Opt-in graph replay: bit-identical logits and the same stats as the eager launch sequence, across replays and
    after a shape change."""
    model = build(pkg, "vit_tiny_patch16_224", C1_SCHEDULE)
    x1, x2 = make_images(8, 224, 7).cuda(), make_images(8, 224, 8).cuda()
    assert model.use_cuda_graph is None                          # default: automatic (small batches replay a graph)
    model.use_cuda_graph = False
    ref1, ref2 = model(x1).clone(), model(x2).clone()
    stats = model.get_last_stats()
    model.use_cuda_graph = True
    for _ in range(2):
        assert torch.equal(model(x1), ref1) and torch.equal(model(x2), ref2)
        assert model.get_last_stats() == stats
    small = make_images(4, 224, 9).cuda()
    y = model(small)
    model.use_cuda_graph = False
    assert torch.equal(y, model(small))
    # automatic mode: graph at batch 8, eager at a batch too large for it (which replaces the workspace the graph was
    # captured with), graph again; and an in-place weight update must not be served from a stale graph
    model.use_cuda_graph = None
    big = make_images(96, 224, 10).cuda()                       # 96 * 197 rows > AUTO_GRAPH_MAX_ROWS
    assert torch.equal(model(x1), ref1) and len(model._graphs) == 1
    yb = model(big)
    assert len(model._graphs) == 0 and torch.equal(yb[:8], model(big[:8].contiguous()))
    assert torch.equal(model(x1), ref1) and torch.equal(model(x1), ref1)
    with torch.no_grad():
        model.m.head.bias.add_(1.0)
    assert torch.allclose(model(x1), ref1 + 1.0, atol=1e-5)


def test_keep_ratio_one_is_identity_and_tiny_ratio_keeps_one_patch(pkg):
    """attention.py:31-39 edge cases: keep_ratio = 1.0 keeps every token (the block still scores and gathers, the result
    must equal the un-pruned model bit for bit); a tiny ratio keeps CLS + exactly one patch (keep = max(1, ...))."""
    x = make_images(3, 224, 21).cuda()
    dense = build(pkg, "vit_tiny_patch16_224", {})(x)
    ident = build(pkg, "vit_tiny_patch16_224", {2: {"keep_ratio": 1.0}, 5: {"keep_ratio": 1.0, "update": False}})
    y = ident(x)
    assert ident.get_last_stats()["token_counts"] == [197] * 12
    assert torch.equal(y, dense)
    for k in ident._last_keep_idx:
        if k is not None:
            assert torch.equal(k.cpu().long(), torch.arange(197).expand(3, -1))
    one = build(pkg, "vit_tiny_patch16_224", {4: {"keep_ratio": 0.001}})
    y1 = one(x)
    assert one.get_last_stats()["token_counts"] == [197] * 5 + [2] * 7 and torch.isfinite(y1).all()
    params = orc.extract_params(copy.deepcopy(one.m).cpu().float())
    ref, _ = orc.forward(params, x.cpu(), {4: {"keep_ratio": 0.001}}, forced_keep=[None if k is None else k.cpu().long() for k in one._last_keep_idx])
    assert (y1.cpu() - ref).abs().max().item() < 0.08


def test_batch_of_one(pkg):
    model = build(pkg, "vit_tiny_patch16_224", C1_SCHEDULE)
    x = make_images(5, 224, 33).cuda()
    full = model(x)
    for b in (0, 4):
        assert torch.equal(model(x[b:b + 1].contiguous()), full[b:b + 1])


def test_second_gpu_in_the_same_process(pkg):
    """One process driving two GPUs: per-device kernel attributes and the device guard in forward()."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    x = make_images(4, 224, 5)
    y0 = build(pkg, "vit_tiny_patch16_224", C1_SCHEDULE)(x.cuda())
    m1 = pkg.RAJNIViTWrapper(__import__("rajni_vit_b200.vit", fromlist=["create_model"]).create_model("vit_tiny_patch16_224", seed=0), C1_SCHEDULE).to("cuda:1").eval()
    y1 = m1(x.to("cuda:1"))
    assert torch.equal(y0.cpu(), y1.cpu())


# ------------------------------------------------------------------ real-weights path (run.py:89-92,126-129)
@pytest.mark.parametrize("name,sched,batch,size", [("vit_micro_patch16_64", MICRO_SCHEDULE, 4, 64),
                                                   ("vit_base_patch16_224", README_SCHEDULE, 8, 224)])
def test_trained_like_checkpoint_end_to_end(pkg, tmp_path, name, sched, batch, size):
    """A checkpoint whose parameters have a trained ViT's statistics (LayerNorm gains 0.3..2.5 and non-zero shifts,
    O(0.5) biases, a few massive-activation channels) goes file -> load_checkpoint -> wrapper -> logits; the oracle
    runs the same fp32 weights with our kept indices forced.  Logits: max |d| <= 3 % of the logit std + 0.02 (bf16
    activations; the random-init models sit at 0.08 for std 0.57); kept sets exact outside a 6 % tie band (the residual
    stream reaches +-250 here and the attention logits are ~3x those of a random-init model, so the bf16 rounding of q.k
    moves the scores ~3x more than in test_forward_vs_oracle_full_models, whose band is 3 %)."""
    from rajni_vit_b200.checkpoint import write_safetensors
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0), seed=1)
    path = str(tmp_path / "w.safetensors")
    write_safetensors(path, pkg.RAJNIViTWrapper(copy.deepcopy(base), sched).state_dict())     # both key families, as a saved wrapper has
    loaded = pkg.load_checkpoint(path)
    for (k, a), (_, b) in zip(base.state_dict().items(), loaded.state_dict().items()):
        assert torch.equal(a, b), k
    params = orc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(loaded, sched).cuda().eval()
    images = make_images(batch, size, 99)
    logits = model(images.cuda()).cpu()
    ours = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
    trace = []
    ref, stats = orc.forward(params, images, sched, trace=trace, forced_keep=ours)
    assert model.get_last_stats() == stats and torch.isfinite(logits).all()
    err, std = (logits - ref).abs().max().item(), ref.std().item()
    xmax = max(rec["x_out"].abs().max().item() for rec in trace)
    print(f"{name} trained-like: max |dlogit| {err:.4f} at logit std {std:.3f}; largest residual-stream value {xmax:.1f}")
    assert err <= 0.03 * std + 0.02
    top2 = ref.topk(2, dim=1).values
    decided = (top2[:, 0] - top2[:, 1]) > 2 * err
    assert bool((logits.argmax(1) == ref.argmax(1))[decided].all())
    for rec, kidx in zip(trace, ours):
        if kidx is None:
            continue
        ov, worst = near_tie_mismatch(kidx, rec["scores"], kidx.shape[1] - 1, 0.06)
        print(f"  block {rec['block']}: kept-set overlap {ov:.4f}, worst disagreeing token {worst:.2e} from the cut")
        assert worst < 0.06 and ov > 0.98


# ------------------------------------------------------------------ f4: schedule sweep / search on the device
def test_schedule_sweep_and_search(pkg):
    """rajni_vit_b200.schedule on a small stand-in: the dense model agrees with itself, every candidate reports the
    token counts its schedule implies, pruning lowers the tensor work, labels switch the accuracy axis to top-1, and the
    greedy search returns a schedule at or above its floor."""
    from rajni_vit_b200 import schedule as S
    from rajni_vit_b200.vit import create_model
    make = lambda: create_model("vit_micro_patch16_64", seed=0)                    # noqa: E731
    depth = len(make().blocks)
    g = torch.Generator().manual_seed(3)
    batches = [torch.randn(16, 3, 64, 64, generator=g) for _ in range(2)]
    res = S.sweep(make, batches, candidates=[("dense", {}), ("half", {1: {"keep_ratio": 0.5}}),
                                              ("carried", {1: {"keep_ratio": 0.7}, 2: {"keep_ratio": 0.7, "update": False}})])
    assert res[0]["agreement"] == 100.0 and res[0]["top1"] is None and res[0]["accuracy"] == 100.0
    for r in res:
        assert r["token_counts"] == S.token_counts(r["schedule"], depth, 17) and r["img_s"] > 0
        assert 0.0 <= r["agreement"] <= 100.0
    assert res[1]["gflop_per_image"] < res[0]["gflop_per_image"]
    assert [r["name"] for r in S.pareto_front(res)][-1] == "dense" or res[0]["img_s"] >= max(r["img_s"] for r in res)
    # labels: the accuracy axis becomes top-1 against them (here: the dense model's own predictions -> 100 % for dense)
    labels = [p.cpu() for p in res[0]["predictions"]]
    lab = S.measure(make, {}, list(zip(batches, labels)))
    assert lab["top1"] == 100.0 and lab["accuracy"] == 100.0
    sched, hist = S.search(make, batches, floor=50.0, ratios=(1.0, 0.75, 0.5), timing_steps=3)
    assert hist[0]["schedule"] == {} and all(h["accuracy"] >= 50.0 for h in hist)
    assert sched == hist[-1]["schedule"]
