"""The two DeiT families on the B200: selection with two always-kept prefix tokens on every score/select path, the
prefix-aware entry points against the old ones at one prefix token, the im2col prefix rows, and the wrapper end to end
(LayerScale folded into proj / fc2, no position for DeiT-III's class token, the distilled model's two-head average)
against the DeiT reference (tests/deit_oracle.py, the oracle extended to the two families)."""
import copy

import pytest
import torch

from tests import deit_oracle as dorc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images

pytestmark = pytest.mark.gpu

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


@pytest.fixture(scope="module")
def ops():
    from rajni_vit_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def _qkv(B, N, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, N, 3 * H * 64, device="cuda", generator=g).to(torch.bfloat16)


def _check_selection(scores, idx, nxt, rmap, keep, prefix):
    """Kept set exact on the kernel's own scores, prefix tokens first, next_scores and row_map consistent."""
    B, N = scores.shape
    idx_all = idx.cpu().long()
    assert idx_all.shape == (B, keep + prefix)
    assert (idx_all[:, :prefix] == torch.arange(prefix)).all() and (idx_all[:, 1:] > idx_all[:, :-1]).all()
    assert torch.equal(nxt.cpu(), torch.gather(scores.cpu(), 1, idx_all))
    if rmap is not None:
        assert torch.equal(rmap.cpu().long().view(B, -1), idx_all + torch.arange(B)[:, None] * N)
    assert torch.equal(idx_all, dorc.select(scores.cpu(), keep, prefix))


def _check_against_oracle(scores, idx, qkv, H, keep, prefix, rows):
    """Scores within rel 1e-5 of the fp64 oracle; the oracle's kept set wherever no tie straddles the cut within rounding."""
    s = scores[rows].cpu().double()
    ref = dorc.importance(qkv[rows].cpu().double(), H)
    torch.testing.assert_close(s, ref, rtol=1e-5, atol=1e-12)
    srt = torch.sort(ref[:, prefix:], dim=1, descending=True).values
    gap = (srt[:, keep - 1] - srt[:, keep]) / srt[:, keep - 1]
    decided = gap > 1e-4
    assert decided.float().mean() > 0.5
    assert torch.equal(idx.cpu().long()[rows][decided], dorc.select(ref, keep, prefix)[decided])


# (B, N, H, ratio, split): N <= 256 takes the rank-by-counting selection, N > 256 the radix one; split=None lets ops pick
# (B <= 148: the split path), False forces the one-launch kernel; 785 tokens need the workspace tail at any batch
PATHS = [(3, 198, 12, 0.88, False), (3, 198, 12, 0.88, None), (200, 198, 6, 0.7, None), (3, 578, 12, 0.88, False),
         (3, 578, 12, 0.8, None), (200, 578, 12, 0.72, None), (2, 786, 12, 0.88, None), (4, 18, 2, 0.5, None)]


@pytest.mark.parametrize("B,N,H,ratio,split", PATHS)
def test_score_select_two_prefix_tokens(ops, B, N, H, ratio, split):
    qkv = _qkv(B, N, H, N * 7 + B)
    keep = dorc.keep_count(N, ratio, 2)
    scores, idx, nxt, rmap = ops.score_select(qkv, H, keep, want_scores=True, split=split, prefix=2)
    _check_selection(scores, idx, nxt, rmap, keep, 2)
    rows = list(range(B)) if B <= 4 else [0, 1, B - 1]
    _check_against_oracle(scores, idx, qkv, H, keep, 2, rows)
    # the scores do not depend on the prefix count
    s1, _, _, _ = ops.score_select(qkv, H, dorc.keep_count(N, ratio), want_scores=True, split=split)
    assert torch.equal(s1, scores)
    from rajni_vit_b200._lib import RajniError
    with pytest.raises(RajniError, match="selected index k out of range") as e:
        ops.score_select(qkv, H, N - 1, split=split, prefix=2)
    assert e.value.code == -4


@pytest.mark.parametrize("B,N,H,ratio", [(3, 198, 12, 0.88), (200, 198, 6, 0.7), (3, 578, 12, 0.8)])
def test_workspace_tail_two_prefix_tokens(ops, monkeypatch, B, N, H, ratio):
    """The workspace tail (forced) selects with the prefix rule too, bit-identical to the shared-memory tail."""
    qkv = _qkv(B, N, H, 5 + N)
    keep = dorc.keep_count(N, ratio, 2)
    a = ops.score_select(qkv, H, keep, want_scores=True, split=True, prefix=2)
    monkeypatch.setenv("RAJNI_SCORE_WS_TAIL", "1")
    b = ops.score_select(qkv, H, keep, want_scores=True, split=True, prefix=2)
    monkeypatch.delenv("RAJNI_SCORE_WS_TAIL")
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    _check_selection(b[0], b[1], b[2], b[3], keep, 2)


@pytest.mark.parametrize("B,N", [(5, 198), (3, 578), (2, 1200)])
def test_select_on_carried_scores_two_prefix_tokens(ops, B, N):
    g = torch.Generator().manual_seed(N)
    s = torch.rand(B, N, generator=g) / N
    s[:, :2] = -1.0                                  # the prefix tokens are kept whatever their scores
    s[0, 10:20] = s[0, 30]                           # a run of ties: lower index first
    for ratio in (0.88, 0.5, 0.01, 1.0):
        keep = dorc.keep_count(N, ratio, 2)
        idx, nxt, rmap = ops.select(s.cuda(), keep, prefix=2)
        _check_selection(s, idx, nxt, rmap, keep, 2)
    from rajni_vit_b200._lib import RajniError
    with pytest.raises(RajniError, match="selected index k out of range"):
        ops.select(s.cuda(), N - 1, prefix=2)


def test_one_prefix_token_through_the_new_entry_points_is_bit_identical(ops):
    """ops calls the *_prefix entry points; at prefix 1 they reproduce the old entry points bit for bit on every path."""
    from rajni_vit_b200 import _lib
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    for B, N, H in ((3, 197, 12), (200, 197, 6), (3, 577, 12), (2, 785, 12)):
        qkv = _qkv(B, N, H, B + N)
        keep = dorc.keep_count(N, 0.8)
        C = 64 * H
        for split in (False, True):
            if not split and ops.needs_score_workspace(N, H):
                continue
            new = ops.score_select(qkv, H, keep, want_scores=True, split=split)
            old = [torch.empty_like(new[0]), torch.empty_like(new[1]), torch.empty_like(new[2]), torch.empty_like(new[3])]
            if split:
                ws = torch.empty(ops.score_workspace_bytes(B, N, C, H), device="cuda", dtype=torch.uint8)
                rc = lib.rajni_score_select_split(qkv.data_ptr(), B, N, C, H, keep, 1e-6, old[0].data_ptr(), old[1].data_ptr(),
                                                  old[2].data_ptr(), old[3].data_ptr(), ws.data_ptr(), ws.numel(), stream)
            else:
                rc = lib.rajni_score_select(qkv.data_ptr(), B, N, C, H, keep, 1e-6, old[0].data_ptr(), old[1].data_ptr(),
                                            old[2].data_ptr(), old[3].data_ptr(), stream)
            _lib.check(rc)
            for a, b in zip(new, old):
                assert torch.equal(a, b), (B, N, split)
        sel_new = ops.select(new[0], keep)
        sel_old = [torch.empty_like(t) for t in sel_new]
        _lib.check(lib.rajni_select(new[0].data_ptr(), B, N, keep, sel_old[0].data_ptr(), sel_old[1].data_ptr(),
                                    sel_old[2].data_ptr(), stream))
        for a, b in zip(sel_new, sel_old):
            assert torch.equal(a, b)
    # im2col at prefix 1: same cols, CLS rows and LayerNorm partials as rajni_patch_im2col
    for p, S in ((16, 224), (8, 72)):
        img = torch.randn(3, 3, S, S, device="cuda")
        P, C = (S // p) ** 2, 192
        cls_pos0 = torch.randn(C, device="cuda").to(torch.bfloat16)
        outs = []
        for use_new in (True, False):
            cols = torch.zeros(3 * P, 3 * p * p, device="cuda", dtype=torch.bfloat16)
            x = torch.zeros(3 * (P + 1), C, device="cuda", dtype=torch.bfloat16)
            st = torch.full((3, 3 * (P + 1), 2), 7.0, device="cuda")
            if use_new:
                ops.patch_im2col(img, p, cols, cls_pos0, x, C, row_stats=st, stats_slots=3, cls_sum=1.25, cls_sumsq=3.5)
            else:
                _lib.check(lib.rajni_patch_im2col(img.data_ptr(), 1, 3, S, p, cols.data_ptr(), cls_pos0.data_ptr(), x.data_ptr(), C,
                                                  st.data_ptr(), st.shape[1], 3, 1.25, 3.5, None, stream))
            outs.append((cols, x, st))
        for a, b in zip(*outs):
            assert torch.equal(a, b)


# ------------------------------------------------------------------ im2col prefix rows
@pytest.mark.parametrize("p,S", [(16, 64), (16, 224), (8, 72)])
@pytest.mark.parametrize("prefix", [1, 2])
def test_im2col_prefix_rows_and_their_partial_sums(ops, p, S, prefix):
    """prefix rows copied in front of every image's patches (a [prefix, C] block: tokens + positions, or the class token
    alone under no_embed_class, which the kernel does not tell apart), slot 0 of their LayerNorm partials = the host's
    (sum, sum of squares), other slots zero, patch rows and their stats untouched; fp32 and uint8 pixels."""
    B, C = 3, 256
    P = (S // p) ** 2
    N0 = P + prefix
    g = torch.Generator().manual_seed(S + prefix)
    rows = torch.randn(prefix, C, generator=g).to(torch.bfloat16)
    r32 = rows.float()
    sums, sqs = r32.sum(1).tolist(), (r32 * r32).sum(1).tolist()
    u8 = torch.randint(0, 256, (B, 3, S, S), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    unf = torch.nn.functional.unfold(xf.to(torch.bfloat16).float(), p, stride=p).transpose(1, 2).reshape(B * P, 3 * p * p)
    for images in (xf, u8):
        cols = torch.full((B * P, 3 * p * p), float("nan"), device="cuda", dtype=torch.bfloat16)
        x = torch.zeros((B * N0, C), device="cuda", dtype=torch.bfloat16)
        st = torch.full((3, B * N0, 2), 7.0, device="cuda")
        ops.patch_im2col(images.cuda(), p, cols, rows.cuda().reshape(-1) if prefix == 1 else rows.cuda(), x, C, row_stats=st,
                         stats_slots=3, cls_sum=sums if prefix > 1 else sums[0], cls_sumsq=sqs if prefix > 1 else sqs[0],
                         norm=(MEAN, STD) if images.dtype == torch.uint8 else None, prefix=prefix)
        assert torch.equal(cols.cpu().float(), unf), images.dtype
        x = x.cpu().view(B, N0, C)
        assert torch.equal(x[:, :prefix], rows.expand(B, -1, -1)) and (x[:, prefix:] == 0).all()
        st = st.cpu().view(3, B, N0, 2)
        want = torch.tensor([sums, sqs]).T                     # [prefix, 2]
        assert torch.equal(st[0, :, :prefix], want.expand(B, -1, -1))
        assert (st[1:, :, :prefix] == 0).all() and (st[:, :, prefix:] == 7.0).all()


# ------------------------------------------------------------------ the wrapper end to end
def _near_tie_mismatch(ours, ref_scores, keep, prefix, rel_gap):
    """test_gpu_e2e.near_tie_mismatch with ``prefix`` always-kept leading tokens."""
    B = ours.shape[0]
    worst, overlap, in_band, cands = 0.0, 0.0, 0, 0
    for b in range(B):
        s = ref_scores[b, prefix:].double()
        cut = torch.sort(s, descending=True).values[keep - 1].item()
        ref_set = set((torch.sort(s, descending=True, stable=True).indices[:keep] + prefix).tolist())
        our_set = set(ours[b, prefix:].tolist())
        overlap += len(ref_set & our_set) / keep
        for t in ref_set ^ our_set:
            worst = max(worst, abs(s[t - prefix].item() - cut) / abs(cut))
        in_band += int(((s - cut).abs() <= rel_gap * abs(cut)).sum())
        cands += s.numel()
    return overlap / B, worst, in_band / max(cands, 1)


def _forward_vs_oracle(pkg, base, sched, images, logit_tol, band):
    """As test_gpu_e2e.test_forward_vs_oracle_full_models, prefix-aware: selection teacher-forced, logits within
    ``logit_tol(std)``, top-1 equal where decided, kept sets exact outside a ``band`` tie band, token counts exact."""
    params = dorc.extract_params(copy.deepcopy(base))
    prefix = params["prefix"]
    model = pkg.RAJNIViTWrapper(base, sched).cuda().eval()
    logits = model(images.cuda()).cpu()
    ours = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
    for k in ours:
        if k is not None:
            assert (k[:, :prefix] == torch.arange(prefix)).all() and (k[:, 1:] > k[:, :-1]).all()
    trace = []
    ref, stats = dorc.forward(params, images, sched, trace=trace, forced_keep=ours)
    assert model.get_last_stats() == stats
    assert torch.isfinite(logits).all()
    err, std = (logits - ref).abs().max().item(), ref.std().item()
    print(f"(selection teacher-forced): max |dlogit| {err:.4f}, logit std {std:.3f}")
    assert err < logit_tol(std)
    top2 = ref.topk(2, dim=1).values
    decided = (top2[:, 0] - top2[:, 1]) > 2 * err
    assert bool((logits.argmax(1) == ref.argmax(1))[decided].all())
    for rec, kidx in zip(trace, ours):
        if kidx is None:
            continue
        keep = kidx.shape[1] - prefix
        ov, worst, frac = _near_tie_mismatch(kidx, rec["scores"], keep, prefix, band)
        print(f"  block {rec['block']}: kept-set overlap {ov:.4f}, worst disagreeing token {worst:.2e} from the cut")
        assert worst < band
        assert ov > 0.97 and (frac < 0.12 or rec["scores"].shape[1] <= 64), (frac, ov)
    return model, logits


@pytest.mark.parametrize("name,batch,size", [("deit3_base_patch16_224", 16, 224), ("deit3_base_patch16_384", 4, 384),
                                             ("deit_base_distilled_patch16_224", 16, 224),
                                             ("deit_base_distilled_patch16_384", 4, 384)])
def test_forward_vs_oracle_deit_models(pkg, name, batch, size):
    """At the tolerances of test_gpu_e2e.test_forward_vs_oracle_full_models (max |dlogit| < 0.08, 3 % tie band)."""
    from rajni_vit_b200.vit import create_model
    model, _ = _forward_vs_oracle(pkg, create_model(name, seed=0), README_SCHEDULE, make_images(batch, size, 1234),
                                  lambda std: 0.08, 0.03)
    P = (size // 16) ** 2
    prefix = 2 if "distilled" in name else 1
    from rajni_vit_b200 import schedule as S
    assert model.get_last_stats()["token_counts"] == S.token_counts(README_SCHEDULE, 12, P + prefix, prefix=prefix)


@pytest.mark.parametrize("name", ["deit3_micro_patch16_64", "deit_micro_distilled_patch16_64"])
def test_trained_like_micro_models_vs_oracle(pkg, name):
    """Trained-like statistics (test_gpu_e2e.test_trained_like_checkpoint_end_to_end's tolerances) with LayerScale gammas
    spread over [1e-6, 1]."""
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0), seed=1)
    _forward_vs_oracle(pkg, base, MICRO_SCHEDULE, make_images(8, 64, 99), lambda std: 0.03 * std + 0.02, 0.06)
    dense = randomize_trained_like(create_model(name, seed=0), seed=1)
    _forward_vs_oracle(pkg, dense, {}, make_images(8, 64, 98), lambda std: 0.03 * std + 0.02, 0.06)


@pytest.mark.parametrize("name", ["deit3_micro_patch16_64", "deit_micro_distilled_patch16_64"])
def test_graph_replay_and_uint8_input_are_bit_identical(pkg, name):
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    model = pkg.RAJNIViTWrapper(randomize_trained_like(create_model(name, seed=0), seed=1), MICRO_SCHEDULE).cuda().eval()
    x1, x2 = make_images(4, 64, 7).cuda(), make_images(4, 64, 8).cuda()
    model.use_cuda_graph = False
    ref1, ref2 = model(x1).clone(), model(x2).clone()
    stats = model.get_last_stats()
    prefix = 2 if "distilled" in name else 1
    assert stats["token_counts"] == [16 + prefix, 16 + prefix, 12 + prefix, 7 + prefix]
    model.use_cuda_graph = True
    for _ in range(2):
        assert torch.equal(model(x1), ref1) and torch.equal(model(x2), ref2)
        assert model.get_last_stats() == stats and len(model._graphs) == 1
    model.use_cuda_graph = None                                 # automatic: 4 x 18 rows replay a graph
    assert torch.equal(model(x1), ref1)
    # uint8 pixels normalised in the im2col kernel = the fp32 ToTensor + Normalize pipeline, eager and replayed
    g = torch.Generator().manual_seed(3)
    u8 = torch.randint(0, 256, (4, 3, 64, 64), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    model.use_cuda_graph = False
    ref = model(xf.cuda()).clone()
    model.set_input_normalization(MEAN, STD)
    assert torch.equal(model(u8.cuda()), ref)
    model.use_cuda_graph = True
    assert torch.equal(model(u8.cuda()), ref)


def test_distilled_head_is_the_average_of_the_two_heads(pkg):
    """Dense distilled micro model: the one K = 2C head GEMM equals the mean of two separate head GEMMs on the same
    normalised rows within fp32 summation order, and a model whose head_dist equals head reproduces a single-head readout."""
    from rajni_vit_b200 import ops
    from rajni_vit_b200.vit import create_model
    base = create_model("deit_micro_distilled_patch16_64", seed=4)
    model = pkg.RAJNIViTWrapper(base, {}).cuda().eval()
    images = make_images(6, 64, 11).cuda()
    y = model(images)
    ws = next(iter(model._ws.values()))
    ln = ws["cls"]                                              # [B, 2C]: LN(x0) | LN(x1)
    m = model.m
    gn, bn, en = m.norm.weight.float(), m.norm.bias.float(), m.norm.eps
    x = ws["xa"][: 6 * 18].view(6, 18, 128).float()
    want = torch.nn.functional.layer_norm(x[:, :2], (128,), gn, bn, en).to(torch.bfloat16)
    assert (ln.view(6, 2, 128).float() - want.float()).abs().max().item() <= 2 ** -7 * want.float().abs().max().item()
    y0 = ops.gemm(ln[:, :128].contiguous(), m.head.weight.to(torch.bfloat16).contiguous(), m.head.bias.float(), 6, 1000, 128, out_f32=True)
    y1 = ops.gemm(ln[:, 128:].contiguous(), m.head_dist.weight.to(torch.bfloat16).contiguous(), m.head_dist.bias.float(), 6, 1000, 128,
                  out_f32=True)
    torch.testing.assert_close(y, (y0 + y1) / 2, rtol=1e-5, atol=1e-5)
    dense = dorc.forward(dorc.extract_params(copy.deepcopy(base).cpu()), images.cpu(), {})[0]
    assert (y.cpu() - dense).abs().max().item() < 0.05
