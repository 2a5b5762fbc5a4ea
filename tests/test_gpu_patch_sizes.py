"""ViTs with 8- and 32-pixel patches on the B200: the any-patch im2col, scores past the per-image kernel's shared memory
(785 tokens of a ViT-B/8 and longer), and the wrapper end to end against the oracle."""
import copy

import pytest
import torch

import tests.test_gpu_e2e as e2e
from oracle import rajni_oracle as orc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, bf16_round, make_images

pytestmark = pytest.mark.gpu

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
BF16_RTOL = 2.0 ** -7


@pytest.fixture(scope="module")
def ops():
    from rajni_vit_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def _im2col(ops, images, p, C=128, stats=True):
    B, _, S, _ = images.shape
    P = (S // p) ** 2
    cols = torch.full((B * P, 3 * p * p), float("nan"), device="cuda", dtype=torch.bfloat16)
    x = torch.zeros((B * (P + 1), C), device="cuda", dtype=torch.bfloat16)
    cls_pos0 = torch.arange(C, device="cuda", dtype=torch.float32).div(64).to(torch.bfloat16)
    row_stats = torch.full((3, B * (P + 1), 2), 7.0, device="cuda") if stats else None
    ops.patch_im2col(images, p, cols, cls_pos0, x, C, row_stats=row_stats, stats_slots=3 if stats else 0,
                     cls_sum=1.5, cls_sumsq=2.5, norm=(MEAN, STD) if images.dtype == torch.uint8 else None)
    return cols.cpu(), x.cpu().view(B, P + 1, C), cls_pos0.cpu(), None if row_stats is None else row_stats.cpu()


# (patch, S): S not a multiple of 16 wherever the patch allows it
@pytest.mark.parametrize("p,S", [(8, 72), (8, 224), (16, 64), (16, 224), (24, 72), (24, 240), (32, 96), (32, 224)])
@pytest.mark.parametrize("B", [1, 3])
def test_im2col_any_patch(ops, p, S, B):
    g = torch.Generator().manual_seed(p * 1000 + S + B)
    f32 = torch.randn(B, 3, S, S, generator=g)
    P = (S // p) ** 2
    unf = torch.nn.functional.unfold(bf16_round(f32), p, stride=p).transpose(1, 2).reshape(B * P, 3 * p * p)
    for images in (f32, f32.to(torch.bfloat16)):
        cols, x, cls_pos0, st = _im2col(ops, images.cuda(), p)
        assert torch.equal(cols.float(), unf), images.dtype
        assert torch.equal(x[:, 0], cls_pos0.expand(B, -1)) and (x[:, 1:] == 0).all()       # CLS rows only
        st = st.view(3, B, P + 1, 2)
        assert (st[0, :, 0] == torch.tensor([1.5, 2.5])).all() and (st[1:, :, 0] == 0).all() and (st[:, :, 1:] == 7.0).all()
    # uint8: the same bf16 patches as the fp32 ToTensor + Normalize pipeline
    u8 = torch.randint(0, 256, (B, 3, S, S), generator=g, dtype=torch.uint8)
    u8[0, :, 0, :2] = torch.tensor([0, 255], dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    c8 = _im2col(ops, u8.cuda(), p, stats=False)[0]
    cf = _im2col(ops, xf.cuda(), p, stats=False)[0]
    assert torch.equal(c8, cf)


def test_im2col_rejects_other_patches(ops):
    from rajni_vit_b200._lib import RajniError
    img = torch.zeros(1, 3, 56, 56, device="cuda")
    for p in (4, 12, 14, 28):
        with pytest.raises(RajniError):
            _im2col(ops, img, p)
    with pytest.raises(RajniError):
        _im2col(ops, torch.zeros(1, 3, 60, 60, device="cuda"), 8)           # S % p != 0


@pytest.mark.parametrize("p,S,C,B", [(8, 72, 128, 3), (32, 224, 192, 2)])
def test_patch_embed_gemm_at_other_k(ops, p, S, C, B):
    """The embed GEMM at K = 3 p^2 = 192 and 3072 against the oracle's Conv2d (tolerance of test_gpu_kernels' patch embed)."""
    g = torch.Generator().manual_seed(p + S + C)
    images = torch.randn(B, 3, S, S, generator=g)
    K = 3 * p * p
    w = bf16_round(torch.randn(C, 3, p, p, generator=g) / K ** 0.5)
    bias = bf16_round(torch.randn(C, generator=g))
    P = (S // p) ** 2
    pos = bf16_round(torch.randn(1, P + 1, C, generator=g) * 0.02)
    cls = bf16_round(torch.randn(1, 1, C, generator=g) * 0.02)
    ref = orc.embed(dict(patch=p, pe_w=w, pe_b=bias, cls=cls, pos=pos), bf16_round(images)).reshape(B * (P + 1), C)
    cols = torch.empty((B * P, K), device="cuda", dtype=torch.bfloat16)
    x = torch.zeros((B * (P + 1), C), device="cuda", dtype=torch.bfloat16)
    ops.patch_im2col(images.cuda(), p, cols, (cls[0, 0] + pos[0, 0]).to("cuda", torch.bfloat16), x, C)
    idx = torch.arange(B * P, dtype=torch.int32)
    ops.gemm(cols, w.reshape(C, K).to("cuda", torch.bfloat16), bias.cuda(), B * P, C, K,
             residual=pos[0].to("cuda", torch.bfloat16), ldres=C, res_row_map=(1 + idx % P).cuda(),
             out=x, ldd=C, out_row_map=((idx // P) * (P + 1) + 1 + idx % P).cuda())
    got = x.cpu().float()
    assert ((got - ref).abs() <= BF16_RTOL * ref.abs() + 4e-3).all()


# ------------------------------------------------------------------ long-sequence scores
def _qkv(B, N, H, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, N, 3 * H * 64, device="cuda", generator=g).to(torch.bfloat16)


def _check_scores_against_oracle(scores, idx, nxt, rmap, qkv, H, keep, rows):
    """rows: the images checked against the fp64 oracle (all of them at small batches)."""
    B, N = scores.shape
    idx_all = idx.cpu().long()
    assert (idx_all[:, 0] == 0).all() and (idx_all[:, 1:] > idx_all[:, :-1]).all()
    assert torch.equal(nxt.cpu(), torch.gather(scores.cpu(), 1, idx_all))
    assert torch.equal(rmap.cpu().long().view(B, -1), idx_all + torch.arange(B)[:, None] * N)
    assert torch.equal(idx_all, orc.select(scores.cpu(), keep))               # selection is exact on the kernel's own scores
    s = scores[rows].cpu().double()
    ref = orc.importance(qkv[rows].cpu().double(), H)
    torch.testing.assert_close(s, ref, rtol=1e-5, atol=1e-12)
    # the oracle's kept set wherever no tie straddles the cut within rounding
    srt = torch.sort(ref[:, 1:], dim=1, descending=True).values
    gap = (srt[:, keep - 1] - srt[:, keep]) / srt[:, keep - 1]
    decided = gap > 1e-4
    assert torch.equal(idx_all[rows][decided], orc.select(ref, keep)[decided])


@pytest.mark.parametrize("N", [724, 785, 1025, 2305])
@pytest.mark.parametrize("H", [6, 12, 16])
@pytest.mark.parametrize("B", [1, 3, 200])
def test_long_sequence_score_select(ops, N, H, B):
    long = ops.needs_score_workspace(N, H)
    assert long or (N, H) == (724, 6)                # 724 tokens still fit the one-launch kernel at 6 heads
    qkv = _qkv(B, N, H, N * 100 + H * 10 + B)
    keep = orc.keep_count(N, 0.88)
    scores, idx, nxt, rmap = ops.score_select(qkv, H, keep, want_scores=True)    # split path on both sides of SPLIT_SCORE_MAX_BATCH
    rows = list(range(B)) if B <= 3 else [0, 1, B - 1]
    _check_scores_against_oracle(scores, idx, nxt, rmap, qkv, H, keep, rows)
    if B > 3:                                    # images are independent: a sub-batch reproduces its rows bit for bit
        s2, i2, _, _ = ops.score_select(qkv[97:100].contiguous(), H, keep, want_scores=True)
        assert torch.equal(s2, scores[97:100]) and torch.equal(i2, idx[97:100])
    # the one-launch entry points keep refusing what needs scratch
    from rajni_vit_b200._lib import RajniError
    if long:
        with pytest.raises(RajniError) as e:
            ops.score_select(qkv[:1], H, keep, split=False)
        assert e.value.code == -1


def test_compute_importance_at_785_tokens(pkg):
    B, N, H = 3, 785, 12
    qkv = _qkv(B, N, H, 7)
    got = pkg.compute_importance(qkv, H)
    assert got.dtype == torch.bfloat16                           # qkv's dtype, as the reference
    f32 = pkg.compute_importance(qkv.float(), H)
    ref = orc.importance(qkv.cpu().double(), H)
    torch.testing.assert_close(f32.cpu().double(), ref, rtol=1e-5, atol=1e-12)
    from rajni_vit_b200 import ops
    s, _, _, _ = ops.score_select(qkv, H, 600, want_scores=True)
    assert torch.equal(f32, s)                                   # scores-only call = the scores of the selecting call


@pytest.mark.parametrize("B,N,H,ratio", [(3, 577, 12, 0.88), (2, 197, 12, 0.88), (200, 197, 6, 0.7), (2, 723, 12, 0.8)])
def test_workspace_tail_matches_shared_memory_tail(ops, monkeypatch, B, N, H, ratio):
    """Where the shared-memory tail fits, the workspace tail (forced) gives the same bits: same reads, same arithmetic."""
    qkv = _qkv(B, N, H, 31 + N)
    keep = orc.keep_count(N, ratio)
    a = ops.score_select(qkv, H, keep, want_scores=True, split=True)
    monkeypatch.setenv("RAJNI_SCORE_WS_TAIL", "1")
    b = ops.score_select(qkv, H, keep, want_scores=True, split=True)
    monkeypatch.delenv("RAJNI_SCORE_WS_TAIL")
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ------------------------------------------------------------------ the wrapper end to end
@pytest.mark.parametrize("name,batch", [("vit_base_patch32_224", 16), ("vit_base_patch8_224", 2)])
def test_forward_vs_oracle_patch_variants(pkg, name, batch):
    """As test_gpu_e2e.test_forward_vs_oracle_full_models: token_counts exact, teacher-forced logits within the bf16
    tolerance with top-1 agreement where decided, kept sets within the tie band."""
    e2e.test_forward_vs_oracle_full_models(pkg, name, README_SCHEDULE, batch, 224)


def test_patch32_full_batch_graph_determinism_and_sub_batch(pkg):
    """ViT-B/32 at 256 images (12 800 token rows): the automatic rule replays a CUDA graph, bit-identical to the eager
    launches; the run is deterministic; a sub-batch reproduces its rows.  Blocks of <= 64 tokens pack k consecutive images
    into one attention tile (k divides the batch), so the sub-batch is images[64:96], which starts and ends on a group
    boundary for every such k up to 32."""
    model = e2e.build(pkg, "vit_base_patch32_224", README_SCHEDULE)
    images = make_images(256, 224, 1234).cuda()
    assert model.use_cuda_graph is None
    y = model(images)
    assert len(model._graphs) == 1                                      # replayed from a graph
    assert model.get_last_stats()["token_counts"] == [50, 50, 50, 50, 44, 38, 38, 38, 30, 21, 21, 21]
    assert torch.isfinite(y).all()
    assert torch.equal(model(images), y)
    model.use_cuda_graph = False
    assert torch.equal(model(images), y)                                # eager = graph replay
    model.use_cuda_graph = None
    sub = model(images[64:96].contiguous())
    assert torch.equal(sub, y[64:96])


def test_uint8_input_matches_fp32_at_patch8(pkg):
    model = e2e.build(pkg, "vit_micro_patch8_72", MICRO_SCHEDULE)
    g = torch.Generator().manual_seed(8)
    u8 = torch.randint(0, 256, (4, 3, 72, 72), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    ref = model(xf.cuda()).clone()
    assert model.get_last_stats()["token_counts"] == [82, 82, 61, 37]
    model.set_input_normalization(MEAN, STD)
    assert torch.equal(model(u8.cuda()), ref)


@pytest.mark.parametrize("name,size", [("vit_micro_patch32_128", 128), ("vit_micro_patch8_72", 72)])
def test_micro_patch_models_vs_oracle(pkg, name, size):
    from rajni_vit_b200.vit import create_model
    base = create_model(name, seed=2)
    params = orc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, {}).cuda().eval()
    images = make_images(5, size, 3)
    logits = model(images.cuda()).cpu()
    ref, stats = orc.forward(params, images, {})
    assert model.get_last_stats() == stats
    assert (logits - ref).abs().max().item() < 0.05
    with pytest.raises(ValueError, match="multiple of the patch size"):
        model(torch.zeros(1, 3, size + 4, size + 4, device="cuda"))


def test_safetensors_round_trip_patch32(pkg, tmp_path):
    from rajni_vit_b200.checkpoint import write_safetensors
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model("vit_micro_patch32_128", seed=0), seed=1)
    path = str(tmp_path / "w.safetensors")
    write_safetensors(path, base.state_dict())
    loaded = pkg.load_checkpoint(path)
    images = make_images(4, 128, 5).cuda()
    a = pkg.RAJNIViTWrapper(copy.deepcopy(base), MICRO_SCHEDULE).cuda().eval()(images)
    b = pkg.RAJNIViTWrapper(loaded, MICRO_SCHEDULE).cuda().eval()(images)
    assert torch.equal(a, b)
