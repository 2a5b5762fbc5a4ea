"""Headless ViTs (head = Identity, timm's num_classes=0) on the B200: the fp32-output LayerNorm and pooling kernels against
fp64 torch and against their bf16 siblings, the bridge to the classifier path through an identity head, the wrapper end to
end against the reference (tests/headless_oracle.py), graph replay, uint8 pixels, batch independence and launch counts."""
import copy

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import headless_oracle as horc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images
from tests.test_gpu_deit import MEAN, STD, _near_tie_mismatch
from tests.test_gpu_pool_prenorm import _affine, _pool_ref, _rows

pytestmark = pytest.mark.gpu

WIDTHS = (128, 384, 768, 1024)


@pytest.fixture(scope="module")
def ops():
    from rajni_vit_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def _ln_ref(x, gamma, beta, eps):
    """fp64 LayerNorm on the same bf16 rows, and |gamma| + |beta|, the scale of a normalised value."""
    v = x.double()
    z = (v - v.mean(1, keepdim=True)) / torch.sqrt(v.var(1, unbiased=False, keepdim=True) + eps)
    return z * gamma.double() + beta.double(), (gamma.double().abs() + beta.double().abs()).expand_as(z)


def _close_fp32(got, ref, scale):
    """fp32 math on bf16 rows: the mean, variance and rsqrt carry a few fp32 ulps, so a normalised value is off by ~1e-6 of
    its scale; 1e-5 leaves a margin and is still 400x below one bf16 ulp at that scale."""
    err = (got.double() - ref).abs()
    bad = err > 1e-5 * scale
    assert not bad.any(), (err[bad][:4], ref[bad][:4])


# ------------------------------------------------------------------ kernels
@pytest.mark.parametrize("C", WIDTHS)
def test_layernorm_f32_against_fp64_and_bf16(ops, C):
    """The final norm of a headless model: the class-token rows of [B, N, C] (strided input) into strided fp32 rows."""
    B, N = 64, 197
    gamma, beta = _affine(C, C)
    x = _rows(B, N, C, C + 1)
    ostride = C + 4
    out = torch.full((B, ostride), float("nan"), device="cuda")
    ops.layernorm(x, gamma, beta, 1e-6, B, C, in_row_stride=N * C, out=out, out_row_stride=ostride)
    assert torch.isnan(out[:, C:]).all()
    y = out[:, :C]
    ref, scale = _ln_ref(x.view(B, N, C)[:, 0], gamma, beta, 1e-6)
    _close_fp32(y, ref, scale)
    # bf16 rounding of the fp32 row is the bf16 kernel's row, bit for bit
    bf = ops.layernorm(x, gamma, beta, 1e-6, B, C, in_row_stride=N * C)
    assert torch.equal(y.to(torch.bfloat16), bf)
    # dense rows, offsets (a distilled layout's second row), every row of the matrix
    dense = ops.layernorm(x, gamma, beta, 1e-6, B * N, C, out=torch.empty(B * N, C, device="cuda"))
    assert torch.equal(dense.to(torch.bfloat16), ops.layernorm(x, gamma, beta, 1e-6, B * N, C))
    off = torch.empty(B, 2 * C, device="cuda")
    ops.layernorm(x, gamma, beta, 1e-6, B, C, in_row_stride=N * C, in_offset=C, out=off, out_row_stride=2 * C, out_offset=C)
    assert torch.equal(off[:, C:].to(torch.bfloat16),
                       ops.layernorm(x, gamma, beta, 1e-6, B, C, in_row_stride=N * C, in_offset=C))


@pytest.mark.parametrize("C", WIDTHS)
@pytest.mark.parametrize("P0", [1, 2])
def test_mean_pool_layernorm_f32_against_fp64_and_bf16(ops, C, P0):
    for N in (17, 197, 785):
        gamma, beta = _affine(C, C + N)
        B = 8 if N == 785 else 32
        x = _rows(B, N, C, N + C + P0)
        ostride = C + 4
        out = torch.full((B, ostride), float("nan"), device="cuda")
        ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=P0, out=out, out_row_stride=ostride)
        assert torch.isnan(out[:, C:]).all()
        y = out[:, :C]
        ref, scale = _pool_ref(x, B, N, P0, gamma, beta, 1e-6)
        _close_fp32(y, ref, scale)
        assert torch.equal(y.to(torch.bfloat16), ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=P0))
        one = ops.mean_pool_layernorm(x[3 * N: 4 * N].contiguous(), 1, N, C, gamma, beta, 1e-6, prefix=P0,
                                      out=torch.empty(1, C, device="cuda"))
        assert torch.equal(one[0], y[3])                  # batch-independent, as the bf16 instance


def test_f32_entry_points_refuse_bad_shapes_and_strides(ops):
    import ctypes
    from rajni_vit_b200 import _lib
    from rajni_vit_b200._lib import RajniError
    lib = _lib.load()
    C = 128
    gamma, beta = _affine(C, 0)
    x = _rows(4, 17, C, 0)
    y = torch.empty(4, 2 * C, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    ln = lambda rows, c, ostride, ptr=y.data_ptr(): lib.rajni_layernorm_strided_f32(                  # noqa: E731
        x.data_ptr(), 17 * C, gamma.data_ptr(), beta.data_ptr(), ctypes.c_float(1e-6), ptr, ostride, rows, c, s)
    assert ln(4, C, C + 4) == 0
    for rows, c, ostride in ((4, C, C + 2), (4, C, C - 4), (4, 12, 16), (0, C, C), (4, 4096, 4096)):
        assert ln(rows, c, ostride) == _lib.RAJNI_EINVAL, (rows, c, ostride)
        assert b"rajni_layernorm_f32" in lib.rajni_last_error()
    assert ln(4, C, C, ptr=None) == _lib.RAJNI_EINVAL
    pool = lambda B, N, P0, c, ostride: lib.rajni_mean_pool_layernorm_f32(                           # noqa: E731
        x.data_ptr(), B, N, P0, c, gamma.data_ptr(), beta.data_ptr(), ctypes.c_float(1e-6), y.data_ptr(), ostride, s)
    assert pool(4, 17, 1, C, C + 4) == 0
    for B, N, P0, c, ostride in ((4, 17, 1, C, C + 2), (4, 17, 1, C, C - 4), (4, 17, 1, 96, 96), (4, 17, 3, C, C),
                                 (4, 2, 2, C, C), (0, 17, 1, C, C)):
        assert pool(B, N, P0, c, ostride) == _lib.RAJNI_EINVAL, (B, N, P0, c, ostride)
        assert b"rajni_mean_pool_layernorm_f32" in lib.rajni_last_error()
    torch.cuda.synchronize()
    # through ops: the output dtype and the row statistics, which describe a stored bf16 row
    with pytest.raises(RajniError, match="multiple of 64"):
        ops.mean_pool_layernorm(_rows(2, 17, 96, 0), 2, 17, 96, *_affine(96, 0), 1e-6, out=torch.empty(2, 96, device="cuda"))
    with pytest.raises(ValueError, match="bf16 or fp32"):
        ops.layernorm(x, gamma, beta, 1e-6, 4, C, in_row_stride=17 * C, out=torch.empty(4, C, device="cuda", dtype=torch.float16))
    with pytest.raises(ValueError, match="bf16 or fp32"):
        ops.mean_pool_layernorm(x, 4, 17, C, gamma, beta, 1e-6, out=torch.empty(4, C, device="cuda", dtype=torch.float16))
    st = torch.zeros(ops.row_stats_slots(C), 4, 2, device="cuda")
    with pytest.raises(ValueError, match="must be bf16"):
        ops.layernorm(x, gamma, beta, 1e-6, 4, C, out=torch.empty(4, C, device="cuda"), row_stats=st, stats_slots=st.shape[0])


# ------------------------------------------------------------------ the bridge to the classifier path
def _identity_head(base):
    C = base.embed_dim
    m = copy.deepcopy(base)
    m.head = nn.Linear(C, C)
    with torch.no_grad():
        m.head.weight.copy_(torch.eye(C))
        m.head.bias.zero_()
    return m


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip",
                                  "vit_base_patch16_224_dino"])
@pytest.mark.parametrize("sched", ["dense", "pruned"])
def test_features_are_the_identity_heads_operand(pkg, name, sched):
    """head = Linear(C, C) with weight I and bias 0: each logit is one exact product, so the logits are the head GEMM's bf16
    operand.  That operand is the bf16 rounding of the headless features, bit for bit."""
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0, num_classes=0), seed=1)
    size = base.patch_embed.img_size[0]
    s = {} if sched == "dense" else (MICRO_SCHEDULE if "micro" in name else README_SCHEDULE)
    images = make_images(8, size, 21).cuda()
    feats = pkg.RAJNIViTWrapper(copy.deepcopy(base), s).cuda().eval()(images)
    classifier = pkg.RAJNIViTWrapper(_identity_head(base), s).cuda().eval()
    logits = classifier(images)
    assert feats.dtype == torch.float32 and feats.shape == (8, base.embed_dim)
    assert torch.equal(logits, feats.to(torch.bfloat16).float())
    assert not torch.equal(feats, logits)                 # the features are not rounded to bf16


# ------------------------------------------------------------------ the wrapper end to end
def _forward_vs_oracle(pkg, base, sched, images, tol, band):
    """The features against the headless reference, selection teacher-forced: max |dfeature| < ``tol`` times the
    reference features' std, every image's cosine similarity above 0.999, token counts exact, and every kept-set
    disagreement inside a ``band`` tie band.  The kept-set overlap must also exceed 0.97 above 64 tokens; at or below
    64 tokens a block keeps only a handful of tokens per image, so one legitimate near-tie swap already costs several
    percent of the overlap, and only the tie band applies there (as for the tie-band fraction)."""
    params = horc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, sched).cuda().eval()
    feats = model(images.cuda()).cpu()
    ours = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
    trace = []
    ref, stats = horc.forward(params, images, sched, trace=trace, forced_keep=ours)
    assert model.get_last_stats() == stats
    assert feats.dtype == torch.float32 and feats.shape == ref.shape and torch.isfinite(feats).all()
    err, std = (feats - ref).abs().max().item(), ref.std().item()
    cos = F.cosine_similarity(feats.double(), ref.double(), dim=1)
    print(f"(selection teacher-forced): max |dfeature| {err:.4f} ({err / std:.4f} std), feature std {std:.3f}, "
          f"min cosine {cos.min().item():.6f}")
    assert err < tol * std
    assert cos.min().item() > 0.999
    for rec, kidx in zip(trace, ours):
        if kidx is None:
            continue
        ov, worst, frac = _near_tie_mismatch(kidx, rec["scores"], kidx.shape[1] - 1, 1, band)
        print(f"  block {rec['block']}: kept-set overlap {ov:.4f}, worst disagreeing token {worst:.2e} from the cut")
        assert worst < band
        assert (ov > 0.97 and frac < 0.12) or rec["scores"].shape[1] <= 64, (frac, ov)
    return model, feats


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip"])
@pytest.mark.parametrize("sched", ["dense", "micro"])
def test_trained_like_micro_models_vs_oracle(pkg, name, sched):
    """Trained-like statistics (spread norm gains and shifts, massive-activation channels), the tie band of
    test_gpu_pool_prenorm.test_trained_like_micro_models_vs_oracle.  Features within 0.05 std: the tolerance of the
    classifier tests scaled from logits to features; on a B200 these models measure 0.012-0.026 std."""
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0, num_classes=0), seed=1)
    _forward_vs_oracle(pkg, base, MICRO_SCHEDULE if sched == "micro" else {}, make_images(8, 64, 99), 0.05, 0.06)


@pytest.mark.parametrize("name,batch", [("vit_small_patch16_224_dino", 16), ("vit_base_patch8_224_dino", 4)])
@pytest.mark.parametrize("sched", ["dense", "readme"])
def test_full_models_vs_oracle(pkg, name, batch, sched):
    """Full DINO backbones at the tie band of test_gpu_pool_prenorm.test_forward_vs_oracle_full_models (3 %).  ViT-B/8 has
    785 tokens: its scores take the workspace path and its attention the long-sequence kernel.  Features within 0.05 std
    (measured on a B200: 0.036-0.041 std)."""
    from rajni_vit_b200 import ops
    from rajni_vit_b200 import schedule as S
    from rajni_vit_b200.vit import VIT_PATCH, create_model
    s = README_SCHEDULE if sched == "readme" else {}
    base = create_model(name, seed=0)
    tokens = (224 // VIT_PATCH[name]) ** 2 + 1
    if tokens > 256:
        assert ops.needs_score_workspace(tokens, base.blocks[0].attn.num_heads) and tokens > ops.LONG_SEQ
    model, _ = _forward_vs_oracle(pkg, base, s, make_images(batch, 224, 1234), 0.05, 0.03)
    assert model.get_last_stats()["token_counts"] == S.token_counts(s, 12, tokens)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_dino", "vit_micro_patch16_64_mae"])
def test_graph_replay_uint8_input_and_batch_independence(pkg, name):
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    model = pkg.RAJNIViTWrapper(randomize_trained_like(create_model(name, seed=0, num_classes=0), seed=1),
                                MICRO_SCHEDULE).cuda().eval()
    x1, x2 = make_images(4, 64, 7).cuda(), make_images(4, 64, 8).cuda()
    model.use_cuda_graph = False
    ref1, ref2 = model(x1).clone(), model(x2).clone()
    stats = model.get_last_stats()
    assert stats["token_counts"] == [17, 17, 13, 8] and ref1.dtype == torch.float32
    model.use_cuda_graph = True
    for _ in range(2):
        y1 = model(x1)
        assert torch.equal(y1, ref1) and torch.equal(model(x2), ref2)
        assert model.get_last_stats() == stats and len(model._graphs) == 1
    y1[0].fill_(0)                                         # a replay's output is the caller's: the next replay is unaffected
    assert torch.equal(model(x1), ref1)
    # one image's features, whatever batch it is in
    model.use_cuda_graph = False
    assert torch.equal(model(x1[2:3].contiguous()), ref1[2:3])
    assert torch.equal(model(torch.cat([x2, x1])), torch.cat([ref2, ref1]))
    # bf16 input: fp32 features cast to the input's dtype, as logits are
    assert model(x1.bfloat16()).dtype == torch.bfloat16
    g = torch.Generator().manual_seed(3)
    u8 = torch.randint(0, 256, (4, 3, 64, 64), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(MEAN), torch.tensor(STD)
    xf = u8.float().div(255).sub(mean[None, :, None, None]).div(std[None, :, None, None])
    ref = model(xf.cuda()).clone()
    model.set_input_normalization(MEAN, STD)
    got = model(u8.cuda())
    assert got.dtype == torch.float32 and torch.equal(got, ref)
    model.use_cuda_graph = True
    assert torch.equal(model(u8.cuda()), ref)


@pytest.mark.parametrize("name,num_classes,launches", [("vit_base_patch16_224_dino", None, 67), ("vit_base_patch16_224_mae", 0, 67),
                                                       ("vit_base_patch16_clip_224", 0, 68)])
def test_launches_per_step(pkg, name, num_classes, launches):
    """No head GEMM: 67 launches a step with class-token or average pooling (68 - 1), 68 with norm_pre.  160 images: above
    SPLIT_SCORE_MAX_BATCH, so each score/select is one launch, as in C2."""
    from rajni_vit_b200 import _lib
    from rajni_vit_b200.vit import create_model
    model = pkg.RAJNIViTWrapper(create_model(name, seed=0, num_classes=num_classes), README_SCHEDULE).cuda().eval()
    model.use_cuda_graph = False
    x = make_images(160, 224, 1).cuda()
    model(x)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    y = model(x)
    torch.cuda.synchronize()
    assert _lib.launch_count() - before == launches
    assert y.shape == (160, 768) and y.dtype == torch.float32
