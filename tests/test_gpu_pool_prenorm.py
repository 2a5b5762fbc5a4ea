"""Average-pooled heads (global_pool='avg' with fc_norm) and the pre-norm stem (norm_pre) on the B200: the pooling kernel
and the LayerNorm pass that emits row statistics against fp64 torch, and the wrapper end to end against the reference
(tests/pool_prenorm_oracle.py), with graph replay, uint8 pixels, batch independence and the launch count."""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests import pool_prenorm_oracle as porc
from tests.cases import MICRO_SCHEDULE, README_SCHEDULE, make_images
from tests.test_gpu_deit import MEAN, STD, _near_tie_mismatch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from rajni_vit_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def pkg():
    import rajni_vit_b200
    return rajni_vit_b200


def _affine(C, seed):
    g = torch.Generator().manual_seed(seed)
    return (0.5 + 1.5 * torch.rand(C, generator=g)).cuda(), (0.3 * torch.randn(C, generator=g)).cuda()


def _rows(B, N, C, seed):
    """bf16 rows with a per-channel offset, so that the LayerNorm's mean subtraction matters."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    off = 2.0 * torch.randn(C, device="cuda", generator=g)
    return (torch.randn(B * N, C, device="cuda", generator=g) + off).to(torch.bfloat16)


def _pool_ref(x, B, N, P0, gamma, beta, eps):
    """fp64 on the same bf16 rows; also |gamma| + |beta|, the scale of the fp32 rounding of a normalised value."""
    C = x.shape[1]
    m = x.view(B, N, C)[:, P0:].double().mean(1)
    z = (m - m.mean(1, keepdim=True)) / torch.sqrt(m.var(1, unbiased=False, keepdim=True) + eps)
    y = z * gamma.double() + beta.double()
    return y, (gamma.double().abs() + beta.double().abs()).expand_as(y)


def _within_one_ulp(got, ref, scale):
    """|got - ref| <= one bf16 ulp of ref, plus 1e-5 of the output's scale for fp32 rounding (a normalised value is off by
    ~1e-7 absolute in fp32, which outweighs a bf16 ulp only where the output is ~0)."""
    ulp = torch.exp2(torch.floor(torch.log2(ref.abs().clamp_min(1e-30))) - 7)
    err = (got.double() - ref).abs()
    bad = err > ulp + 1e-5 * scale
    assert not bad.any(), (err[bad][:4], ref[bad][:4])


@pytest.mark.parametrize("N", [17, 50, 88, 197, 785])
@pytest.mark.parametrize("P0", [1, 2])
def test_mean_pool_layernorm_against_fp64(ops, N, P0):
    for C in (128, 384, 768, 1024):
        gamma, beta = _affine(C, C + N)
        x = _rows(256, N, C, N * 7 + C + P0)
        for B in (1, 3, 256):
            xb = x[: B * N].contiguous()
            y = ops.mean_pool_layernorm(xb, B, N, C, gamma, beta, 1e-6, prefix=P0)
            ref, scale = _pool_ref(xb, B, N, P0, gamma, beta, 1e-6)
            _within_one_ulp(y, ref, scale)
            if B == 256:
                full = y
        # an image's row is the same bits in any batch
        for b in (0, 1, 200, 255):
            one = ops.mean_pool_layernorm(x[b * N: (b + 1) * N].contiguous(), 1, N, C, gamma, beta, 1e-6, prefix=P0)
            assert torch.equal(one[0], full[b]), (C, b)


def test_mean_pool_layernorm_strided_output(ops):
    B, N, C, P0 = 5, 197, 768, 1
    gamma, beta = _affine(C, 1)
    x = _rows(B, N, C, 2)
    out = torch.full((B, 3 * C), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=P0, out=out, out_row_stride=3 * C)
    assert torch.isnan(out[:, C:].float()).all()
    assert torch.equal(out[:, :C], ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=P0))


def test_mean_pool_layernorm_refuses_bad_shapes(ops):
    from rajni_vit_b200._lib import RajniError
    gamma, beta = _affine(96, 0)
    with pytest.raises(RajniError, match="multiple of 64"):
        ops.mean_pool_layernorm(_rows(2, 17, 96, 0), 2, 17, 96, gamma, beta, 1e-6)
    with pytest.raises(ValueError, match="prefix"):
        ops.mean_pool_layernorm(_rows(2, 17, 128, 0), 2, 17, 128, *_affine(128, 0), 1e-6, prefix=3)


@pytest.mark.parametrize("rows,C", [(256 * 197, 768), (8 * 197, 768), (3 * 17, 128), (64 * 50, 1024), (7, 2048)])
def test_layernorm_row_stats(ops, rows, C):
    gamma, beta = _affine(C, rows)
    x = _rows(rows, 1, C, C + rows)
    slots = ops.row_stats_slots(C)
    st = torch.full((slots, rows + 3, 2), 7.0, device="cuda")
    y = ops.layernorm(x, gamma, beta, 1e-5, rows, C, row_stats=st, stats_slots=slots)
    ref = F.layer_norm(x.float(), (C,), gamma, beta, 1e-5)
    torch.testing.assert_close(y.float(), ref, rtol=2 ** -7, atol=1e-2)
    # slot 0 = fp32 sums of the stored bf16 row; within 1e-6 relative of fp64 (of the sum of |v| where the sum cancels)
    v = y.double()
    for got, want, mag in ((st[0, :rows, 0], v.sum(1), v.abs().sum(1)), (st[0, :rows, 1], (v * v).sum(1), (v * v).sum(1))):
        assert ((got.double() - want).abs() <= 1e-6 * mag).all()
    assert (st[1:, :rows] == 0).all() and (st[:, rows:] == 7.0).all()
    # in place: the same bits
    st2 = torch.zeros_like(st)
    xi = x.clone()
    ops.layernorm(xi, gamma, beta, 1e-5, rows, C, out=xi, row_stats=st2, stats_slots=slots)
    assert torch.equal(xi, y) and torch.equal(st2[:, :rows], st[:, :rows])
    # without row_stats the existing kernel runs: same outputs
    assert torch.equal(ops.layernorm(x, gamma, beta, 1e-5, rows, C), y)


# ------------------------------------------------------------------ the wrapper end to end
def _forward_vs_oracle(pkg, base, sched, images, logit_tol, band):
    """test_gpu_deit._forward_vs_oracle against the pooled / pre-norm reference: selection teacher-forced, logits within
    ``logit_tol(std)``, top-1 equal where decided, kept sets exact outside a ``band`` tie band, token counts exact."""
    params = porc.extract_params(copy.deepcopy(base))
    model = pkg.RAJNIViTWrapper(base, sched).cuda().eval()
    logits = model(images.cuda()).cpu()
    ours = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
    trace = []
    ref, stats = porc.forward(params, images, sched, trace=trace, forced_keep=ours)
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
        ov, worst, frac = _near_tie_mismatch(kidx, rec["scores"], kidx.shape[1] - 1, 1, band)
        print(f"  block {rec['block']}: kept-set overlap {ov:.4f}, worst disagreeing token {worst:.2e} from the cut")
        assert worst < band
        assert ov > 0.97 and (frac < 0.12 or rec["scores"].shape[1] <= 64), (frac, ov)
    return model, logits


@pytest.mark.parametrize("name,batch,size", [("vit_base_patch16_224_mae", 16, 224), ("vit_base_patch16_clip_224", 16, 224),
                                             ("vit_base_patch32_clip_224", 16, 224), ("vit_base_patch16_clip_384", 4, 384)])
@pytest.mark.parametrize("sched", ["dense", "readme"])
def test_forward_vs_oracle_full_models(pkg, name, batch, size, sched):
    """At the tolerances of test_gpu_e2e.test_forward_vs_oracle_full_models (max |dlogit| < 0.08, 3 % tie band)."""
    from rajni_vit_b200 import schedule as S
    from rajni_vit_b200.vit import VIT_PATCH, create_model
    s = README_SCHEDULE if sched == "readme" else {}
    model, _ = _forward_vs_oracle(pkg, create_model(name, seed=0), s, make_images(batch, size, 1234), lambda std: 0.08, 0.03)
    tokens = (size // VIT_PATCH[name]) ** 2 + 1
    assert model.get_last_stats()["token_counts"] == S.token_counts(s, 12, tokens)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip"])
@pytest.mark.parametrize("sched", ["dense", "micro"])
def test_trained_like_micro_models_vs_oracle(pkg, name, sched):
    """Trained-like statistics (test_gpu_e2e.test_trained_like_checkpoint_end_to_end's tolerances), fc_norm / norm_pre
    gains and shifts spread too."""
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0), seed=1)
    _forward_vs_oracle(pkg, base, MICRO_SCHEDULE if sched == "micro" else {}, make_images(8, 64, 99),
                       lambda std: 0.03 * std + 0.02, 0.06)


@pytest.mark.parametrize("name", ["vit_base_patch16_224_mae", "vit_base_patch16_clip_224"])
def test_trained_like_full_models_vs_oracle(pkg, name):
    """The images and tolerances of test_gpu_e2e.test_trained_like_checkpoint_end_to_end (ViT-B/16, README schedule)."""
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    base = randomize_trained_like(create_model(name, seed=0), seed=1)
    _forward_vs_oracle(pkg, base, README_SCHEDULE, make_images(8, 224, 99), lambda std: 0.03 * std + 0.02, 0.06)


@pytest.mark.parametrize("name", ["vit_micro_patch16_64_mae", "vit_micro_patch16_64_clip"])
def test_graph_replay_and_uint8_input_are_bit_identical(pkg, name):
    from rajni_vit_b200.vit import create_model, randomize_trained_like
    model = pkg.RAJNIViTWrapper(randomize_trained_like(create_model(name, seed=0), seed=1), MICRO_SCHEDULE).cuda().eval()
    x1, x2 = make_images(4, 64, 7).cuda(), make_images(4, 64, 8).cuda()
    model.use_cuda_graph = False
    ref1, ref2 = model(x1).clone(), model(x2).clone()
    stats = model.get_last_stats()
    assert stats["token_counts"] == [17, 17, 13, 8]
    model.use_cuda_graph = True
    for _ in range(2):
        assert torch.equal(model(x1), ref1) and torch.equal(model(x2), ref2)
        assert model.get_last_stats() == stats and len(model._graphs) == 1
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


def test_pooled_logits_do_not_depend_on_the_batch(pkg):
    """MAE-B/16 with the README schedule at 256 images: a sub-batch, and a single image, reproduce their rows bit for bit."""
    from rajni_vit_b200.vit import create_model
    model = pkg.RAJNIViTWrapper(create_model("vit_base_patch16_224_mae", seed=0), README_SCHEDULE).cuda().eval()
    images = make_images(256, 224, 4321).cuda()
    y = model(images)
    assert model.get_last_stats()["token_counts"] == [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]
    assert torch.equal(model(images[64:96].contiguous()), y[64:96])
    assert torch.equal(model(images[7:8].contiguous()), y[7:8])


@pytest.mark.parametrize("name,launches", [("vit_base_patch16_224", 68), ("vit_base_patch16_224_mae", 68),
                                           ("vit_base_patch16_clip_224", 69)])
def test_launches_per_step(pkg, name, launches):
    """The pooled head replaces the class-token LayerNorm (68 launches a step, as ViT-B/16); norm_pre adds one (69).  160
    images: above SPLIT_SCORE_MAX_BATCH, so each score/select is one launch, as in C2."""
    from rajni_vit_b200 import _lib
    from rajni_vit_b200.vit import create_model
    model = pkg.RAJNIViTWrapper(create_model(name, seed=0), README_SCHEDULE).cuda().eval()
    model.use_cuda_graph = False
    x = make_images(160, 224, 1).cuda()
    model(x)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    model(x)
    torch.cuda.synchronize()
    assert _lib.launch_count() - before == launches
