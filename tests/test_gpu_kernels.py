"""Per-kernel parity on the B200: each C-ABI entry point against the CPU oracle
(oracle/rajni_oracle.py) or a plain torch fp32 restatement, on identical bf16-rounded inputs.

Tolerances (stated here once):
  * scores: rtol 2e-5 (fp32 arithmetic on both sides, different summation order);
  * kept-token indices: bit-exact (rows whose cut is decided by a gap below 1e-5 relative are
    compared as sets against the kernel's own scores instead — SURVEY.md 4.7);
  * bf16 outputs (GEMM, LayerNorm, attention): |err| <= 2^-7 * |ref| + atol  (one bf16 ulp is 2^-8).
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import rajni_oracle as orc
from tests.cases import IMPORTANCE_CASES, SELECT_CASES, bf16_round, make_qkv, make_scores, npz
from tests.conftest import GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

BF16_RTOL = 2.0 ** -7


@pytest.fixture(scope="module")
def ops():
    from rajni_vit_b200 import ops as _ops
    return _ops


def dev(t, dtype=None):
    return t.to("cuda", dtype) if dtype is not None else t.to("cuda")


def report(name, got, ref):
    err = (got - ref).abs()
    print(f"[{name}] max_abs={err.max().item():.3e} max_rel={(err / ref.abs().clamp_min(1e-6)).max().item():.3e} "
          f"ref_rms={ref.pow(2).mean().sqrt().item():.3e}")


# ------------------------------------------------------------------ a1 importance
@pytest.mark.parametrize("name", list(IMPORTANCE_CASES))
def test_importance(ops, name):
    B, N, H, D, seed = IMPORTANCE_CASES[name]
    if D != 64:
        pytest.skip("kernel is specialised for head dim 64")
    qkv = make_qkv(B, N, H, D, seed)
    ref = orc.importance(qkv.double(), H)
    got = ops.importance(dev(qkv, torch.bfloat16), H).cpu()
    report(name, got.double(), ref)
    torch.testing.assert_close(got.double(), ref, rtol=2e-5, atol=1e-10)
    g = npz(f"{GOLDEN}/importance_rand.npz")
    np.testing.assert_allclose(got.numpy(), g[name + "_f64"], rtol=2e-5, atol=1e-10)   # the reference's own output


def test_importance_full_size(ops):
    """BASELINE config 2 block-3 shape; properties that need no oracle run: rows of A_cls sum to one."""
    B, N, H = 256, 197, 12
    g = torch.Generator().manual_seed(5)
    qkv = torch.randn(B, N, 3 * H * 64, generator=g).to(torch.bfloat16)
    s = ops.importance(dev(qkv), H).cpu()
    assert torch.isfinite(s).all() and (s > 0).all()
    ref = orc.importance(qkv[:4].float(), H)
    torch.testing.assert_close(s[:4], ref, rtol=3e-5, atol=1e-10)
    # score = A_cls * z with z in (0,1): so sum_n score < 1 and scale-free in B
    assert (s.sum(dim=1) < 1).all()
    s2 = ops.importance(dev(qkv[100:104].contiguous()), H).cpu()
    assert torch.equal(s2, s[100:104])          # images are independent and the kernel is deterministic


# ------------------------------------------------------------------ a2 select
@pytest.mark.parametrize("name", list(SELECT_CASES))
def test_select(ops, name):
    B, N, ratio, seed = SELECT_CASES[name]
    scores = make_scores(B, N, seed)
    keep = orc.keep_count(N, ratio)
    idx, nxt, rmap = ops.select(dev(scores), keep)
    ref = orc.select(scores, keep)
    assert torch.equal(idx.cpu().long(), ref)
    assert torch.equal(nxt.cpu(), torch.gather(scores, 1, ref))
    assert torch.equal(rmap.cpu().long().view(B, -1), ref + torch.arange(B)[:, None] * N)
    np.testing.assert_array_equal(idx.cpu().numpy(), npz(f"{GOLDEN}/select_cases.npz")[name + "_idx"])


def test_select_ties_and_errors(ops):
    from rajni_vit_b200._lib import RajniError
    s = torch.tensor([[9.0, 1.0, 2.0, 2.0, 2.0, 0.0, 2.0],
                      [0.0, 5.0, 5.0, 5.0, 5.0, 5.0, 5.0],
                      [0.0, -1.0, -2.0, 3.0, float("inf"), -0.0, 0.0]])
    for keep in range(1, 7):
        idx, _, _ = ops.select(dev(s), keep)
        assert torch.equal(idx.cpu().long(), orc.select(s, keep)), keep
    with pytest.raises(RajniError) as e:
        ops.select(dev(s), 7)
    assert "selected index k out of range" in str(e.value) and e.value.code == -4
    # all-equal rows of a realistic size
    flat = torch.full((3, 197), 0.005)
    idx, _, _ = ops.select(dev(flat), 172)
    assert torch.equal(idx.cpu().long(), torch.arange(173).expand(3, -1))


@pytest.mark.parametrize("N,ratio", [(197, 0.88), (173, 0.88), (152, 0.8), (121, 0.72), (577, 0.88), (65, 0.7)])
def test_select_random_large(ops, N, ratio):
    g = torch.Generator().manual_seed(N)
    s = torch.rand(64, N, generator=g) / N
    s[:, 5] = s[:, 9]                      # some exact ties
    s[10:20] = (s[10:20] * 64).round() / 64 / N     # heavy ties
    keep = orc.keep_count(N, ratio)
    idx, nxt, _ = ops.select(dev(s), keep)
    assert torch.equal(idx.cpu().long(), orc.select(s, keep))
    assert torch.equal(nxt.cpu(), torch.gather(s, 1, idx.cpu().long()))


@pytest.mark.parametrize("B,N,H,ratio", [(8, 197, 12, 0.88), (8, 173, 12, 0.88), (4, 197, 3, 0.95), (4, 152, 6, 0.8),
                                         (2, 577, 12, 0.88), (4, 87, 16, 0.5)])
def test_score_select_fused(ops, B, N, H, ratio):
    qkv = make_qkv(B, N, H, 64, 1000 + N + H)
    keep = orc.keep_count(N, ratio)
    scores, idx, nxt, rmap = ops.score_select(dev(qkv, torch.bfloat16), H, keep, want_scores=True)
    scores, idx, nxt = scores.cpu(), idx.cpu().long(), nxt.cpu()
    ref_scores = orc.importance(qkv.double(), H)
    torch.testing.assert_close(scores.double(), ref_scores, rtol=2e-5, atol=1e-10)
    # the select stage is exact on the kernel's own scores
    assert torch.equal(idx, orc.select(scores, keep))
    assert torch.equal(nxt, torch.gather(scores, 1, idx))
    assert torch.equal(rmap.cpu().long().view(B, -1), idx + torch.arange(B)[:, None] * N)
    # and equals the oracle's kept set wherever the cut is not decided by rounding noise
    ref_idx = orc.select(ref_scores, keep)
    srt = torch.sort(ref_scores[:, 1:], dim=1, descending=True).values
    gap = (srt[:, keep - 1] - srt[:, keep]) / srt[:, keep - 1] if keep < N - 1 else torch.ones(B, dtype=torch.float64)
    decided = gap > 1e-4
    print(f"rows decided: {int(decided.sum())}/{B}, min gap {gap.min().item():.2e}")
    assert torch.equal(idx[decided], ref_idx[decided])


# ------------------------------------------------------------------ gather / layernorm
def test_gather_rows(ops):
    g = torch.Generator().manual_seed(3)
    src = torch.randn(1000, 2304, generator=g).to(torch.bfloat16)
    rmap = torch.randint(0, 1000, (777,), generator=g, dtype=torch.int32)
    out = ops.gather_rows(dev(src), dev(rmap)).cpu()
    assert torch.equal(out, src[rmap.long()])
    src2 = torch.randn(50, 8, generator=g).to(torch.bfloat16)
    rmap2 = torch.arange(49, -1, -1, dtype=torch.int32)
    assert torch.equal(ops.gather_rows(dev(src2), dev(rmap2)).cpu(), src2.flip(0))


@pytest.mark.parametrize("rows,C", [(1, 192), (37, 192), (100, 384), (197 * 3, 768), (50, 1024), (9, 128)])
def test_layernorm(ops, rows, C):
    g = torch.Generator().manual_seed(rows + C)
    x = bf16_round(torch.randn(rows, C, generator=g) * 3 + 0.5)
    gamma = torch.randn(C, generator=g)
    beta = torch.randn(C, generator=g)
    ref = torch.nn.functional.layer_norm(x.double(), (C,), gamma.double(), beta.double(), 1e-6)
    got = ops.layernorm(dev(x, torch.bfloat16), dev(gamma), dev(beta), 1e-6, rows, C).cpu().double()
    report(f"ln{rows}x{C}", got, ref)
    assert ((got - ref).abs() <= BF16_RTOL * ref.abs() + 1e-3).all()
    # strided rows (the final norm reads CLS rows only)
    if rows >= 9:
        got2 = ops.layernorm(dev(x, torch.bfloat16), dev(gamma), dev(beta), 1e-6, rows // 3, C, in_row_stride=3 * C).cpu().double()
        assert torch.equal(got2, got[0::3][: rows // 3])


# ------------------------------------------------------------------ GEMM
GEMM_CASES = [
    # M, N, K, gelu, residual, maps, f32
    (128, 256, 64, False, False, False, False),
    (128, 256, 768, False, False, False, False),
    (256, 512, 768, False, False, False, False),
    (300, 2304, 768, False, False, False, False),      # M tail
    (788, 3072, 768, True, False, False, False),       # fc1 + GELU
    (519, 768, 3072, False, True, False, False),       # fc2 + residual
    (519, 768, 768, False, True, True, False),         # proj + gathered residual + row-remapped output
    (16, 1000, 768, False, False, False, True),        # head: N tail, fp32 out
    (100, 192, 192, False, True, False, False),        # vit_tiny widths -> 128/64-wide tiles
    (333, 576, 192, False, False, False, False),
    (64, 128, 128, True, True, False, False),
    (2000, 1024, 4096, False, True, False, False),     # vit_large fc2
    (40000, 768, 768, False, True, False, False),      # many tiles per CTA (persistent loop, phases)
]


@pytest.mark.parametrize("M,N,K,gelu,res,maps,f32", GEMM_CASES)
def test_gemm(ops, M, N, K, gelu, res, maps, f32):
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = bf16_round(torch.randn(M, K, generator=g))
    w = bf16_round(torch.randn(N, K, generator=g) / math.sqrt(K))
    bias = torch.randn(N, generator=g)
    R = M + 50
    residual = bf16_round(torch.randn(R, N, generator=g)) if res else None
    rmap = torch.randint(0, R, (M,), generator=g, dtype=torch.int32) if maps else None
    omap = torch.randperm(M + 13, generator=g)[:M].to(torch.int32) if maps else None

    A, W = dev(a, torch.bfloat16), dev(w, torch.bfloat16)
    ref = A.float() @ W.float().t() + dev(bias)
    if gelu:
        ref = torch.nn.functional.gelu(ref)
    if res:
        rr = dev(residual)
        ref = ref + (rr[dev(rmap).long()] if maps else rr[:M])
    out_rows = M + 13 if maps else M
    out = torch.zeros((out_rows, N), device="cuda", dtype=torch.float32 if f32 else torch.bfloat16)
    ops.gemm(A, W, dev(bias), M, N, K, gelu=gelu,
             residual=None if not res else dev(residual, torch.bfloat16), ldres=N,
             res_row_map=None if rmap is None else dev(rmap), out=out, ldd=N,
             out_row_map=None if omap is None else dev(omap), out_f32=f32)
    torch.cuda.synchronize()
    got = out.float()
    if maps:
        got = got[dev(omap).long()]
    report(f"gemm {M}x{N}x{K}", got, ref)
    tol = (2.0 ** -20 if f32 else BF16_RTOL) * ref.abs() + 2e-3
    bad = (got - ref).abs() > tol
    assert not bad.any(), f"{int(bad.sum())} of {bad.numel()} elements out of tolerance; first at {bad.nonzero()[0].tolist()}"


@pytest.mark.parametrize("M,C,N,gelu", [(300, 768, 2304, False), (788, 768, 3072, True), (100, 192, 576, False),
                                        (333, 384, 1536, True), (260, 1024, 3072, False), (40000, 768, 768, False)])
def test_gemm_layernorm_folded(ops, M, C, N, gelu):
    """model.py:51/59 folded into the GEMM: a producer GEMM stores x (+ per-row partial sums), the consumer runs on x
    with gamma-scaled weights.  Reference: torch LayerNorm (fp32) -> Linear (-> GELU) on the same bf16 x."""
    g = torch.Generator().manual_seed(M + C + N)
    # producer: x = a @ w0^T + b0 + residual  (bias+residual epilogue with ROW_STATS)
    a = bf16_round(torch.randn(M, 64, generator=g))
    w0 = bf16_round(torch.randn(C, 64, generator=g) / 8)
    b0 = torch.randn(C, generator=g) * 0.5 + 0.3
    r0 = bf16_round(torch.randn(M, C, generator=g) * 2)
    slots = ops.row_stats_slots(C)
    stats = torch.full((slots, M + 7, 2), float("nan"), device="cuda")
    x = ops.gemm(dev(a, torch.bfloat16), dev(w0, torch.bfloat16), dev(b0), M, C, 64,
                 residual=dev(r0, torch.bfloat16), ldres=C, row_stats=stats)
    torch.cuda.synchronize()
    xf = x.float()
    tot = stats[:, :M].sum(dim=0).double()
    torch.testing.assert_close(tot[:, 0], xf.double().sum(dim=1), rtol=1e-5, atol=1e-3)
    torch.testing.assert_close(tot[:, 1], (xf.double() ** 2).sum(dim=1), rtol=1e-5, atol=1e-3)
    assert torch.isnan(stats[:, M:]).all()          # rows past M are never written
    # consumer
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.2
    w = bf16_round(torch.randn(N, C, generator=g) / math.sqrt(C))
    bias = torch.randn(N, generator=g)
    wg = bf16_round(w * gamma[None, :])
    ref = torch.nn.functional.layer_norm(xf, (C,), dev(gamma), dev(beta), 1e-6) @ dev(wg / gamma[None, :]).t() + dev(bias)
    if gelu:
        ref = torch.nn.functional.gelu(ref)
    out = ops.gemm(x, dev(wg, torch.bfloat16), dev(bias + (wg / gamma[None, :]) @ beta), M, N, C, gelu=gelu,
                   ln=(stats, slots, dev(wg.sum(dim=1)), 1e-6))
    torch.cuda.synchronize()
    report(f"ln-gemm {M}x{N}x{C}", out.float(), ref)
    tol = BF16_RTOL * ref.abs() + 4e-3
    bad = (out.float() - ref).abs() > tol
    assert not bad.any(), f"{int(bad.sum())} of {bad.numel()} elements out of tolerance; first at {bad.nonzero()[0].tolist()}"


# Stream-K tail (gemm_tcgen05.cu): with a workspace, a long-K CTA-pair GEMM splits the leftover tiles of its last wave
# along K over the pairs and reduces fp32 partials through scratch.  Shapes: tiles % 74 pairs = 1 (the 7.01-wave case of
# 173-token blocks), 3, 26, 39 (of 74), fewer tiles than pairs (44: small shards), and vit_large's K = 4096.
SK_CASES = [
    # M, N, K, mode
    (19200, 768, 3072, "res"),        # 75 x 3 = 225 tiles = 3 waves + 3
    (22272, 768, 3072, "res"),        # 87 x 3 = 261 = 3 waves + 39
    (2784, 1024, 4096, "res"),        # 11 x 4 = 44 tiles < 74 pairs
    (6304, 768, 3072, "res"),         # 25 x 3 = 75 = 1 wave + 1
    (6304, 1024, 4096, "res"),        # vit_large fc2: 25 x 4 = 100 = 1 wave + 26
    (6304, 768, 3072, "bias"),
    (2784, 1024, 4096, "gelu"),
]


@pytest.mark.parametrize("M,N,K,mode", SK_CASES)
def test_gemm_stream_k_tail(ops, M, N, K, mode):
    g = torch.Generator().manual_seed(M + N + K)
    a = bf16_round(torch.randn(M, K, generator=g))
    w = bf16_round(torch.randn(N, K, generator=g) / math.sqrt(K))
    bias = torch.randn(N, generator=g)
    A, W, Bv = dev(a, torch.bfloat16), dev(w, torch.bfloat16), dev(bias)
    ref = A.float() @ W.float().t() + Bv
    res = None
    if mode == "gelu":
        ref = torch.nn.functional.gelu(ref)
    if mode == "res":
        res = dev(bf16_round(torch.randn(M, N, generator=g)), torch.bfloat16)
        ref = ref + res.float()
    ws = ops.gemm_workspace("cuda")
    slots = ops.row_stats_slots(N)
    flags = ops.EPI_BIAS | (ops.EPI_GELU if mode == "gelu" else 0) | ((ops.EPI_RESIDUAL | ops.EPI_ROW_STATS) if mode == "res" else 0)
    assert ops.stream_k_plan(M, N, K, flags | ops.HINT_STREAM_K)[0] > 0, "this shape is meant to take the stream-K path"

    def run(workspace, in_place):
        stats = torch.zeros((slots, M, 2), device="cuda") if mode == "res" else None
        out = res.clone() if (in_place and res is not None) else torch.zeros((M, N), device="cuda", dtype=torch.bfloat16)
        ops.gemm(A, W, Bv, M, N, K, gelu=mode == "gelu", residual=(out if in_place else res) if res is not None else None, ldres=N,
                 out=out, ldd=N, row_stats=stats, workspace=workspace, force_stream_k=True)
        torch.cuda.synchronize()
        return out, stats

    plain, plain_stats = run(None, False)
    for rep in range(3):                                   # the counters re-arm themselves: the workspace is reusable as is
        got, stats = run(ws, rep == 2)                     # (last repetition in place: residual aliases the output, like fc2)
        report(f"stream-k gemm {M}x{N}x{K} {mode} rep {rep}", got.float(), ref)
        bad = (got.float() - ref).abs() > BF16_RTOL * ref.abs() + 2e-3
        assert not bad.any(), f"{int(bad.sum())} of {bad.numel()} elements out of tolerance; first at {bad.nonzero()[0].tolist()}"
        assert int(ws[:4096].count_nonzero()) == 0, "stream-K counters were not re-armed"
        # against the unsplit kernel: same products, fp32 sums in a different order -> at most one bf16 rounding step apart
        assert ((got.float() - plain.float()).abs() <= 2.0 ** -7 * plain.float().abs() + 1e-3).all()
        if stats is not None:
            torch.testing.assert_close(stats.sum(dim=0)[:, 0].double(), got.double().sum(dim=1), rtol=1e-5, atol=1e-3)
            torch.testing.assert_close(stats.sum(dim=0)[:, 1].double(), (got.double() ** 2).sum(dim=1), rtol=1e-5, atol=1e-3)
    # deterministic: the pieces of a tile are summed in a fixed order
    again, _ = run(ws, False)
    got2, _ = run(ws, False)
    assert torch.equal(again, got2)


@pytest.mark.parametrize("ratio", [0.0, 10.0, 50.0, 100.0])
def test_layernorm_fold_statistics_at_large_mean(ops, ratio):
    """The folded LayerNorm takes the variance as E[x^2] - mean^2 from fp32 partial sums (gemm_tcgen05.cu epilogue).
    Rows whose mean is `ratio` standard deviations from zero (massive-activation rows of trained ViTs sit near 10-30)
    must still normalise correctly: reference = fp64 LayerNorm -> Linear on the same bf16 x."""
    M, C, N = 256, 768, 256
    g = torch.Generator().manual_seed(int(ratio) + 5)
    sigma = 0.5 + torch.rand(M, 1, generator=g)
    x = bf16_round(ratio * sigma * torch.sign(torch.randn(M, 1, generator=g)) + sigma * torch.randn(M, C, generator=g))
    eye = torch.eye(C)
    slots = ops.row_stats_slots(C)
    stats = torch.zeros((slots, M, 2), device="cuda")
    zero = torch.zeros(M, C)
    xd = ops.gemm(dev(x, torch.bfloat16), dev(eye, torch.bfloat16), dev(torch.zeros(C)), M, C, C,
                  residual=dev(zero, torch.bfloat16), ldres=C, row_stats=stats)          # stores x itself + its row sums
    assert torch.equal(xd.float().cpu(), x)
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.2
    w = bf16_round(torch.randn(N, C, generator=g) / math.sqrt(C))
    bias = torch.randn(N, generator=g)
    wg = bf16_round(w * gamma[None, :])
    xs = x.double()
    mean, var = xs.mean(1, keepdim=True), xs.var(1, unbiased=False, keepdim=True)
    ref = ((xs - mean) / torch.sqrt(var + 1e-6) * gamma.double() + beta.double()) @ (wg.double() / gamma.double()[None, :]).t() + bias.double()
    out = ops.gemm(xd, dev(wg, torch.bfloat16), dev(bias + (wg / gamma[None, :]) @ beta), M, N, C,
                   ln=(stats, slots, dev(wg.sum(dim=1)), 1e-6)).float().cpu().double()
    # rstd as the kernel's statistics give it, against the exact one
    tot = stats.sum(dim=0).double().cpu()
    m_k = tot[:, 0] / C
    v_k = (tot[:, 1] / C - m_k * m_k).clamp_min(0)
    rstd_err = ((1 / torch.sqrt(v_k + 1e-6)) / (1 / torch.sqrt(var[:, 0] + 1e-6)) - 1).abs().max().item()
    err = (out - ref).abs()
    print(f"[ln stats] |mean|/sigma = {ratio:5.1f}: rstd relative error {rstd_err:.2e}, max |dout| {err.max().item():.3e} (ref rms {ref.pow(2).mean().sqrt().item():.2f})")
    assert rstd_err < 5e-3
    assert (err <= BF16_RTOL * ref.abs() + 4e-3 + 4 * rstd_err * ref.abs()).all()


def test_gelu_matches_erf(ops):
    """The epilogue's GELU is a polynomial form of x*Phi(x); check it against erf over the whole useful range.
    acc = 0 (zero weights), so out[m, n] = gelu(bias[n]) exactly as the epilogue sees fp32 inputs."""
    K = 64
    a = torch.zeros(128, K)
    w = torch.zeros(256, K)
    x = torch.linspace(-9, 9, 256 * 64)
    worst = 0.0
    for i in range(64):
        xb = x[i::64].contiguous()
        out = ops.gemm(dev(a, torch.bfloat16), dev(w, torch.bfloat16), dev(xb), 128, 256, K, gelu=True, out_f32=True)
        ref = torch.nn.functional.gelu(xb.double())
        got = out[i % 128].cpu().double()
        worst = max(worst, ((got - ref).abs() / ref.abs().clamp_min(1e-3)).max().item())
        torch.testing.assert_close(got, ref, rtol=1e-4, atol=2e-6)
    print(f"gelu worst error relative to max(|ref|,1e-3): {worst:.2e}")
    # the hot bf16 epilogue (packed fp32x2 evaluation of the same fit): within one bf16 rounding of the exact value
    a2, w2 = torch.zeros(256, K), torch.zeros(256, K)
    for i in range(0, 64, 7):
        xb = x[i::64].contiguous()
        out = ops.gemm(dev(a2, torch.bfloat16), dev(w2, torch.bfloat16), dev(xb), 256, 256, K, gelu=True)
        ref = torch.nn.functional.gelu(xb.double())
        got = out[i].cpu().double()
        assert ((got - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-6).all()


def test_select_nan_sorts_largest(ops):
    """torch.topk treats NaN (either sign bit) as larger than every number: NaN-scored tokens are kept first."""
    s = make_scores(2, 33, 5)
    s[0, 7] = float("nan")
    s[1, 20] = -float("nan")
    keep = 5
    idx, _, _ = ops.select(dev(s), keep)
    assert 7 in idx[0].tolist() and 20 in idx[1].tolist()
    ref = torch.topk(s[:, 1:], keep, dim=1).indices + 1
    for b in range(2):
        assert set(idx[b, 1:].tolist()) == set(ref[b].tolist())


# ------------------------------------------------------------------ attention
@pytest.mark.parametrize("B,N,Np,H", [(2, 17, 17, 2), (3, 197, 197, 3), (2, 197, 173, 12), (2, 173, 152, 12),
                                      (2, 152, 121, 12), (2, 121, 87, 12), (1, 577, 507, 12), (2, 577, 577, 3), (1, 507, 446, 12), (3, 357, 257, 6), (2, 300, 300, 2), (1, 1000, 700, 2), (2, 64, 64, 1),
                                      (2, 65, 65, 1), (2, 197, 2, 3), (2, 250, 250, 2), (1, 300, 240, 3), (2, 256, 256, 1), (3, 130, 129, 2), (2, 192, 192, 2), (2, 200, 193, 2),
                                      # short images packed k to a tile (k divides B, k * Np <= 128): k = 8, 3, 4, 5, 2, and 3 images that cannot pack
                                      (16, 20, 14, 2), (6, 33, 33, 3), (4, 50, 23, 4), (5, 16, 16, 1), (10, 70, 58, 2), (3, 64, 64, 2), (8, 12, 11, 6),
                                      # several items per CTA (> 148 items): the second tile's rows rotate over the lane quadrants (24, 45, 64 live
                                      # rows), one-tile items alternate between the two exp-warp sets
                                      (40, 173, 152, 12), (36, 197, 173, 12), (60, 192, 192, 6), (40, 130, 129, 12), (50, 87, 87, 12), (48, 121, 87, 12)])
def test_attention(ops, B, N, Np, H):
    """Every kernel that covers the shape (include/rajni_b200.h: RAJNI_ATTN_*), not only the one the dispatcher picks."""
    from rajni_vit_b200 import _lib
    C = H * 64
    qkv = make_qkv(B, N, H, 64, 500 + N + Np)
    g = torch.Generator().manual_seed(N * Np)
    if Np < N:
        keep_idx = torch.stack([torch.cat([torch.zeros(1, dtype=torch.long),
                                           torch.sort(torch.randperm(N - 1, generator=g)[: Np - 1]).values + 1])
                                for _ in range(B)])
        rmap = (keep_idx + torch.arange(B)[:, None] * N).to(torch.int32).flatten()
        kept = torch.gather(qkv, 1, keep_idx[:, :, None].expand(-1, -1, 3 * C))
    else:
        rmap, kept = None, qkv
    ref = orc.mha(kept.double(), H, 0.125).reshape(B * Np, C)
    impls = [("auto", _lib.ATTN_AUTO)]
    if (Np + 15) // 16 * 16 <= 224:
        impls.append(("pipe", _lib.ATTN_PIPE))
    if Np <= 256:
        impls.append(("tc", _lib.ATTN_TC))
    outs = {}
    for name, impl in impls:
        for reverse in (False, True):
            got = ops.attention(dev(qkv, torch.bfloat16).view(B * N, 3 * C), None if rmap is None else dev(rmap),
                                B, N, Np, C, H, 0.125, impl=impl, reverse=reverse).cpu()
            outs[name] = got
            report(f"attn[{name}{',rev' if reverse else ''}] N={N} Np={Np}", got.double(), ref)
            assert ((got.double() - ref).abs() <= 2 * BF16_RTOL * ref.abs() + 4e-3).all(), name
    if "pipe" in outs:
        # the two short-sequence kernels take the row sum in the same order: bit-identical outputs, so a keep_ratio of 1.0
        # (gathered call) reproduces the un-pruned block (dense call) whichever kernel each call is dispatched to
        # (short images packed several to a tile by attention_tc - Np <= 64 and a divisor of B that fits - accumulate P V in
        # another order: equal to rounding, not to the bit)
        packed = Np <= 64 and any(B % k == 0 for k in range(2, 128 // Np + 1))
        if packed:
            assert (outs["pipe"].float() - outs["tc"].float()).abs().max() <= 2e-2
        else:
            assert torch.equal(outs["pipe"], outs["tc"])


def test_attention_packed_tiles_match_one_image_per_tile(ops, tmp_path):
    """Short images share a 128-row tile (block-diagonal softmax mask).  Against the same call with one image per tile the
    outputs differ only by the order of the fp32 accumulation of P V (the masked P entries are exactly 0)."""
    import subprocess
    import sys
    code = (
        "import torch, sys; sys.path.insert(0, %r)\n"
        "from rajni_vit_b200 import ops\n"
        "torch.manual_seed(5)\n"
        "B, N, Np, H = 32, 40, 26, 4; C = H * 64\n"
        "qkv = torch.randn(B * N, 3 * C, device='cuda').bfloat16()\n"
        "idx = torch.stack([torch.sort(torch.randperm(N, device='cuda')[:Np]).values for _ in range(B)])\n"
        "rmap = (idx + torch.arange(B, device='cuda')[:, None] * N).int().flatten()\n"
        "out = ops.attention(qkv, rmap, B, N, Np, C, H, 0.125)\n"
        "torch.save(out.cpu(), sys.argv[1])\n" % ROOT)
    outs = []
    for nopack in ("", "1"):
        path = str(tmp_path / f"pack_{nopack or 0}.pt")
        env = dict(os.environ)
        env.pop("RAJNI_ATTN_NOPACK", None)
        if nopack:
            env["RAJNI_ATTN_NOPACK"] = "1"
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env)
        outs.append(torch.load(path).float())
    assert torch.isfinite(outs[0]).all()
    assert (outs[0] - outs[1]).abs().max() <= 1e-2 and (outs[0] - outs[1]).abs().mean() < 1e-4


@pytest.mark.parametrize("N", [197, 130, 87, 300])
def test_attention_images_are_isolated(ops, N):
    """A NaN/Inf in one image must not reach another image's output (dense calls load per-image, zero-filled boxes)."""
    from rajni_vit_b200 import _lib
    B, H = 3, 2
    C = H * 64
    qkv = make_qkv(B, N, H, 64, 77 + N)
    clean = dev(qkv, torch.bfloat16).view(B * N, 3 * C)
    dirty = qkv.clone()
    dirty[1] = float("nan")
    dirty = dev(dirty, torch.bfloat16).view(B * N, 3 * C)
    impls = [_lib.ATTN_AUTO] + ([_lib.ATTN_PIPE, _lib.ATTN_TC] if N <= 224 else [])
    for impl in impls:
        a = ops.attention(clean, None, B, N, N, C, H, 0.125, impl=impl).view(B, N, C)
        b = ops.attention(dirty, None, B, N, N, C, H, 0.125, impl=impl).view(B, N, C)
        assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]), impl
        assert torch.isfinite(a).all()


# ------------------------------------------------------------------ patch embed
@pytest.mark.parametrize("S,C,B", [(64, 128, 3), (224, 192, 2)])
def test_patch_embed(ops, S, C, B):
    g = torch.Generator().manual_seed(S + C)
    images = torch.randn(B, 3, S, S, generator=g)
    w = bf16_round(torch.randn(C, 3, 16, 16, generator=g) / 27.7)
    bias = bf16_round(torch.randn(C, generator=g))
    P = (S // 16) ** 2
    pos = bf16_round(torch.randn(1, P + 1, C, generator=g) * 0.02)
    cls = bf16_round(torch.randn(1, 1, C, generator=g) * 0.02)
    params = dict(patch=16, pe_w=w, pe_b=bias, cls=cls, pos=pos)
    ref = orc.embed(params, bf16_round(images)).reshape(B * (P + 1), C)
    cols = torch.empty((B * P, 768), device="cuda", dtype=torch.bfloat16)
    x = torch.zeros((B * (P + 1), C), device="cuda", dtype=torch.bfloat16)
    cls_pos0 = dev((cls[0, 0] + pos[0, 0]), torch.bfloat16)
    ops.patch_im2col(dev(images), 16, cols, cls_pos0, x, C)
    unf = torch.nn.functional.unfold(bf16_round(images), 16, stride=16).transpose(1, 2).reshape(B * P, 768)
    assert torch.equal(cols.cpu().float(), unf)
    idx = torch.arange(B * P, dtype=torch.int32)
    ops.gemm(cols, dev(w.reshape(C, 768), torch.bfloat16), dev(bias), B * P, C, 768,
             residual=dev(pos[0], torch.bfloat16), ldres=C, res_row_map=dev(1 + idx % P),
             out=x, ldd=C, out_row_map=dev((idx // P) * (P + 1) + 1 + idx % P))
    got = x.cpu().float()
    report("embed", got, ref)
    assert ((got - ref).abs() <= BF16_RTOL * ref.abs() + 4e-3).all()


def test_reverse_traversal_hints_do_not_change_results(ops):
    """RAJNI_HINT_REVERSE_M / rajni_attention_fwd(reverse=1) only change the order in which tiles are visited."""
    g = torch.Generator().manual_seed(11)
    M, N, K = 3000, 768, 768
    a = dev(bf16_round(torch.randn(M, K, generator=g)), torch.bfloat16)
    w = dev(bf16_round(torch.randn(N, K, generator=g) / math.sqrt(K)), torch.bfloat16)
    bias = dev(torch.randn(N, generator=g))
    res = dev(bf16_round(torch.randn(M, N, generator=g)), torch.bfloat16)
    st0 = torch.zeros(ops.row_stats_slots(N), M, 2, device="cuda")
    st1 = torch.zeros_like(st0)
    y0 = ops.gemm(a, w, bias, M, N, K, residual=res, row_stats=st0)
    y1 = ops.gemm(a, w, bias, M, N, K, residual=res, row_stats=st1, reverse=True)
    assert torch.equal(y0, y1) and torch.equal(st0, st1)
    for B, Nt, H in ((3, 197, 3), (2, 300, 2)):
        qkv = dev(make_qkv(B, Nt, H, 64, 77), torch.bfloat16).view(B * Nt, 3 * H * 64)
        o0 = ops.attention(qkv, None, B, Nt, Nt, H * 64, H, 0.125)
        o1 = ops.attention(qkv, None, B, Nt, Nt, H * 64, H, 0.125, reverse=True)
        assert torch.equal(o0, o1)


@pytest.mark.parametrize("B,N,H,ratio", [(8, 197, 12, 0.88), (3, 577, 12, 0.88), (5, 197, 6, 0.7), (4, 197, 16, 0.9),
                                         (300, 197, 12, 0.8), (2, 33, 3, 0.5), (7, 32, 2, 0.9), (1, 2, 1, 1.0), (2, 257, 3, 0.6)])
def test_score_select_split_path_is_bit_identical(ops, B, N, H, ratio):
    """The two-launch path for small batches (rajni_score_select_split) must reproduce the fused kernel exactly."""
    qkv = dev(make_qkv(B, N, H, 64, 900 + N + H), torch.bfloat16)
    keep = max(1, min(N - 1, orc.keep_count(N, ratio)))
    s0, i0, n0, r0 = ops.score_select(qkv, H, keep, want_scores=True, split=False)
    s1, i1, n1, r1 = ops.score_select(qkv, H, keep, want_scores=True, split=True)
    assert torch.equal(s0, s1) and torch.equal(i0, i1) and torch.equal(n0, n1) and torch.equal(r0, r1)


# ------------------------------------------------------------------ f3: Resize(256, bicubic) + CenterCrop(224) on the GPU
def test_gpu_resize_center_crop_matches_torchvision(ops):
    """csrc/resize.cu against torchvision on PIL images (run.py:62-66) and against the oracle: bit-exact uint8 crops for a
    batch of frames of different sizes, portrait and landscape, up- and down-scaled."""
    np = pytest.importorskip("numpy")
    Image = pytest.importorskip("PIL.Image")
    T = pytest.importorskip("torchvision.transforms")
    from oracle.resize_oracle import resize_center_crop as oracle_resize
    from rajni_vit_b200.data import gpu_resize_center_crop, pack_frames
    sizes = [(375, 500), (500, 375), (256, 256), (224, 224), (300, 257), (257, 256), (333, 999), (480, 640), (227, 1500), (1200, 1600), (2048, 1365)]
    rng = np.random.default_rng(5)
    frames = []
    for i, (h, w) in enumerate(sizes):
        a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if i % 2:
            a = (np.cumsum(a.astype(np.int32), axis=1) // 5 % 256).astype(np.uint8)
        frames.append(torch.from_numpy(a))
    got = gpu_resize_center_crop(frames, "cuda").cpu()
    tf = T.Compose([T.Resize(256, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(224), T.PILToTensor()])
    for i, f in enumerate(frames):
        ref = tf(Image.fromarray(f.numpy()))
        assert torch.equal(got[i], ref), f"frame {i} {tuple(f.shape)}: {(got[i].int() - ref.int()).abs().max().item()} off"
        if i < 4:
            assert np.array_equal(oracle_resize(f.numpy()), ref.numpy())
    # frames the kernel cannot take are reported, not silently mangled
    buf, meta, max_h = pack_frames([frames[0]])
    with pytest.raises(ValueError, match="cannot be resized"):
        ops.resize_center_crop(buf.cuda(), meta.cuda(), max_h - 1)


def test_gpu_preprocess_loader_feeds_the_wrapper():
    """GpuPreprocessLoader + set_input_normalization reproduce the reference loader's tensors: logits from raw frames equal
    the logits from torchvision-preprocessed float images."""
    np = pytest.importorskip("numpy")
    Image = pytest.importorskip("PIL.Image")
    T = pytest.importorskip("torchvision.transforms")
    import rajni_vit_b200 as pkg
    from rajni_vit_b200 import run
    from rajni_vit_b200.data import GpuPreprocessLoader
    from rajni_vit_b200.vit import create_model
    rng = np.random.default_rng(9)
    frames = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)) for h, w in ((300, 400), (375, 500), (640, 480), (256, 300))]
    labels = torch.arange(4)
    loader = GpuPreprocessLoader([(frames, labels)], "cuda")
    tf = T.Compose([T.Resize(256, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(224), T.ToTensor(),
                    T.Normalize(mean=run.IMAGENET_MEAN, std=run.IMAGENET_STD)])
    ref_images = torch.stack([tf(Image.fromarray(f.numpy())) for f in frames])
    model = pkg.RAJNIViTWrapper(create_model("vit_tiny_patch16_224", seed=0), {3: {"keep_ratio": 0.8}}).cuda().eval()
    ref_logits = model(ref_images.cuda())
    model.set_input_normalization(run.IMAGENET_MEAN, run.IMAGENET_STD)
    (crops, lab), = list(loader)
    assert crops.dtype == torch.uint8 and crops.shape == (4, 3, 224, 224) and torch.equal(lab, labels)
    assert torch.equal(model(crops), ref_logits)
