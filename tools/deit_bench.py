"""Throughput of the DeiT families against ViT-B/16 on one B200, and the cost of the score/select prefix parameter.

    python tools/deit_bench.py [--batch 256] [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]
                               [--models A,B,...] [--kernels]

1. vit_base_patch16_224, deit3_base_patch16_224 and deit_base_distilled_patch16_224 (random-init stand-ins, fp32 images
   already on the device), dense and with the README schedule, alternating model by model within each round so that
   clock and neighbour noise spread over all of them.  img/s from CUDA events around `steps` forwards after `warmup`.
   DeiT-III runs the same kernels at the same shapes as ViT-B/16 (LayerScale is folded into the proj / fc2 weights); the
   distilled model has one more token in every block and a K = 2C head.
2. score_select (the one-launch kernel: B > 148) at B images of 197 tokens with one prefix token and 198 tokens with two,
   plus 198 tokens with one, so the prefix parameter is compared at the same shape too.  Median of CUDA-event timings of
   `inner` back-to-back launches, L2 flushed before each group.
``--models``: the comma-separated stand-ins to compare in section 1 instead (the first one is the baseline of the ratios),
e.g. ``vit_base_patch16_224,vit_base_patch16_224_mae,vit_base_patch16_clip_224`` for the average-pooled and pre-norm models.
3. ``--kernels``: the two kernels of those models in isolation - the pooled head (mean of the patch rows + fc_norm) and the
   LayerNorm pass that also writes row statistics (norm_pre) - at ViT-B/16 shapes (197 tokens, C = 768) for 256 and 8
   images, and the final LayerNorm on the class-token rows and the pooled head with bf16 and with fp32 rows out (fp32: a
   headless model's features).  Each launch timed alone with CUDA events after a 256 MB write has flushed L2; median over the launches.
   Achieved bytes/s are the bytes each kernel must move (rows read, rows and statistics written) over that time, and
   are also given as a share of the 6.45 TB/s a device-to-device copy reaches on a B200.
The card name and power limit are read in the same run and printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rajni_vit_b200 import RAJNIViTWrapper, ops  # noqa: E402
from rajni_vit_b200.vit import create_model  # noqa: E402

README_SCHEDULE = {3: {"keep_ratio": 0.88}, 4: {"keep_ratio": 0.88}, 7: {"keep_ratio": 0.8}, 8: {"keep_ratio": 0.72}}
MODELS = ["vit_base_patch16_224", "deit3_base_patch16_224", "deit_base_distilled_patch16_224"]


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # the numbers below still stand, without the card's settings beside them
        return f"(nvidia-smi unavailable: {e})"


def time_forward(model, x, steps, warmup) -> float:
    for _ in range(warmup):
        model(x)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        model(x)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def time_kernel(fn, iters=15, inner=20) -> float:
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / inner)
    return statistics.median(ts) * 1e3          # us


COPY_BYTES_PER_S = 6.45e12          # measured device-to-device copy rate of a B200 (the bound the kernels are compared to)


def time_kernel_cold(fn, iters=50) -> float:
    """Median of single-launch CUDA-event timings, L2 flushed before every launch (us)."""
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        fn()
    ev = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        ev.append((a, b))
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in ev) * 1e3


def kernel_report(say):
    C, N = 768, 197
    slots = ops.row_stats_slots(C)
    g = torch.Generator(device="cuda").manual_seed(0)
    gamma = 0.5 + torch.rand(C, device="cuda", generator=g)
    beta = 0.1 * torch.randn(C, device="cuda", generator=g)
    say("## pooled head, final LayerNorm and norm_pre kernels, C = %d, %d tokens per image, L2 flushed before each launch" % (C, N))
    for B in (256, 8):
        x = torch.randn(B * N, C, device="cuda", generator=g).to(torch.bfloat16)
        out = torch.empty(B, C, device="cuda", dtype=torch.bfloat16)
        t = time_kernel_cold(lambda: ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=1, out=out))
        nbytes = B * (N - 1) * C * 2 + B * C * 2
        say(f"mean_pool_layernorm   B={B:3d}: {t:8.2f} us  {nbytes / 1e6:8.2f} MB  {nbytes / t / 1e6:7.3f} TB/s  "
            f"{nbytes / t / 1e-6 / COPY_BYTES_PER_S * 100:5.1f} % of copy")
        outf = torch.empty(B, C, device="cuda", dtype=torch.float32)
        t = time_kernel_cold(lambda: ops.mean_pool_layernorm(x, B, N, C, gamma, beta, 1e-6, prefix=1, out=outf))
        nbytes = B * (N - 1) * C * 2 + B * C * 4
        say(f"mean_pool_layernorm_f32 B={B:3d}: {t:8.2f} us  {nbytes / 1e6:8.2f} MB  {nbytes / t / 1e6:7.3f} TB/s  "
            f"{nbytes / t / 1e-6 / COPY_BYTES_PER_S * 100:5.1f} % of copy")
        for kname, o in (("layernorm (CLS rows)", out), ("layernorm_f32 (CLS rows)", outf)):
            t = time_kernel_cold(lambda: ops.layernorm(x, gamma, beta, 1e-6, B, C, in_row_stride=N * C, out=o))
            nbytes = B * C * 2 + B * C * o.element_size()
            say(f"{kname:24s} B={B:3d}: {t:8.2f} us  {nbytes / 1e6:8.2f} MB  {nbytes / t / 1e6:7.3f} TB/s")
        st = torch.empty(slots, B * N, 2, device="cuda")
        y = torch.empty_like(x)
        t = time_kernel_cold(lambda: ops.layernorm(x, gamma, beta, 1e-5, B * N, C, out=y, row_stats=st, stats_slots=slots))
        nbytes = 2 * B * N * C * 2 + B * N * slots * 8
        say(f"layernorm_row_stats   B={B:3d}: {t:8.2f} us  {nbytes / 1e6:8.2f} MB  {nbytes / t / 1e6:7.3f} TB/s  "
            f"{nbytes / t / 1e-6 / COPY_BYTES_PER_S * 100:5.1f} % of copy")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="also write the report to this file")
    ap.add_argument("--models", default=",".join(MODELS), help="comma-separated stand-ins; the first is the baseline")
    ap.add_argument("--kernels", action="store_true", help="also time the pooled-head, final LayerNorm and norm_pre kernels")
    args = ap.parse_args()
    models = args.models.split(",")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"# card (name, power.limit, clocks.max.sm): {card()}")
    say(f"# batch {args.batch}, {args.steps} timed forwards after {args.warmup} per measurement, {args.rounds} rounds")
    B = args.batch
    x = torch.randn(B, 3, 224, 224, device="cuda")
    runs = {}
    for name in models:
        for label, sched in (("dense", {}), ("readme", README_SCHEDULE)):
            runs[(name, label)] = RAJNIViTWrapper(create_model(name, seed=0), sched).cuda().eval()
    res = {k: [] for k in runs}
    counts = {}
    for r in range(args.rounds):
        for k, model in runs.items():
            ms = time_forward(model, x, args.steps, args.warmup)
            res[k].append(B / ms * 1e3)
            counts[k] = model.get_last_stats()["token_counts"]
    say("## img/s per round (higher is better)")
    for (name, label), v in res.items():
        say(f"{name:34s} {label:6s} " + "  ".join(f"{i:9.1f}" for i in v) +
            f"   median {statistics.median(v):9.1f}   tokens {counts[(name, label)]}")
    for label in ("dense", "readme"):
        base = statistics.median(res[(models[0], label)])
        for name in models[1:]:
            say(f"{label}: {name} / {models[0]} = {statistics.median(res[(name, label)]) / base:.4f}")

    say("## score_select, one-launch kernel, B = %d, 12 heads (us, median)" % B)
    for N, prefix in ((197, 1), (198, 2), (198, 1)):
        g = torch.Generator(device="cuda").manual_seed(N)
        qkv = torch.randn(B, N, 3 * 768, device="cuda", generator=g).to(torch.bfloat16)
        keep = max(1, int(0.88 * (N - prefix)))
        out = ops.score_select(qkv, 12, keep, split=False, prefix=prefix)
        t = time_kernel(lambda: ops.score_select(qkv, 12, keep, split=False, prefix=prefix, keep_idx=out[1],
                                                 next_scores=out[2], row_map=out[3]))
        say(f"N={N} prefix={prefix} keep={keep}: {t:8.2f} us")
    if args.kernels:
        kernel_report(say)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
