"""Throughput of the DeiT families against ViT-B/16 on one B200, and the cost of the score/select prefix parameter.

    python tools/deit_bench.py [--batch 256] [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

1. vit_base_patch16_224, deit3_base_patch16_224 and deit_base_distilled_patch16_224 (random-init stand-ins, fp32 images
   already on the device), dense and with the README schedule, alternating model by model within each round so that
   clock and neighbour noise spread over all of them.  img/s from CUDA events around `steps` forwards after `warmup`.
   DeiT-III runs the same kernels at the same shapes as ViT-B/16 (LayerScale is folded into the proj / fc2 weights); the
   distilled model has one more token in every block and a K = 2C head.
2. score_select (the one-launch kernel: B > 148) at B images of 197 tokens with one prefix token and 198 tokens with two,
   plus 198 tokens with one, so the prefix parameter is compared at the same shape too.  Median of CUDA-event timings of
   `inner` back-to-back launches, L2 flushed before each group.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="also write the report to this file")
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say(f"# card (name, power.limit, clocks.max.sm): {card()}")
    say(f"# batch {args.batch}, {args.steps} timed forwards after {args.warmup} per measurement, {args.rounds} rounds")
    B = args.batch
    x = torch.randn(B, 3, 224, 224, device="cuda")
    runs = {}
    for name in MODELS:
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
        base = statistics.median(res[(MODELS[0], label)])
        for name in MODELS[1:]:
            say(f"{label}: {name} / {MODELS[0]} = {statistics.median(res[(name, label)]) / base:.4f}")

    say("## score_select, one-launch kernel, B = %d, 12 heads (us, median)" % B)
    for N, prefix in ((197, 1), (198, 2), (198, 1)):
        g = torch.Generator(device="cuda").manual_seed(N)
        qkv = torch.randn(B, N, 3 * 768, device="cuda", generator=g).to(torch.bfloat16)
        keep = max(1, int(0.88 * (N - prefix)))
        out = ops.score_select(qkv, 12, keep, split=False, prefix=prefix)
        t = time_kernel(lambda: ops.score_select(qkv, 12, keep, split=False, prefix=prefix, keep_idx=out[1],
                                                 next_scores=out[2], row_map=out[3]))
        say(f"N={N} prefix={prefix} keep={keep}: {t:8.2f} us")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
