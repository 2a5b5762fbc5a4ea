"""Cost of token-level features on one B200: ``forward`` against ``forward_features`` and ``forward_intermediates(indices=4)``.

    python tools/features_bench.py [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

DINO ViT-B/16 at 224 px and batch 256, and ViT-B/8 DINO (785 tokens) at batch 64, both with the README schedule
(random-init stand-ins, fp32 images already on the device, eager launches: both batches are above the CUDA-graph limit).
The three methods alternate within each round, so that clock and neighbour noise spread over all of them; img/s from
CUDA events around ``steps`` calls after ``warmup``, median over the rounds.  ``forward_features`` adds one row gather and
one LayerNorm over all B·N0 rows in place of the class-row LayerNorm, and writes every stage's rows to a region of its
own; the extra traffic is about B·N0·C·10 bytes (gather read and write in bf16, LayerNorm read in bf16 and write in fp32),
printed beside each model.  The card name and power limit are read in the same run and printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rajni_vit_b200 import RAJNIViTWrapper  # noqa: E402
from rajni_vit_b200.vit import create_model  # noqa: E402

README_SCHEDULE = {3: {"keep_ratio": 0.88}, 4: {"keep_ratio": 0.88}, 7: {"keep_ratio": 0.8}, 8: {"keep_ratio": 0.72}}
CASES = [("vit_base_patch16_224_dino", 256), ("vit_base_patch8_224_dino", 64)]


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # the numbers below still stand, without the card's settings beside them
        return f"(nvidia-smi unavailable: {e})"


def time_calls(fn, steps, warmup) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"# card (name, power.limit, clocks.max.sm): {card()}")
    say(f"# {args.steps} timed calls after {args.warmup} per measurement, {args.rounds} rounds, README schedule, eager")
    for name, B in CASES:
        model = RAJNIViTWrapper(create_model(name, seed=0), README_SCHEDULE).cuda().eval()
        x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(0)).cuda()
        methods = {"forward": lambda: model(x), "forward_features": lambda: model.forward_features(x),
                   "forward_intermediates(4)": lambda: model.forward_intermediates(x, indices=4)}
        rates = {k: [] for k in methods}
        for _ in range(args.rounds):
            for k, fn in methods.items():
                rates[k].append(B / (time_calls(fn, args.steps, args.warmup) / 1e3))
        N0, C = model.forward_features(x).shape[1:]
        say(f"## {name}, batch {B}, {N0} tokens, C = {C}; token counts {model.get_last_stats()['token_counts']}; "
            f"gather + LayerNorm traffic ~{B * N0 * C * 10 / 1e6:.0f} MB per call")
        base = statistics.median(rates["forward"])
        for k, r in rates.items():
            med = statistics.median(r)
            say(f"{k:26s} " + " ".join(f"{v:9.1f}" for v in r) + f"   median {med:9.1f} img/s  "
                f"{B / med * 1e3:7.3f} ms/call  {med / base:6.4f} of forward")
        del model, x
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
