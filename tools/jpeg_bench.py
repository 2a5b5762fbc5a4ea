"""GPU JPEG decode against Pillow, and the end-to-end CLI pipeline with and without it, in one call.

    python tools/jpeg_bench.py --out profiles/jpeg_bench.json

Writes seeded, ImageNet-like JPEGs to a temporary directory (mostly 500x375 / 375x500, some larger; 4:2:0 with some 4:4:4
and grayscale; textured so the mean file is near ImageNet's ~128 KB) and prints, with the GPU's name and power limit and
the host's core count:
  * GPU decode-only img/s: jpeg.decode_batch on the items the loader workers hand over (bytes + parsed headers, in host
    memory), whole calls (staging, one H2D copy, the kernels, the status read), warmed, >= 1 s, at 256 images per call
    and at data.DECODE_GROUP_IMAGES per call (what GpuDecodeLoader launches); plus each kernel's time from
    torch.profiler in a separate pass;
  * Pillow decode img/s (``Image.open(f).convert("RGB")``) on all host cores;
  * end-to-end img/s of ``--gpu_decode`` against ``--gpu_preprocess``: ViT-B/16, bench.py's schedule, batch 256,
    8 loader workers, the wall clock over whole epochs of the folder (worker start-up, loading, decode, resize, forward),
    alternating, 3 rounds.
"""
from __future__ import annotations

import argparse
import io
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def make_files(root: str, n: int, seed: int = 0, first: int = 0):
    from PIL import Image
    rng = np.random.default_rng(seed)
    sizes = []
    for i in range(first, first + n):
        r = rng.random()
        h, w = (375, 500) if r < 0.45 else (500, 375) if r < 0.9 else (int(rng.integers(600, 1100)), int(rng.integers(600, 1100)))
        y, x = np.mgrid[0:h, 0:w]
        f1, f2 = rng.uniform(3, 12, 2)
        a = np.stack([(x * f1 / 4 + y) % 256, np.sin(x / f1) * 100 + 128, np.cos(y / f2) * 90 + (x % 64)], axis=2)
        a = np.clip(a + rng.normal(0, 26, (h, w, 3)), 0, 255).astype(np.uint8)
        im = Image.fromarray(a)
        kind = rng.random()
        kw = dict(quality=int(rng.integers(85, 96)), subsampling=2)
        if kind < 0.1:
            kw["subsampling"] = 0
        elif kind < 0.15:
            im = im.convert("L")
        d = os.path.join(root, f"n{i % 10:08d}")
        os.makedirs(d, exist_ok=True)
        p = os.path.join(d, f"img_{i:05d}.JPEG")
        im.save(p, "JPEG", **kw)
        sizes.append(os.path.getsize(p))
    return sizes


def _pil_decode(path):
    from PIL import Image
    with Image.open(path) as im:
        return np.asarray(im.convert("RGB")).shape[0]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception as e:                                   # noqa: BLE001 - reported, not hidden
        name, power = f"unknown ({e})", "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=6144)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    import torch
    from rajni_vit_b200 import data, jpeg, run
    from bench import SCHEDULE
    assert torch.cuda.is_available(), "this benchmark measures the GPU; there is no CPU mode"
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, host_cores=os.cpu_count(), files=args.files, batch=args.batch)
    with tempfile.TemporaryDirectory() as root:
        with mp.get_context("fork").Pool(os.cpu_count()) as pool:          # seeded per chunk, same files on every box
            chunk = 256
            sizes = sum(pool.starmap(make_files, [(root, min(chunk, args.files - i), i, i)
                                                   for i in range(0, args.files, chunk)]), [])
        res["mean_file_kb"] = round(float(np.mean(sizes)) / 1024, 1)
        print(f"{args.files} files, mean {res['mean_file_kb']} KB; {name}, power limit {power}, {os.cpu_count()} host cores", flush=True)
        paths = sorted(os.path.join(dp, f) for dp, _, fs in os.walk(root) for f in fs)
        blobs = [open(p, "rb").read() for p in paths]
        # ---- GPU decode only, on the loader workers' items
        items = [jpeg.read_file(b) for b in blobs]

        def rate(per_call):
            calls = [items[i:i + per_call] for i in range(0, len(items) - per_call + 1, per_call)]
            jpeg.decode_batch(calls[0], "cuda")
            torch.cuda.synchronize()
            n, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < 1.0 or n < 2 * per_call:
                for c in calls:
                    jpeg.decode_batch(c, "cuda")                 # ends in the status read, which synchronises
                    n += len(c)
            return round(n / (time.perf_counter() - t0), 1)

        res["gpu_decode_img_s"] = {str(args.batch): rate(args.batch), str(data.DECODE_GROUP_IMAGES): rate(data.DECODE_GROUP_IMAGES)}
        from torch.profiler import ProfilerActivity, profile
        group = items[:data.DECODE_GROUP_IMAGES]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            jpeg.decode_batch(group, "cuda")
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        jpeg.decode_batch(group, "cuda")
        res["decode_call_ms"] = {"images": len(group), "wall": round((time.perf_counter() - t0) * 1e3, 2)}
        for ev in prof.key_averages():
            if "jpeg_" in ev.key:
                res["decode_call_ms"][ev.key.split("(")[0].split("::")[-1]] = round(ev.device_time_total / 1e3, 2)
        print(f"GPU decode: {res['gpu_decode_img_s']} img/s per call size; one call of {len(group)} images: "
              f"{res['decode_call_ms']} ms", flush=True)
        # ---- Pillow on all host cores
        with mp.get_context("fork").Pool(os.cpu_count()) as pool:
            pool.map(_pil_decode, paths[:64])
            t0 = time.perf_counter()
            pool.map(_pil_decode, paths, chunksize=8)
            res["pillow_img_s_all_cores"] = round(len(paths) / (time.perf_counter() - t0), 1)
        print(f"Pillow decode: {res['pillow_img_s_all_cores']} img/s on {os.cpu_count()} cores", flush=True)
        # ---- end to end through the CLI's loaders: run.build_loader as `run.py --gpu_decode / --gpu_preprocess` builds it
        from rajni_vit_b200 import RAJNIViTWrapper
        from rajni_vit_b200.vit import create_model
        model = RAJNIViTWrapper(create_model("vit_base_patch16_224", seed=0), SCHEDULE).cuda().eval()
        model.set_input_normalization(run.IMAGENET_MEAN, run.IMAGENET_STD)

        def epoch(flag):
            a = run.get_args(["--data_path", root, "--schedule", "unused", "--batch_size", str(args.batch),
                              "--num_workers", str(args.workers), flag])
            loader = run.build_loader(a, 224)
            n, t0 = 0, time.perf_counter()
            with torch.no_grad():
                for images, _ in loader:
                    model(images)
                    n += images.shape[0]
            torch.cuda.synchronize()
            return n / (time.perf_counter() - t0)

        epoch("--gpu_decode")
        epoch("--gpu_preprocess")                                 # warm both arms (modules, allocator, page cache)
        e2e = {"--gpu_decode": [], "--gpu_preprocess": []}
        for r in range(args.rounds):
            for flag in ("--gpu_decode", "--gpu_preprocess") if r % 2 == 0 else ("--gpu_preprocess", "--gpu_decode"):
                e2e[flag].append(round(epoch(flag), 1))
                print(f"round {r} {flag}: {e2e[flag][-1]} img/s", flush=True)
        res["e2e_img_s"] = {k.lstrip("-"): v for k, v in e2e.items()}
        res["e2e_median_img_s"] = {k.lstrip("-"): float(np.median(v)) for k, v in e2e.items()}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return res


if __name__ == "__main__":
    main()
