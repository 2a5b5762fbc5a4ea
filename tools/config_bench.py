"""Images/s of the five BASELINE configs on ONE GPU at their per-GPU batch (device-resident inputs, CUDA events).
usage: python tools/config_bench.py [--eager] [name filter ...]   (--eager: no CUDA-graph replay; default: automatic)"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rajni_vit_b200 import RAJNIViTWrapper, ops  # noqa: E402
from rajni_vit_b200.vit import create_model  # noqa: E402

README = {3: {"keep_ratio": 0.88}, 4: {"keep_ratio": 0.88}, 7: {"keep_ratio": 0.8}, 8: {"keep_ratio": 0.72}}
C1 = {3: {"keep_ratio": 0.95, "update": False}, 4: {"keep_ratio": 0.95}, 5: {"keep_ratio": 0.85}, 6: {"keep_ratio": 0.85}, 7: {"keep_ratio": 0.95}}
CASES = [("C1 vit_tiny  bs8", "vit_tiny_patch16_224", C1, 8, 224),
         ("C2 vit_base  bs256", "vit_base_patch16_224", README, 256, 224),
         ("C3 vit_small bs256 (512 over 2 GPUs)", "vit_small_patch16_224", {i: {"keep_ratio": 0.7} for i in range(3, 12)}, 256, 224),
         ("C3 vit_small bs64  (512 over 8 GPUs)", "vit_small_patch16_224", {i: {"keep_ratio": 0.7} for i in range(3, 12)}, 64, 224),
         ("C4 vit_large bs32  (256 over 8 GPUs)", "vit_large_patch16_224", {i: {"keep_ratio": 0.9} for i in range(24)}, 32, 224),
         ("C5 deit_384  bs16  (128 over 8 GPUs)", "deit_base_patch16_384", README, 16, 384),
         ("B/32 vit_base_patch32 bs256 dense", "vit_base_patch32_224", {}, 256, 224),
         ("B/32 vit_base_patch32 bs256 README", "vit_base_patch32_224", README, 256, 224),
         ("B/8  vit_base_patch8  bs64  dense", "vit_base_patch8_224", {}, 64, 224),
         ("B/8  vit_base_patch8  bs64  README", "vit_base_patch8_224", README, 64, 224),
         ("B/8  vit_base_patch8  bs256 dense", "vit_base_patch8_224", {}, 256, 224),
         ("B/8  vit_base_patch8  bs256 README", "vit_base_patch8_224", README, 256, 224)]
eager = "--eager" in sys.argv
only = [a for a in sys.argv[1:] if a != "--eager"]
for name, model_name, sched, B, S in CASES:
    if only and not any(o in name for o in only):
        continue
    m = RAJNIViTWrapper(create_model(model_name, seed=0), sched).cuda().eval()
    m.use_cuda_graph = False if eager else None
    x = torch.randn(B, 3, S, S, device="cuda")
    for _ in range(5):
        m(x)
    torch.cuda.synchronize()
    n = 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        m(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    m.use_cuda_graph = False
    prof = ops.profile_steps(lambda: m(x), steps=2)
    top = sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:5]
    print(f"{name:40s} {ms:8.3f} ms/step {B / ms * 1e3:10.0f} img/s   " + "  ".join(f"{k}={v['ms']:.3f}" for k, v in top), flush=True)
    del m
