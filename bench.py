#!/usr/bin/env python
"""Headline benchmark: ViT-B/16 + README RAJNI schedule, batch 256 per GPU, images/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one RAJNIViTWrapper.forward over one synthetic batch (BASELINE.json configs[1]).
Prints ONE JSON line (rank 0).  Data-parallel: every rank runs the same per-GPU batch
(weak scaling), no data-path collective; the only collective is the timing reduction.

  value       images/s with the inputs already resident in HBM (CUDA events, max over ranks), exactly K steps
  sustained   the same loop run for >= 1 s (the K-step burst finishes before the 1 kW cap pulls the clock down)
  e2e         images/s through the public API from pinned HOST images: H2D copy of every batch and
              D2H read of its predictions are inside the timed region (copy/compute double-buffered)
  roofline    the dominant kernel class (the tcgen05 GEMM): algorithmic FLOPs / its CUDA-event time
  kernels     per-kernel-class CUDA-event times of separate instrumented steps (event bracketing breaks the
              programmatic-dependent-launch overlap, so their sum exceeds ms_per_step by a few %: fractions are pessimistic)
  strong      north_star's reading "the batch is sharded": the GLOBAL batch 256 split over the N ranks
  configs     BASELINE configs 3/4/5 with their global batch sharded over the N ranks (img/s, fraction of tensor roofline)
  cpu_baseline  the reference's own CPU path (oracle/_ref: the unmodified reference wrapper + evaluate_model on the
              stand-in ViT) on this box's host cores, bounded sample; falls back to the oracle port if _ref is absent
  gpu_eager_reference  the unmodified reference wrapper in eager PyTorch on THIS GPU (fp32 as shipped, and .bfloat16())
  parity      top-1 agreement and max |dlogit| of the GPU path vs the CPU oracle on 256 seeded images, and the kept-token
              sets against the oracle's own scores with the tie band (tokens within 3 % of the cut score) counted

--impl reference times the reference's CPU implementation alone (rank 0 only).
--dump-outputs DIR writes what rank 0's last timed step returned as DIR/<name>.npy (see dump_outputs), so that two builds
can be compared output for output: with the same arguments the weights and input batches are the same on every run.
It is refused with --impl reference, whose timed path (the reference's evaluate_model) returns no logits to its caller.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL = "vit_base_patch16_224"
SCHEDULE = {3: {"keep_ratio": 0.88, "update": True}, 4: {"keep_ratio": 0.88, "update": True},
            7: {"keep_ratio": 0.8, "update": True}, 8: {"keep_ratio": 0.72, "update": True}}
BATCH = 256
METRIC = "ViT-B/16 RAJNI images/sec @bs256"
WORKLOAD = f"C2: {MODEL} random-init + README schedule {{3:.88,4:.88,7:.8,8:.72}}, 224px, bf16 batch 256 per GPU"
TOKENS = [197, 197, 197, 197, 173, 152, 152, 152, 121, 87, 87, 87]
TIE_BAND = 0.03          # kept-set disagreements are legitimate only within this relative distance of the cut score
DUMP_BYTES = 64 << 20    # --dump-outputs writes at most this much in all

# BASELINE.json configs 3-5: (model, schedule, global batch, image size); SURVEY.md 8(d)
CONFIGS = {
    "C3": ("vit_small_patch16_224", {i: {"keep_ratio": 0.7, "update": True} for i in range(3, 12)}, 512, 224),
    "C4": ("vit_large_patch16_224", {i: {"keep_ratio": 0.9, "update": True} for i in range(24)}, 256, 224),
    "C5": ("deit_base_patch16_384", SCHEDULE, 128, 384),
}


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        p.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
        p["source"] = "measured"
    except Exception:
        pass
    return p


def flops_per_image(C=768, depth=12, P=196, schedule=None, hidden=None, classes=1000):
    """SURVEY.md 8(d): sum over blocks of qkv(6 N C^2) + attention(4 Np^2 C) + proj(2 Np C^2) + mlp(4 Np C hidden),
    plus patch-embed (2 P C 768) and head (2 C classes)."""
    sched = {int(i): c["keep_ratio"] for i, c in (SCHEDULE if schedule is None else schedule).items()}
    hidden = 4 * C if hidden is None else hidden
    n = P + 1
    total = 2.0 * P * C * 768 + 2.0 * C * classes
    for i in range(depth):
        np_ = max(1, int(sched[i] * (n - 1))) + 1 if i in sched else n
        total += 6.0 * n * C * C + 4.0 * np_ * np_ * C + 2.0 * np_ * C * C + 4.0 * np_ * C * hidden
        n = np_
    return total


def model_flops_per_image():
    return flops_per_image()


class ClockSampler:
    """nvidia-smi clocks and throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start_ready(self, timeout=5.0):
        """start(), then wait for the first sample: forking nvidia-smi and its driver attach take tens of ms during which
        kernel launches can stall - that must happen BEFORE the timed region, not inside it.  Samples taken so far are dropped."""
        self.start()
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)
        self.rows.clear()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "25"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for nme, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows else None,
                "power_w_max": max((float(r[2]) for r in self.rows if len(r) > 2), default=None),
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads() -> int:
    """Every core this process may run on (torchrun exports OMP_NUM_THREADS=1, which is not what the CPU leg wants)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(n)
    return torch.get_num_threads()


def dump_outputs(out_dir, logits, token_counts):
    """Write one step's results as a caller receives them: the logits [B, classes] (float32) and get_last_stats()'s
    per-block token counts (float64).  Logits larger than half of DUMP_BYTES are cut to a fixed, seeded sample of images;
    logits_rows.npy (float64) holds the batch index of every row written."""
    os.makedirs(out_dir, exist_ok=True)
    logits = logits.float().cpu().numpy()
    rows = np.arange(logits.shape[0])
    if logits.nbytes > DUMP_BYTES // 2:
        n = DUMP_BYTES // 2 // logits[0].nbytes
        rows = np.sort(np.random.default_rng(0).choice(logits.shape[0], n, replace=False))
    np.save(os.path.join(out_dir, "logits.npy"), logits[rows])
    np.save(os.path.join(out_dir, "logits_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "token_counts.npy"), np.asarray(token_counts, dtype=np.float64))


# --------------------------------------------------------------------------- the reference, unmodified (oracle/_ref)
def reference_pkg():
    """The staged copy of the reference package (oracle/make_ref.py), or None when it did not travel."""
    try:
        from oracle import make_ref
        return make_ref.import_reference() if make_ref.available() else None
    except Exception as e:                                     # edited copy, import error: say so, fall back to the port
        print(f"bench: oracle/_ref unusable ({e}); using the oracle port", file=sys.stderr)
        return None


def reference_model(pkg, device="cpu", dtype=torch.float32):
    """rajni.RAJNIViTWrapper (the reference's own class) around the stand-in ViT, as README.md:33-42 builds it."""
    from rajni_vit_b200.vit import create_model
    model = pkg.RAJNIViTWrapper(create_model(MODEL, seed=0), SCHEDULE).eval()
    return model.to(device=device, dtype=dtype)


def cpu_reference(batch, steps, warmup):
    """Time the reference path on the host cores: (images/s, s/step, kind).  kind "reference" = the unmodified reference
    wrapper driven by the reference's own evaluate_model (eval.py:6-75: wall clock around model(images) only);
    kind "port" = oracle/rajni_oracle.py when oracle/_ref is absent."""
    g = torch.Generator().manual_seed(1234)
    data = [(torch.randn(batch, 3, 224, 224, generator=g), torch.randint(0, 1000, (batch,), generator=g)) for _ in range(max(steps, 1))]
    pkg = reference_pkg()
    if pkg is not None:
        model = reference_model(pkg)
        with contextlib.redirect_stdout(sys.stderr):           # evaluate_model prints; stdout carries the ONE JSON line
            _, ips = pkg.evaluate_model(model, data, device="cpu", max_batches=steps, warmup=warmup)
        return ips, batch / ips, "reference"
    from oracle import rajni_oracle as orc
    from rajni_vit_b200.vit import create_model
    params = orc.extract_params(create_model(MODEL, seed=0))
    for _ in range(warmup):
        orc.forward(params, data[0][0], SCHEDULE)
    t0 = time.time()
    for i in range(steps):
        orc.forward(params, data[i][0], SCHEDULE)
    dt = time.time() - t0
    return batch * steps / dt, dt / steps, "port"


def gpu_eager_reference(dev, batch=BATCH, steps=5):
    """The unmodified reference wrapper, eager PyTorch, on this GPU: the same-box bar (SURVEY.md 8d).  fp32 is how the
    reference ships; .bfloat16() is the cast README.md:34 allows.  Timed like eval.py (sync, wall clock around model(x))."""
    pkg = reference_pkg()
    if pkg is None:
        return {"unavailable": "oracle/_ref did not travel to this box"}
    out = {"batch": batch, "steps": steps, "impl": "oracle/_ref: rajni.RAJNIViTWrapper (unmodified) on the stand-in ViT, eager PyTorch"}
    g = torch.Generator().manual_seed(1234)
    x32 = torch.randn(batch, 3, 224, 224, generator=g).to(dev)
    for name, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        try:
            model = reference_model(pkg, dev, dtype)
            x = x32.to(dtype)
            with torch.no_grad():
                for _ in range(2):
                    model(x)
                torch.cuda.synchronize(dev)
                t0 = time.time()
                for _ in range(steps):
                    model(x)
                torch.cuda.synchronize(dev)
            out[name] = {"value": round(batch * steps / (time.time() - t0), 1), "unit": "images/s"}
            del model
        except Exception as e:                                  # never let the context number kill the bench line
            out[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- parity on 256 images
def parity_sample(model, dev, images_total=256, chunk=64):
    """The metric's "top-1 agreement vs ref": 256 seeded images through the sm_100a path and through the CPU oracle
    (fp32, same weights), in chunks of 64.
    `teacher_forced`: the oracle is given OUR kept-token indices, so only the arithmetic is compared;
    `free_running`: the oracle selects for itself (random-init scores are nearly flat, so selections - and with them
    the logits - drift; SURVEY.md 4.6).
    `kept_sets`: our kept indices against the top-k of the ORACLE's scores on the same block input (teacher-forced
    trace); a disagreement is legitimate only inside the tie band (|score - cut| <= 3 % of the cut)."""
    from oracle import rajni_oracle as orc
    from rajni_vit_b200.vit import create_model
    params = orc.extract_params(create_model(MODEL, seed=0))
    g = torch.Generator().manual_seed(1234)
    ours_l, forced_l, free_l = [], [], []
    counts_ok = True
    sets = {"tokens_selected": 0, "tokens_disagreeing": 0, "disagreeing_outside_band": 0, "tokens_in_band": 0,
            "candidate_tokens": 0, "worst_rel_distance_of_a_disagreement": 0.0}
    for _ in range(images_total // chunk):
        images = torch.randn(chunk, 3, 224, 224, generator=g)
        ours_l.append(model(images.to(dev)).float().cpu())
        keep = [None if k is None else k.cpu().long() for k in model._last_keep_idx]
        counts = model.get_last_stats()["token_counts"]
        trace = []
        forced, stats = orc.forward(params, images, SCHEDULE, trace=trace, forced_keep=keep)
        counts_ok = counts_ok and counts == stats["token_counts"]
        forced_l.append(forced)
        for rec, kidx in zip(trace, keep):
            if kidx is None:
                continue
            k = kidx.shape[1] - 1
            s = rec["scores"][:, 1:].double()                                   # the oracle's scores on the same block input
            srt = torch.sort(s, dim=1, descending=True, stable=True)
            cut = srt.values[:, k - 1:k]
            ref_mask = torch.zeros_like(s, dtype=torch.bool).scatter_(1, srt.indices[:, :k], True)
            our_mask = torch.zeros_like(s, dtype=torch.bool).scatter_(1, kidx[:, 1:] - 1, True)
            rel = (s - cut).abs() / cut.abs()
            diff = ref_mask ^ our_mask
            sets["tokens_selected"] += int(our_mask.sum())
            sets["candidate_tokens"] += s.numel()
            sets["tokens_in_band"] += int((rel <= TIE_BAND).sum())
            sets["tokens_disagreeing"] += int(diff.sum())
            sets["disagreeing_outside_band"] += int((diff & (rel > TIE_BAND)).sum())
            if diff.any():
                sets["worst_rel_distance_of_a_disagreement"] = max(sets["worst_rel_distance_of_a_disagreement"], float(rel[diff].max()))
        del trace
        free_l.append(orc.forward(params, images, SCHEDULE)[0])
    ours, forced, free = torch.cat(ours_l), torch.cat(forced_l), torch.cat(free_l)

    def cmp(ref):
        err = (ours - ref).abs().max().item()
        top2 = ref.topk(2, dim=1).values
        margin = top2[:, 0] - top2[:, 1]                       # the oracle's own top-1 margin per image
        same = ours.argmax(1) == ref.argmax(1)
        decided = margin > 2 * err                             # images whose top-1 the logit error cannot flip
        return {"top1_agreement": round(same.float().mean().item(), 4),
                "max_abs_dlogit": round(err, 4),
                # random-init logits are nearly flat: a disagreement only counts where the reference's margin exceeds the error
                "top1_agreement_where_margin_exceeds_2x_error": round(same[decided].float().mean().item(), 4) if decided.any() else None,
                "images_with_such_margin": int(decided.sum()),
                "smallest_margin_of_a_disagreement": round(margin[~same].min().item(), 4) if (~same).any() else None}
    sets["worst_rel_distance_of_a_disagreement"] = round(sets["worst_rel_distance_of_a_disagreement"], 5)
    sets["tie_band"] = TIE_BAND
    sets["band_fraction_of_candidates"] = round(sets["tokens_in_band"] / max(sets["candidate_tokens"], 1), 5)
    sets["disagreeing_fraction_of_selected"] = round(sets["tokens_disagreeing"] / max(sets["tokens_selected"], 1), 6)
    return {"images": images_total, "token_counts_equal": counts_ok, "logit_std": round(forced.std().item(), 3),
            "teacher_forced": cmp(forced), "free_running": cmp(free), "kept_sets": sets}


def run_reference(args):
    """--impl reference: the reference path's own CPU implementation, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = host_threads()
    ips4, t4, kind = cpu_reference(4, 1, 1)
    budget = 150.0 / max(1, args.steps + args.warmup)           # seconds per step
    batch = int(max(1, min(32, budget / (t4 / 4))))
    ips, t_step, kind = cpu_reference(batch, args.steps, args.warmup)
    what = ("oracle/_ref: the unmodified reference wrapper + its evaluate_model on the stand-in ViT" if kind == "reference"
            else "oracle port of the reference path (oracle/_ref absent)")
    sample = f"{batch} images/step of {MODEL} + README schedule, fp32, {cores} threads (bounded sample of the bs-256 workload); {what}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(ips, 2), "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t_step * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_batch": batch,
                   "note": "img/s of a bounded sample (the CPU path's img/s does not depend on the batch beyond ~8 images)"},
        "cpu_baseline": {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(ips, 2), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # defaults long enough (~0.7 s timed) to sit in the sustained, power-capped clock regime the peaks file calls
    # "bf16_tflops_sustained"; a 10-step run finishes before the 1 kW cap pulls the SM clock down and reads ~10 % high
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="per-GPU batch (default = BASELINE config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip strong / configs / gpu_eager_reference / parity (quick runs)")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling as the headline: --batch is the GLOBAL batch, sharded over the ranks (the default line "
                         "is weak scaling and carries the sharded reading under the key `strong`)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what rank 0's last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the b200 path; --impl reference has no outputs to write")

    if args.impl == "reference":
        args.warmup = max(args.warmup, 1)
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from rajni_vit_b200 import RAJNIViTWrapper, _lib, ops
    from rajni_vit_b200.vit import VIT_CONFIGS, create_model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch // world if args.strong else args.batch          # per-GPU batch
    if B <= 0:
        raise SystemExit("--strong: the global batch must be at least the number of ranks")
    model = RAJNIViTWrapper(create_model(MODEL, seed=0), SCHEDULE).to(dev).eval()
    # weak scaling (the default): every launch goes through the C ABI and is counted.  --strong leaves the wrapper's default
    # (graph replay for small per-GPU batches); the launch count then comes from one eager step.
    model.use_cuda_graph = None if args.strong else False
    g = torch.Generator().manual_seed(1234 + rank)
    host = [torch.randn(B, 3, 224, 224, generator=g).pin_memory() for _ in range(2)]
    resident = [h.to(dev) for h in host]              # 154 MB each: larger than the 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """ms for `steps` calls of fn(i): CUDA events on the launch stream, barrier + synchronize on both sides, MAX over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---------------- device-resident throughput ----------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start_ready()                              # nvidia-smi is attached and polling before the warm-up ends
    for i in range(args.warmup):
        model(resident[i & 1])
    barrier()
    if rank == 0:
        sampler.rows.clear()                               # keep only the samples of the timed region
    launches0 = _lib.launch_count()
    last = {}

    def step(i):
        last["logits"] = model(resident[i & 1])
    ms_total = timed(step, args.steps)
    logits = last["logits"]
    launches = _lib.launch_count() - launches0
    if args.strong and launches == 0:                      # graph replay: count the launches of one eager step instead
        c0 = _lib.launch_count()
        model._forward_eager(resident[0])
        launches = (_lib.launch_count() - c0) * args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_total * 1e-3)
    assert model.get_last_stats()["token_counts"] == TOKENS and torch.isfinite(logits).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logits, model.get_last_stats()["token_counts"])

    # ---------------- the same loop for >= 1 s: the power-capped regime ----------------
    sus_steps = max(args.steps, int(math.ceil(1200.0 / (ms_total / args.steps))))
    sampler2 = ClockSampler(local)
    if rank == 0:
        sampler2.start_ready()
    sus_ms = timed(step, sus_steps)
    sus_clocks = sampler2.stop() if rank == 0 else None
    sustained = {"value": round(world * B * sus_steps / (sus_ms * 1e-3), 1), "unit": "images/s", "steps": sus_steps,
                 "seconds": round(sus_ms * 1e-3, 3), "ms_per_step": round(sus_ms / sus_steps, 3),
                 "sm_mhz": None if sus_clocks is None else sus_clocks.get("sm_mhz"),
                 "reasons": None if sus_clocks is None else sus_clocks.get("reasons")}

    # ---------------- end to end from pinned host memory ----------------
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)
    stage = [torch.empty_like(resident[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    preds_host = torch.empty((args.steps, B), dtype=torch.int64).pin_memory()

    def e2e_loop(n, host=host, stage=stage):
        with torch.cuda.stream(copy_stream):
            stage[0].copy_(host[0], non_blocking=True)
            ready[0].record(copy_stream)
        for i in range(n):
            s = i & 1
            if i + 1 < n:
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(freed[s ^ 1])
                    stage[s ^ 1].copy_(host[(i + 1) & 1], non_blocking=True)
                    ready[s ^ 1].record(copy_stream)
            main_stream.wait_event(ready[s])
            out = model(stage[s])
            freed[s].record(main_stream)
            preds_host[i % args.steps].copy_(out.argmax(dim=1), non_blocking=True)
        torch.cuda.synchronize(dev)

    e2e_loop(2)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(dt.item())

    # the same loop fed with raw uint8 pixels (extension: normalisation inside the patch kernel, a quarter of the H2D bytes)
    from rajni_vit_b200.run import IMAGENET_MEAN, IMAGENET_STD
    model.set_input_normalization(IMAGENET_MEAN, IMAGENET_STD)
    host8 = [torch.randint(0, 256, (B, 3, 224, 224), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    stage8 = [torch.empty((B, 3, 224, 224), device=dev, dtype=torch.uint8) for _ in range(2)]
    e2e_loop(2, host8, stage8)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps, host8, stage8)
    dt8 = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(dt8, op=dist.ReduceOp.MAX)
    e2e_u8_value = world * B * args.steps / float(dt8.item())
    del host8, stage8

    # ---------------- per-kernel CUDA-event profile (separate instrumented steps) ----------------
    prof = ops.profile_steps(lambda: model(resident[0]), steps=5)
    pk = peaks()
    gemm = {"ms": 0.0, "work": 0.0, "launches": 0}
    for name, v in prof.items():
        if name.startswith("gemm"):
            for k in gemm:
                gemm[k] += v[k]
    gemm_tflops = gemm["work"] / (gemm["ms"] * 1e-3) / 1e12 if gemm["ms"] else 0.0
    peak_tf = pk["bf16_tflops_sustained"]
    traffic, traffic_src = None, None
    try:                               # ncu dram bytes per GEMM launch, captured once per round (bench.py cannot run ncu itself)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["gemm"]
        traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05, all GEMM launches of a step)",
                "achieved": round(gemm_tflops, 1), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(gemm_tflops / peak_tf, 4), "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)",
                "traffic_source": traffic_src, "flop_per_launch": round(gemm["work"] / max(gemm["launches"], 1), 1),
                "peak_source": pk["source"] + " sustained",
                "launches_per_step": gemm["launches"], "ms_per_step": round(gemm["ms"], 3)}
    step_ms = sum(v["ms"] for v in prof.values())
    kernels = {}
    for name, v in sorted(prof.items()):
        rate = v["work"] / (v["ms"] * 1e-3) if v["ms"] else 0.0
        unit, peak = ("TFLOP/s", pk["bf16_tflops_sustained"] * 1e12) if name.startswith("gemm") or name == "attention" else ("GB/s", pk["hbm_gbs"] * 1e9)
        kernels[name] = {"ms_per_step": round(v["ms"], 3), "share": round(v["ms"] / step_ms, 4) if step_ms else None,
                         "launches": v["launches"], "achieved": round(rate / (1e12 if unit == "TFLOP/s" else 1e9), 1),
                         "unit": unit, "frac_of_peak": round(rate / peak, 4)}
    kernels_note = (f"per-launch CUDA-event pairs on separate instrumented steps: their sum is {step_ms:.3f} ms against "
                    f"{ms_total / args.steps:.3f} ms per un-instrumented step (event bracketing serialises the programmatic-dependent-"
                    "launch overlap), so per-kernel frac_of_peak values are pessimistic by that ratio")

    # ---------------- north_star's sharded reading, and BASELINE configs 3-5 sharded over the ranks ----------------
    strong, configs = None, None
    if not args.no_extras:
        model.input_norm = None
        model._graphs = {}
        Bs = max(1, BATCH // world)
        model.use_cuda_graph = None                             # the wrapper's default: graph replay for launch-bound shards
        xs = [torch.randn(Bs, 3, 224, 224, generator=g).to(dev) for _ in range(2)]
        for i in range(5):
            model(xs[i & 1])
        st_steps = max(20, min(200, args.steps))
        ms_s = timed(lambda i: model(xs[i & 1]), st_steps)
        strong = {"value": round(world * Bs * st_steps / (ms_s * 1e-3), 1), "unit": "images/s", "global_batch": Bs * world,
                  "per_gpu_batch": Bs, "steps": st_steps, "ms_per_step": round(ms_s / st_steps, 3),
                  "frac_of_tensor_roofline": round(Bs * st_steps / (ms_s * 1e-3) * flops_per_image() / 1e12 / peak_tf, 4),
                  "cuda_graph": bool(Bs * 197 <= 16384),
                  "note": "the GLOBAL batch 256 sharded over the ranks (north_star: 'the batch is sharded'); value is the whole job"}
        model.use_cuda_graph = False
        del xs
        configs = {}
        for cname, (mname, sched, gbatch, size) in CONFIGS.items():
            del model
            torch.cuda.empty_cache()
            dim, depth, heads, _ = VIT_CONFIGS[mname]
            model = RAJNIViTWrapper(create_model(mname, seed=0), sched).to(dev).eval()
            Bc = max(1, gbatch // world)
            xs = [torch.randn(Bc, 3, size, size, generator=g).to(dev) for _ in range(2)]
            for i in range(4):
                model(xs[i & 1])
            c_steps = 20
            ms_c = timed(lambda i: model(xs[i & 1]), c_steps)
            fl = flops_per_image(C=dim, depth=depth, P=(size // 16) ** 2, schedule=sched)
            ips = Bc * c_steps / (ms_c * 1e-3)
            configs[cname] = {"model": mname, "global_batch": Bc * world, "per_gpu_batch": Bc, "value": round(world * ips, 1),
                              "unit": "images/s", "ms_per_step": round(ms_c / c_steps, 3), "gflop_per_image": round(fl / 1e9, 3),
                              "frac_of_tensor_roofline": round(ips * fl / 1e12 / peak_tf, 4),
                              "token_counts": model.get_last_stats()["token_counts"]}
            del xs
        del model
        torch.cuda.empty_cache()
        model = RAJNIViTWrapper(create_model(MODEL, seed=0), SCHEDULE).to(dev).eval()
        model.use_cuda_graph = False

    out = None
    if rank == 0:
        flops_img = model_flops_per_image()
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "two alternating 154 MB input batches and >1 GB of activations per step (larger than the 126 MB L2)",
                       "token_counts": TOKENS, "gflop_per_image": round(flops_img / 1e9, 3)},
            "model_tflops": round(value * flops_img / 1e12 / world, 1),
            "model_frac_of_tensor_peak": round(value * flops_img / 1e12 / world / peak_tf, 4),
            "sustained": sustained,
            "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "h2d_bytes_per_step": B * 3 * 224 * 224 * 4,
                    "d2h_bytes_per_step": B * 8, "note": "pinned fp32 images, H2D double-buffered on a copy stream"},
            "e2e_uint8": {"value": round(e2e_u8_value, 1), "unit": "images/s", "h2d_bytes_per_step": B * 3 * 224 * 224,
                          "d2h_bytes_per_step": B * 8, "note": "extension: pinned uint8 pixels, ToTensor+Normalize inside the patch kernel"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels, "kernels_note": kernels_note,
        }
        if strong is not None:
            out["strong"] = strong
            out["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            cores = host_threads()
            ips, t_step, kind = cpu_reference(16, 2, 1)
            what = ("oracle/_ref: the unmodified reference wrapper + its evaluate_model on the stand-in ViT" if kind == "reference"
                    else "oracle port of the reference path")
            out["cpu_baseline"] = {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": kind,
                                   "sample": f"3 forwards (1 warm-up + 2 timed) of 16 images, {what}, fp32, {cores} threads"}
            if not args.no_extras:
                out["gpu_eager_reference"] = gpu_eager_reference(dev)
                out["parity"] = parity_sample(model, dev)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
