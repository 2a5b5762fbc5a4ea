"""Pruning-schedule search: throughput against accuracy (SURVEY.md 8f item 4).

The reference leaves the schedule to the user (README.md quick start, schedule.json; `rajni/run.py:108-123` just loads it).
This module measures candidates on the device the model will run on and picks one:

* ``measure(make_model, schedule, batches)`` - images/s of the wrapped model, tensor work per image, and the accuracy axis:
  top-1 accuracy when the batches carry labels (real weights: ``load_checkpoint`` + an ImageNet loader), and always the
  agreement with the UN-PRUNED model's predictions on the same inputs (with random-init stand-ins this only says how much
  the pruning perturbs the logits - it is the axis the tests use).  A headless model (``head`` = Identity, num_classes=0)
  has no predictions: its accuracy axis is the mean cosine similarity, in %, between each image's pruned and dense features
  (``cosine_agreement``).
* ``pareto_front(results)`` - the candidates no other candidate beats on both axes.
* ``search(make_model, batches, ...)`` - greedy descent from the dense model: repeatedly lower the keep ratio of the one
  block whose step buys the most images/s per point of accuracy lost, while the accuracy stays above the floor.

Everything that decides (``pareto_front``, ``greedy_search`` over an arbitrary ``measure`` callable, ``candidate_grid``,
``flops_per_image``) is host logic and is tested on the CPU; the measurement itself needs the GPU.
"""
from __future__ import annotations

import copy
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import torch

Schedule = Dict[int, Dict]


def flops_per_image(token_counts: Sequence[int], C: int, hidden: int, patches: int, classes: int = 1000, patch_dim: int = 768) -> float:
    """Tensor work of one image under a schedule (SURVEY 8d): token_counts[i] = tokens ENTERING block i.
    ``patch_dim`` = 3 p^2, the patch-embed GEMM's K (768 at p = 16)."""
    total = 2.0 * patches * C * patch_dim + 2.0 * C * classes
    for i, n in enumerate(token_counts):
        kept = token_counts[i + 1] if i + 1 < len(token_counts) else n    # tokens after this block's pruning
        total += 6.0 * n * C * C + 4.0 * kept * kept * C + 2.0 * kept * C * C + 4.0 * kept * C * hidden
    return total


def token_counts(schedule: Schedule, depth: int, tokens: int, prefix: int = 1) -> List[int]:
    """Tokens entering each block: block i listed in the schedule keeps max(1, int(r * (N - prefix))) patches + the
    ``prefix`` leading tokens (attention.py:31-32; prefix 2 for a distilled DeiT's CLS + distillation token), and the kept
    tokens are what the block's own attention and MLP run on."""
    out, n = [], tokens
    for i in range(depth):
        out.append(n)
        if i in schedule:
            n = max(1, int(float(schedule[i].get("keep_ratio", 1.0)) * (n - prefix))) + prefix
    return out


def candidate_grid(depth: int, first_block: int = 3, ratios: Sequence[float] = (0.9, 0.8, 0.7, 0.5)) -> List[Tuple[str, Schedule]]:
    """A small fixed family: the README schedule, uniform pruning from `first_block` on, every third block."""
    out: List[Tuple[str, Schedule]] = [("dense", {})]
    readme = {3: 0.88, 4: 0.88, 7: 0.8, 8: 0.72}
    if depth > max(readme):
        out.append(("README", {i: {"keep_ratio": r} for i, r in readme.items()}))
    for r in ratios:
        out.append((f"every block from {first_block}, keep {r}", {i: {"keep_ratio": r} for i in range(first_block, depth)}))
        thirds = [i for i in range(first_block, depth, 3)]
        out.append((f"blocks {thirds}, keep {r}", {i: {"keep_ratio": r} for i in thirds}))
        if len(thirds) > 1:
            out.append((f"blocks {thirds}, keep {r}, scores carried",
                        {i: {"keep_ratio": r, "update": j == 0} for j, i in enumerate(thirds)}))
    return out


def pareto_front(results: Iterable[Dict], speed: str = "img_s", quality: str = "accuracy") -> List[Dict]:
    """Results not dominated on (speed, quality), fastest first.  Equal points keep the first seen."""
    rs = sorted(results, key=lambda r: (-r[speed], -r[quality]))
    front, best_q = [], float("-inf")
    for r in rs:
        if r[quality] > best_q:
            front.append(r)
            best_q = r[quality]
    return front


def greedy_search(measure_fn: Callable[[Schedule], Dict], depth: int, floor: float, blocks: Optional[Sequence[int]] = None,
                  ratios: Sequence[float] = (1.0, 0.9, 0.8, 0.7, 0.6, 0.5), quality: str = "accuracy", speed: str = "img_s",
                  max_steps: int = 64) -> Tuple[Schedule, List[Dict]]:
    """Greedy descent.  State: one ratio index per candidate block (0 = not pruned).  Each step tries lowering every block
    by one notch, keeps the move with the best (speed gained) / (quality lost, at least 1e-6) whose quality stays >= floor,
    and stops when no move is admissible.  Returns (schedule, history of accepted results; history[0] is the dense model)."""
    blocks = list(range(depth)) if blocks is None else list(blocks)
    level = {b: 0 for b in blocks}

    def to_schedule(lv):
        return {b: {"keep_ratio": ratios[i]} for b, i in sorted(lv.items()) if i > 0}

    cur = dict(measure_fn({}))
    cur["schedule"] = {}
    history = [cur]
    for _ in range(max_steps):
        best = None
        for b in blocks:
            if level[b] + 1 >= len(ratios):
                continue
            trial = dict(level)
            trial[b] += 1
            r = dict(measure_fn(to_schedule(trial)))
            if r[quality] < floor or r[speed] <= cur[speed]:
                continue
            gain = (r[speed] - cur[speed]) / max(cur[quality] - r[quality], 1e-6)
            if best is None or gain > best[0]:
                best = (gain, b, r)
        if best is None:
            break
        _, b, r = best
        level[b] += 1
        r["schedule"] = to_schedule(level)
        history.append(r)
        cur = r
    return to_schedule(level), history


# ------------------------------------------------------------------ measurement (GPU)
def cosine_agreement(features: Sequence[torch.Tensor], dense_features: Sequence[torch.Tensor]) -> float:
    """Mean over images of the cosine similarity between an image's features and its dense features, in % (batches of
    [B, C] in the same order on both sides; fp64 arithmetic)."""
    total, seen = 0.0, 0
    for f, d in zip(features, dense_features, strict=True):
        total += float(torch.nn.functional.cosine_similarity(f.double(), d.to(f.device).double(), dim=1).sum())
        seen += f.shape[0]
    return 100.0 * total / seen


def _split(batch):
    if isinstance(batch, (tuple, list)):
        return batch[0], (batch[1] if len(batch) > 1 else None)
    return batch, None


@torch.no_grad()
def measure(make_model: Callable[[], torch.nn.Module], schedule: Schedule, batches: Sequence, device="cuda",
            dense_predictions: Optional[List[torch.Tensor]] = None, timing_steps: int = 10) -> Dict:
    """One candidate: wrap a FRESH base model (the wrapper replaces its attention modules: `model.py:7-25`), run every batch
    once for the accuracy axis, then time `timing_steps` forwards of the first batch with CUDA events.
    ``accuracy`` is top-1 against the labels when the batches have them, else the agreement with `dense_predictions`.
    A headless model's ``predictions`` are its features, and ``accuracy`` is their ``cosine_agreement`` with
    `dense_predictions`, labels or not."""
    from .wrapper import RAJNIViTWrapper
    base = make_model()
    model = RAJNIViTWrapper(base, copy.deepcopy(schedule)).to(device).eval()
    preds, correct, labelled, agree, seen = [], 0, 0, 0, 0
    for i, batch in enumerate(batches):
        x, y = _split(batch)
        if model.headless:
            preds.append(model(x.to(device, non_blocking=True)))
            continue
        p = model(x.to(device, non_blocking=True)).argmax(dim=1)
        preds.append(p)
        seen += p.numel()
        if y is not None:
            correct += int((p.cpu() == y.cpu()).sum())
            labelled += p.numel()
        if dense_predictions is not None:
            agree += int((p == dense_predictions[i].to(p.device)).sum())
    x0 = _split(batches[0])[0].to(device)
    for _ in range(3):
        model(x0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(timing_steps):
        model(x0)
    e1.record()
    torch.cuda.synchronize()
    counts = model.get_last_stats()["token_counts"]
    blk = base.blocks[0]
    C = base.patch_embed.proj.out_channels
    size = x0.shape[-1]
    p = base.patch_embed.proj.kernel_size[0]
    out = {
        "schedule": copy.deepcopy(schedule), "img_s": x0.shape[0] * timing_steps / (e0.elapsed_time(e1) * 1e-3),
        "token_counts": counts,
        "gflop_per_image": flops_per_image(counts, C, blk.mlp.fc1.out_features, (size // p) ** 2,
                                           classes=0 if model.headless else base.head.out_features, patch_dim=3 * p * p) / 1e9,
        "top1": (100.0 * correct / labelled) if labelled else None,
        "agreement": (100.0 if dense_predictions is None else cosine_agreement(preds, dense_predictions) if model.headless
                      else 100.0 * agree / seen),
        "predictions": preds,
    }
    out["accuracy"] = out["top1"] if out["top1"] is not None else out["agreement"]
    return out


def sweep(make_model, batches, candidates: Optional[Sequence[Tuple[str, Schedule]]] = None, device="cuda", timing_steps: int = 10) -> List[Dict]:
    """Measure a family of schedules (default: `candidate_grid`); every result carries its name and both accuracy readings."""
    dense = measure(make_model, {}, batches, device, None, timing_steps)
    depth = len(make_model().blocks)
    out = []
    for name, sched in (candidates if candidates is not None else candidate_grid(depth)):
        r = dense if not sched else measure(make_model, sched, batches, device, dense["predictions"], timing_steps)
        r = dict(r, name=name)
        out.append(r)
    return out


def search(make_model, batches, floor: float, device="cuda", blocks: Optional[Sequence[int]] = None,
           ratios: Sequence[float] = (1.0, 0.9, 0.8, 0.7, 0.6, 0.5), timing_steps: int = 5) -> Tuple[Schedule, List[Dict]]:
    """`greedy_search` with `measure` as the evaluator: the fastest schedule found whose accuracy (top-1 with labels, else
    agreement with the dense model; for a headless model the features' cosine agreement; all in %) stays at or above
    `floor`."""
    dense = measure(make_model, {}, batches, device, None, timing_steps)
    depth = len(make_model().blocks)
    cache: Dict[str, Dict] = {}

    def fn(sched: Schedule) -> Dict:
        key = repr(sorted((k, sorted(v.items())) for k, v in sched.items()))
        if key not in cache:
            cache[key] = dense if not sched else measure(make_model, sched, batches, device, dense["predictions"], timing_steps)
        return cache[key]

    return greedy_search(fn, depth, floor, blocks if blocks is not None else range(1, depth), ratios)
