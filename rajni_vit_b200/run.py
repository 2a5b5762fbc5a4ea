"""Command-line evaluation — same flags as ``python -m rajni.run`` (rajni/run.py:17-43), B200 path.

    python -m rajni_vit_b200.run --data_path /data/imagenet/val --schedule schedule.json --compare_base
    python -m rajni_vit_b200.run --synthetic 20 --schedule schedule.json            # no dataset needed
    torchrun --nproc-per-node 8 -m rajni_vit_b200.run ...                           # data parallel (SURVEY 8e)

Differences from the reference CLI, all deliberate (SURVEY.md section 5):
  * schedule keys from JSON are strings; they are normalised to block indices (the reference prunes nothing);
  * timings are synchronised (the reference passes a torch.device, which disables its own sync);
  * ``--compare_base`` runs the un-pruned model through the same sm_100a kernels (empty schedule), so the
    speed-up isolates the pruning and not the kernel implementation;
  * ``--synthetic N`` replaces the ImageFolder pipeline by N seeded random batches (no dataset, no labels that mean
    anything: accuracy is only a consistency check then);
  * ``--uint8_input`` ships uint8 crops and normalises inside the patch kernel (extension; same logits, 4x fewer H2D bytes);
  * ``--gpu_preprocess`` leaves only the JPEG decode to the CPU workers: Resize(256, bicubic) + CenterCrop(224) run in
    ``csrc/resize.cu`` (bit-identical to torchvision on PIL images), ToTensor + Normalize in the patch kernel;
  * ``--gpu_decode`` (implies ``--gpu_preprocess``) moves the JPEG decode to the GPU as well (``csrc/jpeg.cu``, frames
    equal to Pillow's); the workers read files and decode on the CPU only what the GPU decoder does not take;
  * ``--ckpt file`` loads timm-named weights from a .safetensors / .pt file (no hub access needed);
  * under torchrun every rank decodes only its shard of each batch (``data.sharded_loader``);
  * without ``timm`` (not installable here) the stand-in ViT with random weights is used and the fact is printed;
  * a headless model (num_classes=0) is refused: it has no class scores to take a top-1 accuracy of.
"""
from __future__ import annotations

import argparse
import json
import os

import torch

from .eval import evaluate_model
from .wrapper import RAJNIViTWrapper
from .wrapper.model import _is_identity


def get_args(argv=None):
    ap = argparse.ArgumentParser("RAJNI evaluation (B200)")
    ap.add_argument("--data_path", type=str, default=None, help="ImageNet-style dataset root (ImageFolder)")
    ap.add_argument("--synthetic", type=int, default=0, help="use this many synthetic batches instead of --data_path")
    ap.add_argument("--batch_size", type=int, default=256)
    ap.add_argument("--num_workers", type=int, default=8)
    ap.add_argument("--pin_mem", action="store_true", default=True)
    ap.add_argument("--model", type=str, default="vit_base_patch16_224",
                    help="timm model name; without timm, a stand-in of vit.VIT_CONFIGS (e.g. vit_base_patch16_224, "
                         "deit3_base_patch16_224, deit_base_distilled_patch16_224)")
    ap.add_argument("--device", type=str, default="cuda")
    ap.add_argument("--schedule", type=str, default=None, help="JSON file with the RAJNI pruning schedule")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--max_batches", type=int, default=None)
    ap.add_argument("--compare_base", action="store_true", help="also evaluate the un-pruned model")
    ap.add_argument("--ckpt", type=str, default=None,
                    help="timm-named ViT weights (.safetensors / .pt) to load instead of timm's hub (rajni_vit_b200.load_checkpoint)")
    ap.add_argument("--gpu_preprocess", action="store_true",
                    help="workers only decode; Resize(256, bicubic) + CenterCrop(224) + ToTensor + Normalize run on the GPU "
                         "(bit-identical to the torchvision pipeline; implies --uint8_input)")
    ap.add_argument("--gpu_decode", action="store_true",
                    help="decode baseline JPEGs on the GPU too (frames equal to Pillow's; other files are decoded by the "
                         "workers); implies --gpu_preprocess")
    ap.add_argument("--uint8_input", action="store_true",
                    help="ship uint8 crops to the GPU and normalise inside the patch kernel (4x fewer H2D bytes; same logits)")
    args = ap.parse_args(argv)
    if args.gpu_decode:
        args.gpu_preprocess = True
    if args.gpu_preprocess:
        args.uint8_input = True
    if not args.data_path and args.synthetic <= 0:
        ap.error("give --data_path or --synthetic N")
    return args


def build_model(name: str, ckpt: str = None):
    """A checkpoint file when given (architecture inferred from its shapes), else timm's pretrained model when timm is
    present, otherwise the random-init stand-in with timm's attribute names."""
    if ckpt:
        from .checkpoint import load_checkpoint
        return load_checkpoint(ckpt), f"weights from {ckpt}"
    try:
        import timm                                             # noqa: F401
        return timm.create_model(name, pretrained=True), "timm (pretrained)"
    except ImportError:
        from .vit import create_model
        return create_model(name, seed=0), "stand-in ViT, random init (timm is not installed)"


IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)      # run.py:68


def build_loader(args, image_size: int, rank: int = 0, world: int = 1):
    if args.synthetic > 0:
        g = torch.Generator().manual_seed(1234)
        shape = (args.batch_size, 3, image_size, image_size)
        return [(torch.randint(0, 256, shape, generator=g, dtype=torch.uint8) if args.uint8_input else torch.randn(shape, generator=g),
                 torch.randint(0, 1000, (args.batch_size,), generator=g)) for _ in range(args.synthetic)]
    import torchvision.datasets as datasets
    import torchvision.transforms as T
    if args.gpu_preprocess:
        if image_size != 224:
            raise ValueError("--gpu_preprocess: the GPU resize kernel crops to 224 x 224")
        from .data import (GpuDecodeLoader, GpuPreprocessLoader, collate_frames, decode_only, read_for_gpu_decode,
                           sharded_loader)
        ds = (datasets.ImageFolder(args.data_path, loader=read_for_gpu_decode) if args.gpu_decode else
              datasets.ImageFolder(args.data_path, decode_only))
        kw = dict(num_workers=args.num_workers, pin_memory=False, collate_fn=collate_frames)
        inner = (sharded_loader(ds, args.batch_size, rank, world, **kw) if world > 1 else
                 torch.utils.data.DataLoader(ds, batch_size=args.batch_size, shuffle=False, drop_last=False, **kw))
        wrap = GpuDecodeLoader if args.gpu_decode else GpuPreprocessLoader
        return wrap(inner, torch.device(args.device if world == 1 else f"cuda:{torch.cuda.current_device()}"))
    tail = [T.PILToTensor()] if args.uint8_input else [T.ToTensor(), T.Normalize(mean=IMAGENET_MEAN, std=IMAGENET_STD)]
    tf = T.Compose([T.Resize(int(image_size * 256 / 224), interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(image_size), *tail])
    ds = datasets.ImageFolder(args.data_path, tf)
    if world > 1:          # every rank decodes only its shard of each global batch (data.py); same images per rank as slicing
        from .data import sharded_loader
        return sharded_loader(ds, args.batch_size, rank, world, num_workers=args.num_workers, pin_memory=args.pin_mem)
    return torch.utils.data.DataLoader(ds, batch_size=args.batch_size, shuffle=False, num_workers=args.num_workers,
                                       pin_memory=args.pin_mem, drop_last=False)


def main(argv=None):
    args = get_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    say = print if rank == 0 else (lambda *a, **k: None)
    say("Args:", vars(args))

    if args.schedule is None:
        raise ValueError("a pruning schedule is required (--schedule file.json)")      # run.py:115-116
    with open(args.schedule) as f:
        schedule = json.load(f)

    base, origin = build_model(args.model, args.ckpt)
    say(f"model {args.model}: {origin}")
    if hasattr(base, "head") and _is_identity(base.head):
        raise ValueError(f"{args.model} is headless (head = Identity, num_classes=0): it outputs features, not class scores, "
                         "so it has no top-1 accuracy to measure; rajni_vit_b200.schedule.measure reports the features' cosine "
                         "agreement with the un-pruned model instead")
    size = getattr(getattr(base, "patch_embed", None), "img_size", (224, 224))
    size = size[0] if isinstance(size, (tuple, list)) else int(size)
    loader = build_loader(args, size, rank, world)

    results = {}
    if args.compare_base:
        dense, _ = build_model(args.model, args.ckpt)
        dense = RAJNIViTWrapper(dense, {})                       # no block pruned: the same kernels, all tokens
        if args.uint8_input:
            dense.set_input_normalization(IMAGENET_MEAN, IMAGENET_STD)
        acc, ips = evaluate_model(dense, loader, device=args.device, max_batches=args.max_batches, warmup=args.warmup)
        results["base"] = (acc, ips)
        say(f"[base ] accuracy {acc:.2f} %   throughput {ips:.1f} img/s")
        del dense
    model = RAJNIViTWrapper(base, schedule)
    if args.uint8_input:
        model.set_input_normalization(IMAGENET_MEAN, IMAGENET_STD)
    acc, ips = evaluate_model(model, loader, device=args.device, max_batches=args.max_batches, warmup=args.warmup)
    results["rajni"] = (acc, ips)
    say(f"[rajni] accuracy {acc:.2f} %   throughput {ips:.1f} img/s   token_counts {model.get_last_stats()['token_counts']}")
    if "base" in results:
        say(f"speed-up {results['rajni'][1] / results['base'][1]:.2f}x   accuracy drop {results['base'][0] - results['rajni'][0]:.2f} points")
    if world > 1:
        torch.distributed.destroy_process_group()
    return results


if __name__ == "__main__":
    main()
