"""Loader-side data parallelism: every rank decodes only ITS shard of each global batch.

The reference builds one ``DataLoader(ImageFolder, batch_size=B, shuffle=False)`` (``rajni/run.py:72-82``) and has no
notion of ranks.  ``evaluate_model`` can shard any foreign loader by slicing each batch after it was loaded — correct,
but every rank then decodes and resizes the WHOLE batch and throws (N-1)/N of it away.  When the loader is ours, the
sharding moves into the sampler: ``RankShardedBatchSampler`` yields, for global batch k = indices [kB, (k+1)B), exactly
the contiguous slice ``shard_bounds`` would have cut for this rank, so the images a rank sees (and their order) are the
same as on the slice path, with 1/N of the decode work.  A loader built this way carries ``rajni_sharded = True`` and
``evaluate_model`` then leaves its batches alone (the final all-reduce of the counters is unchanged).
"""
from __future__ import annotations

from typing import Iterator, List

import torch

from .eval import shard_bounds


class RankShardedBatchSampler(torch.utils.data.Sampler):
    """Batch sampler over ``range(n)`` in order: global batches of ``batch_size`` (last one partial unless ``drop_last``),
    each cut into ``world`` contiguous shards; this rank's shard is yielded.  Shards that come out empty (fewer images
    than ranks in the last batch) are skipped."""

    def __init__(self, n: int, batch_size: int, rank: int, world: int, drop_last: bool = False):
        if not 0 <= rank < world:
            raise ValueError(f"rank {rank} outside world of {world}")
        self.n, self.batch_size, self.rank, self.world, self.drop_last = n, batch_size, rank, world, drop_last

    def _batches(self) -> Iterator[List[int]]:
        for start in range(0, self.n, self.batch_size):
            size = min(self.batch_size, self.n - start)
            if size < self.batch_size and self.drop_last:
                return
            lo, hi = shard_bounds(size, self.rank, self.world)
            if hi > lo:
                yield list(range(start + lo, start + hi))

    def __iter__(self):
        return self._batches()

    def __len__(self):
        return sum(1 for _ in self._batches())


def sharded_loader(dataset, batch_size: int, rank: int, world: int, **kw) -> torch.utils.data.DataLoader:
    """``DataLoader(dataset, batch_size, shuffle=False)`` whose batches are this rank's shards (see module docstring)."""
    kw.pop("shuffle", None)
    drop_last = kw.pop("drop_last", False)
    loader = torch.utils.data.DataLoader(
        dataset, batch_sampler=RankShardedBatchSampler(len(dataset), batch_size, rank, world, drop_last), **kw)
    loader.rajni_sharded = True
    return loader


# ------------------------------------------------------------------ GPU-side Resize + CenterCrop (run.py:62-66)
def decode_only(img) -> torch.Tensor:
    """Dataset transform for the GPU pipeline: the decoded frame as a uint8 [H,W,3] tensor, nothing else (the CPU workers
    only decode; Resize(256, bicubic) + CenterCrop(224) + ToTensor + Normalize all run on the GPU)."""
    import numpy as np
    return torch.from_numpy(np.asarray(img.convert("RGB")).copy())


def collate_frames(batch):
    """Frames have different sizes: keep them as a list; labels become one tensor."""
    return [b[0] for b in batch], torch.as_tensor([b[1] for b in batch])


def pack_frames(frames):
    """[H_i,W_i,3] uint8 frames -> (one pinned 1-D uint8 buffer, meta int64 [B,3] = (byte offset, H, W), max H)."""
    sizes = [int(f.numel()) for f in frames]
    buf = torch.empty(sum(sizes), dtype=torch.uint8)
    if torch.cuda.is_available():
        buf = buf.pin_memory()
    meta = torch.empty((len(frames), 3), dtype=torch.int64)
    off = 0
    for i, f in enumerate(frames):
        if f.dtype != torch.uint8 or f.dim() != 3 or f.shape[2] != 3:
            raise ValueError(f"frame {i}: expected uint8 [H,W,3], got {f.dtype} {tuple(f.shape)}")
        buf[off:off + sizes[i]] = f.reshape(-1)
        meta[i, 0], meta[i, 1], meta[i, 2] = off, f.shape[0], f.shape[1]
        off += sizes[i]
    return buf, meta, int(meta[:, 1].max())


def gpu_resize_center_crop(frames, device, size: int = 256, crop: int = 224) -> torch.Tensor:
    """Decoded uint8 frames (list of [H,W,3]) -> uint8 [B,3,crop,crop] on ``device``, bit-identical to
    ``Resize(size, BICUBIC) -> CenterCrop(crop) -> PILToTensor`` (one H2D copy of the packed frames, three kernels)."""
    from . import ops
    buf, meta, max_h = pack_frames(frames)
    return ops.resize_center_crop(buf.to(device, non_blocking=True), meta.to(device, non_blocking=True), max_h, size=size, crop=crop)


class GpuPreprocessLoader:
    """Wraps a loader that yields ``(list of decoded uint8 frames, labels)`` (``decode_only`` + ``collate_frames``): every batch
    is resized and cropped on ``device`` and comes out as ``(uint8 [B,3,crop,crop] CUDA tensor, labels)`` - what the wrapper
    takes after ``set_input_normalization`` (ToTensor + Normalize happen in the patch kernel).  The CPU workers are left with
    JPEG decoding only; at 30 k img/s per GPU the reference's CPU Resize/CenterCrop would need ~100 cores."""

    def __init__(self, loader, device, size: int = 256, crop: int = 224):
        self.loader, self.device, self.size, self.crop = loader, torch.device(device), size, crop
        self.rajni_sharded = bool(getattr(loader, "rajni_sharded", False))

    def __len__(self):
        return len(self.loader)

    def __iter__(self):
        for frames, labels in self.loader:
            yield gpu_resize_center_crop(frames, self.device, self.size, self.crop), labels


# ------------------------------------------------------------------ GPU JPEG decode (csrc/jpeg.cu) in front of the above
def read_for_gpu_decode(path: str):
    """``ImageFolder`` loader for ``GpuDecodeLoader``: a ``jpeg.JpegFile`` (bytes + parsed headers) when the GPU decoder
    takes the file (host-only header parse), else the frame Pillow decodes (uint8 [H,W,3]) - progressive, CMYK, PNG named
    .JPEG, images above Pillow's pixel limit and the like."""
    from . import jpeg
    with open(path, "rb") as f:
        return jpeg.read_file(f.read())


# The GPU decodes images one sequential decoder per image, so its throughput grows with the images in one launch: the
# loader's batches are decoded in groups of at least this many images (2048 decoders fill a B200's 148 SMs ~14 deep).
DECODE_GROUP_IMAGES = 2048


class GpuDecodeLoader(GpuPreprocessLoader):
    """``GpuPreprocessLoader`` for a loader whose items come from ``read_for_gpu_decode`` (+ ``collate_frames``): the JPEG
    decode runs on ``device`` too (``jpeg.decode_batch``, several loader batches per launch, see DECODE_GROUP_IMAGES),
    so the CPU workers only read files and parse headers.  Same ``(uint8 [B,3,crop,crop] CUDA tensor, labels)`` batches,
    bit for bit."""

    def __iter__(self):
        from . import jpeg, ops
        group, n = [], 0
        it = iter(self.loader)
        while True:
            batch = next(it, None)
            if batch is not None:
                group.append(batch)
                n += len(batch[0])
            if group and (batch is None or n >= DECODE_GROUP_IMAGES):
                frames, meta, max_h = jpeg.decode_batch([x for items, _ in group for x in items], self.device)
                start = 0
                for items, labels in group:
                    yield ops.resize_center_crop(frames, meta[start:start + len(items)], max_h, size=self.size,
                                                 crop=self.crop), labels
                    start += len(items)
                group, n = [], 0
            if batch is None:
                return
