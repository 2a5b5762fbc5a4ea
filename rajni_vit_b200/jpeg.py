"""ctypes binding of librajni_jpeg.so (include/rajni_jpeg.h): GPU JPEG decode for the input pipeline.

``parse`` is host-only (no CUDA call), so data-loader workers use it to decide which files the GPU decodes.
``decode_batch`` turns a batch of such files, plus frames the workers decoded themselves, into the packed frames that
``ops.resize_center_crop`` takes.  Every frame equals ``PIL.Image.open(f).convert("RGB")``: files the GPU does not take,
or finds malformed, are decoded by Pillow, so their errors (e.g. "image file is truncated") are Pillow's own.

These signatures are kept apart from ``_lib.SIGNATURES``, which mirrors include/rajni_b200.h one to one.
"""
from __future__ import annotations

import ctypes
import io
import os
from collections import namedtuple
from ctypes import POINTER, Structure, c_char, c_char_p, c_int, c_longlong, c_size_t, c_ubyte, c_ushort, c_void_p

import numpy as np
import torch

from . import _lib

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "librajni_jpeg.so")
VERSION = 1
OK, SKIPPED, TRUNCATED, BAD_CODE, BAD_RUN, BAD_RESTART = 0, 1, 2, 3, 4, 5


class Info(Structure):
    """struct rajni_jpeg_info"""
    _fields_ = [("gpu", c_int), ("width", c_int), ("height", c_int), ("ncomp", c_int), ("h_samp", c_int), ("v_samp", c_int),
                ("restart_interval", c_int), ("scan_offset", c_longlong), ("file_bytes", c_longlong),
                ("qt", c_int * 3), ("dc", c_int * 3), ("ac", c_int * 3), ("quant", (c_ushort * 64) * 4),
                ("huff_bits", (c_ubyte * 16) * 8), ("huff_vals", (c_ubyte * 256) * 8), ("why", c_char * 64)]


SIGNATURES = {
    "rajni_jpeg_version": (c_int, []),
    "rajni_jpeg_last_error": (c_char_p, []),
    "rajni_jpeg_parse": (c_int, [c_char_p, c_longlong, POINTER(Info)]),
    "rajni_jpeg_workspace_bytes": (c_size_t, [POINTER(Info), c_int]),
    "rajni_jpeg_decode": (c_int, [c_void_p, POINTER(c_longlong), POINTER(Info), c_int, c_void_p, POINTER(c_longlong), c_void_p,
                                  c_size_t, c_void_p]),
    "rajni_jpeg_status": (c_int, [c_void_p, c_int, POINTER(c_int), c_void_p]),
}

_jlib = None


def load() -> ctypes.CDLL:
    """Load the library (once).  Raises if it has not been built - there is no fallback decoder behind it."""
    global _jlib
    if _jlib is not None:
        return _jlib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m rajni_vit_b200.csrc.build`")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.rajni_jpeg_version() != VERSION:
        raise RuntimeError(f"librajni_jpeg.so version {lib.rajni_jpeg_version()} != expected {VERSION}; rebuild")
    _jlib = lib
    return lib


def _check(rc: int) -> None:
    if rc != _lib.RAJNI_OK:
        raise _lib.RajniError(rc, load().rajni_jpeg_last_error().decode("utf-8", "replace"))


# A file the GPU decodes, as a loader worker hands it over: its bytes (uint8 1-D tensor, so that it travels through shared
# memory) and its parsed headers (``Info``), so the main process does not parse it again.
JpegFile = namedtuple("JpegFile", "data info")


def parse(data: bytes) -> Info:
    """Headers of one file (host only).  ``.gpu`` says whether the GPU decodes it, ``.why`` why not."""
    data = bytes(data)
    info = Info()
    load().rajni_jpeg_parse(data, len(data), ctypes.byref(info))
    return info


def gpu_takes(info: Info) -> bool:
    """The GPU decodes the file: ``parse`` took it and Pillow would open it without its decompression-bomb warning or
    error (``Image.MAX_IMAGE_PIXELS``), which larger images keep by going through Pillow."""
    from PIL import Image
    limit = Image.MAX_IMAGE_PIXELS
    return bool(info.gpu) and (limit is None or info.width * info.height <= limit)


def read_file(data: bytes):
    """A loader worker's item for ``decode_batch``: a ``JpegFile`` when the GPU decodes the file, else Pillow's frame."""
    info = parse(data)
    if gpu_takes(info):
        return JpegFile(torch.frombuffer(bytearray(data), dtype=torch.uint8), info)
    return pil_frame(data)


def pil_frame(data: bytes) -> torch.Tensor:
    """``PIL.Image.open(f).convert("RGB")`` of the file's bytes as a uint8 [H,W,3] tensor (what the reference's loader
    decodes; its errors propagate)."""
    from PIL import Image
    with Image.open(io.BytesIO(data)) as im:
        return torch.from_numpy(np.asarray(im.convert("RGB")).copy())


def decode_batch(items, device, return_status: bool = False):
    """A batch of loader items -> ``(frames, meta, max_h)`` for ``ops.resize_center_crop``: frames a 1-D uint8 CUDA tensor
    of the HWC frames back to back, meta int64 [B,3] = (byte offset, H, W) on ``device``.

    Each item is a ``JpegFile`` (``read_file``), the bytes of a file (decoded on the GPU when ``gpu_takes`` it, by Pillow
    otherwise) or a frame a worker already decoded (uint8 [H,W,3]).  All bytes travel in one pinned buffer and one host-to-device copy; the
    per-image statuses are read once and the files the GPU found malformed are decoded again by Pillow.
    ``return_status``: also return the per-item RAJNI_JPEG_* status list (SKIPPED for items the GPU did not decode)."""
    device = torch.device(device)
    lib = load()
    B = len(items)
    infos = (Info * B)()
    files, frames = {}, {}                       # batch index -> bytes / host frame
    for b, it in enumerate(items):
        if isinstance(it, JpegFile):
            infos[b] = it.info
            files[b] = it.data.numpy()
            continue
        if isinstance(it, torch.Tensor):
            if it.dtype != torch.uint8 or it.dim() != 3 or it.shape[2] != 3:
                raise ValueError(f"item {b}: expected file bytes or a uint8 [H,W,3] frame, got {it.dtype} {tuple(it.shape)}")
            frames[b] = it
            continue
        data = bytes(it)
        lib.rajni_jpeg_parse(data, len(data), ctypes.byref(infos[b]))
        if gpu_takes(infos[b]):
            files[b] = np.frombuffer(data, np.uint8)
        else:
            infos[b].gpu = 0
            frames[b] = pil_frame(data)
    meta_np = np.empty((B, 3), dtype=np.int64)
    off = 0
    for b in range(B):
        h, w = (infos[b].height, infos[b].width) if b in files else frames[b].shape[:2]
        meta_np[b] = off, h, w
        off += h * w * 3
    meta = torch.from_numpy(meta_np)
    # one pinned staging buffer: the files, then the frames decoded on the host
    src_off, n = {}, 0
    for b, d in files.items():
        src_off[b], n = n, n + len(d)
    for b, f in frames.items():
        src_off[b], n = n, n + f.numel()
    host = torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    for b, d in files.items():
        hv[src_off[b]:src_off[b] + len(d)] = d
    for b, f in frames.items():
        hv[src_off[b]:src_off[b] + f.numel()] = f.reshape(-1).numpy()
    src = host.to(device, non_blocking=True)
    out = torch.empty(max(off, 1), dtype=torch.uint8, device=device)
    for b, f in frames.items():
        out[meta[b, 0]:meta[b, 0] + f.numel()].copy_(src[src_off[b]:src_off[b] + f.numel()])
    status = [SKIPPED] * B
    if files:
        stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        nbytes = int(lib.rajni_jpeg_workspace_bytes(infos, B))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
        file_offs = (c_longlong * B)(*[src_off.get(b, 0) for b in range(B)])
        frame_offs = (c_longlong * B)(*meta_np[:, 0].tolist())
        with torch.cuda.device(device):
            _check(lib.rajni_jpeg_decode(src.data_ptr(), file_offs, infos, B, out.data_ptr(), frame_offs, ws.data_ptr(), nbytes, stream))
            st = (c_int * B)()
            _check(lib.rajni_jpeg_status(ws.data_ptr(), B, st, stream))
        status = list(st)
        for b in files:
            if status[b] != OK:
                f = pil_frame(files[b].tobytes())    # Pillow's frame, or Pillow's error
                if tuple(f.shape[:2]) != (int(meta[b, 1]), int(meta[b, 2])):
                    raise ValueError(f"item {b}: Pillow decodes {tuple(f.shape[:2])}, the headers say {tuple(meta[b, 1:].tolist())}")
                out[meta[b, 0]:meta[b, 0] + f.numel()].copy_(f.reshape(-1).to(device))
    res = (out, meta.to(device, non_blocking=True), int(meta[:, 1].max()))
    return res + (status,) if return_status else res
