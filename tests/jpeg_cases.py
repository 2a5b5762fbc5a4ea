"""Seeded JPEG files for the GPU decoder's tests (tests/test_host_jpeg.py, tests/test_gpu_jpeg.py), all made here with
Pillow and OpenCV: the supported matrix, the files the decoder must leave to Pillow, and malformed streams."""
from __future__ import annotations

import io

import numpy as np
from PIL import Image

SMALL_SIZES = [(1, 1), (1, 17), (17, 1), (2, 3), (7, 9), (8, 8), (15, 17), (16, 16), (33, 47)]      # (h, w)
LARGE_SIZES = [(224, 224), (375, 500), (500, 375), (16, 2048)]
QUALITIES = [10, 35, 60, 85, 95, 100]


def content(h: int, w: int, kind: str, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[0:h, 0:w]
    if kind == "grad":
        a = np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) * 7 % 256], axis=2)
        return a.astype(np.uint8)
    if kind == "flat":
        return np.full((h, w, 3), (200, 30, 90), np.uint8)
    # "texture": gradients, stripes and noise, the bulk of a natural image's bits
    a = np.stack([(x * 3 + y) % 256, np.sin(x / 7.0) * 100 + 128, (y * 2) % 256], axis=2) + rng.normal(0, 20, (h, w, 3))
    return np.clip(a, 0, 255).astype(np.uint8)


def pil_jpeg(a: np.ndarray, gray: bool = False, **kw) -> bytes:
    im = Image.fromarray(a)
    b = io.BytesIO()
    (im.convert("L") if gray else im).save(b, "JPEG", **kw)
    return b.getvalue()


def cv2_jpeg(a: np.ndarray, quality: int, sampling: str, rst: int = 0) -> bytes:
    import cv2
    sf = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
          "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
          "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}[sampling]
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(a[:, :, ::-1]),
                           [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
    assert ok
    return enc.tobytes()


def supported_small():
    """(name, bytes): every small size x content x 4:4:4 / 4:2:2 / 4:2:0 and grayscale, qualities 10..100."""
    out = []
    i = 0
    for h, w in SMALL_SIZES:
        for kind in ("noise", "grad", "flat"):
            a = content(h, w, kind, seed=i)
            for ss in (0, 1, 2):
                q = QUALITIES[i % len(QUALITIES)]
                out.append((f"pil-{h}x{w}-{kind}-ss{ss}-q{q}", pil_jpeg(a, quality=q, subsampling=ss)))
                i += 1
            q = QUALITIES[i % len(QUALITIES)]
            out.append((f"pil-{h}x{w}-{kind}-gray-q{q}", pil_jpeg(a, gray=True, quality=q)))
            i += 1
    return out


def supported_large():
    """(name, bytes): the larger sizes with Pillow (optimized tables, restart markers) and OpenCV (444/422/420 + RST)."""
    out = []
    for j, (h, w) in enumerate(LARGE_SIZES):
        a = content(h, w, "texture", seed=100 + j)
        out.append((f"pil-{h}x{w}-q90-420", pil_jpeg(a, quality=90, subsampling=2)))
        out.append((f"pil-{h}x{w}-q75-444-opt", pil_jpeg(a, quality=75, subsampling=0, optimize=True)))
        out.append((f"pil-{h}x{w}-q95-422-rst3", pil_jpeg(a, quality=95, subsampling=1, restart_marker_blocks=3)))
        out.append((f"pil-{h}x{w}-q50-gray-rst1", pil_jpeg(a, gray=True, quality=50, restart_marker_blocks=1)))
        for k, sf in enumerate(("444", "422", "420")):
            out.append((f"cv2-{h}x{w}-{sf}-rst{k * 4}", cv2_jpeg(a, quality=(20, 85, 100)[k], sampling=sf, rst=k * 4)))
    return out


def fallbacks():
    """(name, bytes): files the GPU decoder must leave to Pillow."""
    a = content(40, 56, "texture", seed=7)
    prog = pil_jpeg(a, quality=80, progressive=True)
    b = io.BytesIO()
    Image.fromarray(a).convert("CMYK").save(b, "JPEG", quality=80)
    cmyk = b.getvalue()
    b = io.BytesIO()
    Image.fromarray(a).save(b, "PNG")
    png = b.getvalue()
    base = pil_jpeg(a, quality=80)
    return [("progressive", prog), ("cmyk", cmyk), ("440", cv2_jpeg(a, 80, "440")), ("411", cv2_jpeg(a, 80, "411")),
            ("png", png), ("truncated-scan", base[:len(base) * 2 // 3]), ("truncated-header", base[:120])]


def scan_start(data: bytes) -> int:
    """Offset of the first byte after the SOS segment."""
    i = data.index(b"\xff\xda")
    return i + 2 + ((data[i + 2] << 8) | data[i + 3])


def malformed():
    """(name, bytes): files whose headers the GPU takes but whose entropy-coded data is broken (EOI still at the end):
    the scan cut short, and a run of ones no Huffman code matches."""
    a = content(64, 80, "texture", seed=9)
    base = pil_jpeg(a, quality=85)
    s = scan_start(base)
    cut = base[:s + (len(base) - s) // 3] + b"\xff\xd9"
    ones = b"\xff\x00" * 8
    bad = base[:s + 40] + ones + base[s + 40 + len(ones):]
    return [("cut-scan", cut), ("bad-code", bad)]
