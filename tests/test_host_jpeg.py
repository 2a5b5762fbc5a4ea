"""CPU tests of the GPU JPEG decoder's host side: the numpy oracle (oracle/jpeg_oracle.py) equals Pillow bit for bit on
the supported matrix, and the host-only header parse of librajni_jpeg.so (no CUDA call) takes exactly those files and
leaves the rest - progressive, CMYK, 4:4:0, 4:1:1, PNG bytes, truncated files - to Pillow."""
import io

import numpy as np
import pytest
from PIL import Image

from oracle import jpeg_oracle as jo
from rajni_vit_b200 import jpeg
from tests import jpeg_cases as jc

SMALL = jc.supported_small()
LARGE = jc.supported_large()


def _pillow(data: bytes) -> np.ndarray:
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


@pytest.mark.parametrize("name,data", SMALL, ids=[n for n, _ in SMALL])
def test_oracle_equals_pillow_small(name, data):
    np.testing.assert_array_equal(jo.decode(data), _pillow(data))


@pytest.mark.parametrize("name,data", LARGE, ids=[n for n, _ in LARGE])
def test_oracle_equals_pillow_large(name, data):
    np.testing.assert_array_equal(jo.decode(data), _pillow(data))


def test_host_parse_takes_the_supported_matrix():
    for name, data in SMALL + LARGE:
        info = jpeg.parse(data)
        assert info.gpu == 1, (name, info.why)
        hdr = jo.parse(data)
        assert (info.height, info.width, info.ncomp) == (hdr["h"], hdr["w"], len(hdr["comps"])), name
        assert info.scan_offset == hdr["scan"] and info.restart_interval == hdr["restart"], name
        assert info.why == b""


@pytest.mark.parametrize("name,data", jc.fallbacks(), ids=[n for n, _ in jc.fallbacks()])
def test_host_parse_leaves_the_rest_to_pillow(name, data):
    info = jpeg.parse(data)
    assert info.gpu == 0 and info.why, name
    with pytest.raises(jo.Unsupported):
        jo.parse(data)


def test_malformed_streams_are_found_by_the_oracle():
    """The headers are fine (the GPU takes the files), the entropy-coded data is not: the decoder reports it."""
    for name, data in jc.malformed():
        assert jpeg.parse(data).gpu == 1, name
        with pytest.raises(jo.Malformed):
            jo.decode(data)


def _segments(data: bytes):
    """(offset of the length field, length) of every marker segment before the scan data."""
    out, i = [], 2
    while i + 4 <= len(data) and data[i] == 0xFF:
        n = (data[i + 2] << 8) | data[i + 3]
        out.append((i + 2, n))
        if data[i + 1] == 0xDA:
            break
        i += 2 + n
    return out


def test_parse_never_reads_past_the_bytes():
    """Prefixes of a file that still end in EOI, and files whose segment lengths point outside the bytes or inside other
    segments, parse without a fault: a refusal, or the headers with the scan inside the file."""
    data = jc.pil_jpeg(jc.content(24, 24, "grad"), quality=70, restart_marker_blocks=2)
    scan = jo.parse(data)["scan"]
    for n in range(0, len(data), 3):
        info = jpeg.parse(data[:n] + b"\xff\xd9")
        assert info.gpu == 0 or info.scan_offset <= n + 2, n
    segs = _segments(data)
    assert len(segs) >= 5                                        # APP0, DQT, SOF, DHT, DRI, SOS
    for off, n in segs:
        for bad in (0, 1, 2, n - 1, n + 1, n + 7, 0xFFFF):
            d = bytearray(data)
            d[off], d[off + 1] = bad >> 8, bad & 0xFF
            info = jpeg.parse(bytes(d))
            assert info.gpu == 0 or 0 < info.scan_offset <= len(d), (off, bad)
    assert jpeg.parse(data).scan_offset == scan
    assert jpeg.parse(b"").gpu == 0 and jpeg.parse(b"\xff\xd8\xff").gpu == 0 and jpeg.parse(b"\xff\xd8\xff\xd9").gpu == 0


def _with_size(data: bytes, h: int, w: int) -> bytes:
    i = data.index(b"\xff\xc0")
    d = bytearray(data)
    d[i + 5:i + 9] = bytes([h >> 8, h & 255, w >> 8, w & 255])
    return bytes(d)


def test_images_over_pillows_pixel_limit_are_left_to_pillow():
    """Pillow warns above Image.MAX_IMAGE_PIXELS and raises above twice that: such files take the Pillow path, so the
    warning or the DecompressionBombError is the reference's own (the GPU could decode up to 16384 x 16384)."""
    base = jc.pil_jpeg(jc.content(16, 16, "grad"), quality=80)
    bomb = _with_size(base, 11000, 16384)                        # 180 M pixels > 2 * 89.5 M
    info = jpeg.parse(bomb)
    assert info.gpu == 1 and not jpeg.gpu_takes(info)
    with pytest.raises(Image.DecompressionBombError):
        jpeg.read_file(bomb)
    with pytest.raises(Image.DecompressionBombError):
        jpeg.decode_batch([bomb], "cpu")                         # refused before any device work
    assert jpeg.gpu_takes(jpeg.parse(_with_size(base, 9000, 9000)))
    assert not jpeg.gpu_takes(jpeg.parse(_with_size(base, 9000, 10000)))   # 90 M: Pillow's warning range
    f = jpeg.read_file(base)
    assert isinstance(f, jpeg.JpegFile) and f.info.width == 16 and bytes(f.data.numpy()) == base
