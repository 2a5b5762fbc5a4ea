"""CPU ORACLE (TEST INFRASTRUCTURE ONLY) for the GPU JPEG decoder (``csrc/jpeg.cu``).

``PIL.Image.open(f).convert("RGB")`` decodes a baseline JPEG with libjpeg(-turbo) at its defaults: Huffman decoding,
the ``ISLOW`` integer IDCT (``jidctint.c``: CONST_BITS 13, PASS1_BITS 2, 64-bit intermediates), the post-IDCT range
limit (``jdmaster.c``: mask to 10 bits, then a table that is a clamp of the sign-extended value plus 128), "fancy"
triangle upsampling of the chroma planes (``jdsample.c``: h2v1 and h2v2, plain replication when the chroma plane is at
most 2 samples wide; context rows replicated at the top and bottom of the plane) and the fixed-point YCbCr -> RGB tables
of ``jdcolor.c``.  Grayscale becomes R = G = B = Y, as ``convert("RGB")`` does.

This file restates that for the subset the GPU decodes (``classify``), integer for integer, so that the CUDA kernels can
be checked against it and it can be checked against Pillow (``tests/test_host_jpeg.py``).  Files outside the subset
raise ``Unsupported``; a stream the decoder finds malformed raises ``Malformed`` (the GPU reports those as a status and
Pillow decodes them).
"""
from __future__ import annotations

import numpy as np

# jpeg_natural_order: zig-zag index -> natural (row-major) index
ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63], dtype=np.int64)

MAX_SIDE = 16384


class Unsupported(ValueError):
    """The file is not in the subset the GPU decodes (or is not a JPEG at all)."""


class Malformed(ValueError):
    """The entropy-coded data is not a valid stream for the headers."""


def _u16(d, i):
    if i + 2 > len(d):
        raise Unsupported("truncated header")
    return (d[i] << 8) | d[i + 1]


def parse(data: bytes) -> dict:
    """Headers of a JPEG up to its first SOS -> the fields the decoder needs; ``Unsupported`` for anything outside the
    GPU subset (progressive, arithmetic, 12-bit, lossless, CMYK/YCCK, RGB, 4:4:0 / 4:1:1 / other sampling, multi-scan,
    missing tables, not a JPEG)."""
    d = bytes(data)
    if len(d) < 4 or d[0] != 0xFF or d[1] != 0xD8:
        raise Unsupported("not a JPEG (no SOI)")
    if d[-2] != 0xFF or d[-1] != 0xD9:
        raise Unsupported("no EOI at the end (truncated?)")
    i = 2
    qt, dc, ac = {}, {}, {}
    frame = None
    jfif = adobe = False
    transform = -1
    restart = 0
    while True:
        # next marker: skip anything up to 0xFF, then fill bytes (libjpeg's next_marker)
        while i < len(d) and d[i] != 0xFF:
            i += 1
        while i < len(d) and d[i] == 0xFF:
            i += 1
        if i >= len(d):
            raise Unsupported("no scan before the end of the file")
        m = d[i]
        i += 1
        if m == 0xD8 or m == 0xD9:
            raise Unsupported("SOI/EOI before the scan")
        if 0xD0 <= m <= 0xD7 or m == 0x01:
            continue
        n = _u16(d, i)
        if n < 2 or i + n > len(d):
            raise Unsupported("truncated segment")
        seg = d[i + 2:i + n]
        i += n
        if m in (0xC0, 0xC1):
            if frame is not None or len(seg) < 6:
                raise Unsupported("bad SOF")
            p, h, w, nc = seg[0], (seg[1] << 8) | seg[2], (seg[3] << 8) | seg[4], seg[5]
            if p != 8:
                raise Unsupported(f"{p}-bit samples")
            if h == 0 or w == 0 or h > MAX_SIDE or w > MAX_SIDE:
                raise Unsupported(f"size {w}x{h}")
            if nc not in (1, 3) or len(seg) < 6 + 3 * nc:
                raise Unsupported(f"{nc} components")
            comps = [dict(id=seg[6 + 3 * c], h=seg[7 + 3 * c] >> 4, v=seg[7 + 3 * c] & 15, tq=seg[8 + 3 * c]) for c in range(nc)]
            frame = dict(h=h, w=w, comps=comps)
        elif 0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC):
            raise Unsupported(f"SOF{m - 0xC0} (progressive, lossless or arithmetic)")
        elif m == 0xCC:
            raise Unsupported("arithmetic conditioning (DAC)")
        elif m == 0xDB:
            j = 0
            while j < len(seg):
                pq, tq = seg[j] >> 4, seg[j] & 15
                size = 128 if pq else 64
                if tq > 3 or pq > 1 or j + 1 + size > len(seg):
                    raise Unsupported("bad DQT")
                raw = seg[j + 1:j + 1 + size]
                vals = [(raw[2 * k] << 8) | raw[2 * k + 1] for k in range(64)] if pq else list(raw)
                q = np.zeros(64, np.int64)
                q[ZIGZAG] = vals
                qt[tq] = q
                j += 1 + size
        elif m == 0xC4:
            j = 0
            while j < len(seg):
                if j + 17 > len(seg):
                    raise Unsupported("bad DHT")
                tc, th = seg[j] >> 4, seg[j] & 15
                bits = list(seg[j + 1:j + 17])
                cnt = sum(bits)
                if tc > 1 or th > 3 or cnt > 256 or j + 17 + cnt > len(seg):
                    raise Unsupported("bad DHT")
                vals = list(seg[j + 17:j + 17 + cnt])
                (ac if tc else dc)[th] = _huff_table(bits, vals, tc == 0)
                j += 17 + cnt
        elif m == 0xDD:
            if len(seg) < 2:
                raise Unsupported("bad DRI")
            restart = (seg[0] << 8) | seg[1]
        elif m == 0xE0:
            if len(seg) >= 14 and seg[:5] == b"JFIF\0":
                jfif = True
        elif m == 0xEE:
            if len(seg) >= 12 and seg[:5] == b"Adobe":
                adobe, transform = True, seg[11]
        elif m == 0xDA:
            if frame is None:
                raise Unsupported("SOS before SOF")
            ns = seg[0] if seg else 0
            comps = frame["comps"]
            if ns != len(comps) or len(seg) < 4 + 2 * ns:
                raise Unsupported("the first scan does not hold every component (multi-scan)")
            for c in range(ns):
                cid, t = seg[1 + 2 * c], seg[2 + 2 * c]
                if cid != comps[c]["id"]:
                    raise Unsupported("scan component order")
                comps[c]["td"], comps[c]["ta"] = t >> 4, t & 15
            ss, se, ahal = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns]
            if ss != 0 or se != 63 or ahal != 0:
                raise Unsupported("not a sequential scan")
            break
        # APPn, COM and anything else: skipped
    if len(comps) == 3:
        ids = [c["id"] for c in comps]
        if jfif:
            ycc = True
        elif adobe:
            if transform != 1:
                raise Unsupported("Adobe RGB / unknown transform")
            ycc = True
        else:
            ycc = ids != [82, 71, 66]
        if not ycc:
            raise Unsupported("RGB components")
        if [(c["h"], c["v"]) for c in comps[1:]] != [(1, 1), (1, 1)] or (comps[0]["h"], comps[0]["v"]) not in ((1, 1), (2, 1), (2, 2)):
            raise Unsupported("sampling " + " ".join(f"{c['h']}x{c['v']}" for c in comps))
    else:
        if not (1 <= comps[0]["h"] <= 4 and 1 <= comps[0]["v"] <= 4):
            raise Unsupported("bad sampling factor")
    for c in comps:
        if c["tq"] not in qt or c["td"] not in dc or c["ta"] not in ac:
            raise Unsupported("a table the scan uses is not defined")
        c["q"], c["dc"], c["ac"] = qt[c["tq"]], dc[c["td"]], ac[c["ta"]]
    return dict(h=frame["h"], w=frame["w"], comps=comps, restart=restart, scan=i, data=d)


def _huff_table(bits, vals, is_dc):
    """jpeg_make_d_derived_tbl: canonical codes -> {(length, code): symbol}; invalid tables are Unsupported."""
    codes = {}
    code, k = 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[(length, code)] = vals[k]
            code += 1
            k += 1
        if code >= (1 << length):          # no code may be all ones
            raise Unsupported("bad Huffman table")
        code <<= 1
    if is_dc and any(v > 15 for v in vals):
        raise Unsupported("bad DC Huffman table")
    return codes


class _Bits:
    """MSB-first bit reader over entropy-coded data: 0xFF 0x00 -> 0xFF, a marker ends the data (zeros follow)."""

    def __init__(self, d, pos):
        self.d, self.pos, self.acc, self.n, self.fake, self.marker = d, pos, 0, 0, 0, False

    def _byte(self):
        d = self.d
        if self.marker or self.pos >= len(d):
            self.fake += 8
            return 0
        c = d[self.pos]
        if c != 0xFF:
            self.pos += 1
            return c
        j = self.pos + 1
        while j < len(d) and d[j] == 0xFF:
            j += 1
        if j < len(d) and d[j] == 0:
            self.pos = j + 1
            return 0xFF
        self.marker = True        # pos stays on the marker's first 0xFF
        self.fake += 8
        return 0

    def get(self, k):
        while self.n < k:
            self.acc = (self.acc << 8) | self._byte()
            self.n += 8
        self.n -= k
        v = (self.acc >> self.n) & ((1 << k) - 1)
        self.acc &= (1 << self.n) - 1
        if self.n < self.fake:     # consumed bits that are not in the file
            raise Malformed("entropy-coded data ends early")
        self.fake = min(self.fake, self.n)
        return v

    def huff(self, table):
        code = 0
        for length in range(1, 17):
            code = (code << 1) | self.get(1)
            s = table.get((length, code))
            if s is not None:
                return s
        raise Malformed("invalid Huffman code")

    def restart(self, num):
        self.acc = self.n = self.fake = 0
        self.marker = False
        d, j = self.d, self.pos
        if j >= len(d) or d[j] != 0xFF:
            raise Malformed("data before a restart marker")
        while j < len(d) and d[j] == 0xFF:
            j += 1
        if j >= len(d) or d[j] != 0xD0 + (num & 7):
            raise Malformed("missing restart marker")
        self.pos = j + 1


def _extend(v, s):
    return v - (1 << s) + 1 if s and v < (1 << (s - 1)) else v


def layout(hdr):
    """Block grid per component: (blocks wide, blocks high) as stored, MCU grid, max sampling factors."""
    comps = hdr["comps"]
    if len(comps) == 1:
        bw, bh = -(-hdr["w"] // 8), -(-hdr["h"] // 8)
        return [(bw, bh)], (bw, bh), (1, 1)
    hm, vm = comps[0]["h"], comps[0]["v"]
    mx, my = -(-hdr["w"] // (8 * hm)), -(-hdr["h"] // (8 * vm))
    return [(mx * c["h"], my * c["v"]) for c in comps], (mx, my), (hm, vm)


def entropy_decode(hdr):
    """-> list of int16 coefficient arrays [bh, bw, 64] (natural order), one per component."""
    comps = hdr["comps"]
    grids, (mx, my), _ = layout(hdr)
    coef = [np.zeros((bh, bw, 64), np.int16) for bw, bh in grids]
    bits = _Bits(hdr["data"], hdr["scan"])
    pred = [0] * len(comps)
    restart, rst_num = hdr["restart"], 0
    nmcu = mx * my
    for m in range(nmcu):
        if restart and m and m % restart == 0:
            bits.restart(rst_num)
            rst_num += 1
            pred = [0] * len(comps)
        ux, uy = m % mx, m // mx
        for ci, c in enumerate(comps):
            hs, vs = (c["h"], c["v"]) if len(comps) > 1 else (1, 1)
            for by in range(vs):
                for bx in range(hs):
                    blk = coef[ci][uy * vs + by, ux * hs + bx]
                    s = bits.huff(c["dc"])
                    diff = _extend(bits.get(s), s) if s else 0
                    pred[ci] += diff
                    blk[0] = np.int64(pred[ci]).astype(np.int16)
                    k = 1
                    while k < 64:
                        rs = bits.huff(c["ac"])
                        r, s = rs >> 4, rs & 15
                        if s:
                            k += r
                            if k > 63:
                                raise Malformed("AC run past the block")
                            blk[ZIGZAG[k]] = np.int64(_extend(bits.get(s), s)).astype(np.int16)
                            k += 1
                        elif r == 15:
                            k += 16
                        else:
                            break
    # the last MCU must not have used bits past the data (checked by get()); nothing after it is read
    return coef


C13, P2 = 13, 2
FIX = dict(f0_298=2446, f0_390=3196, f0_541=4433, f0_765=6270, f0_899=7373, f1_175=9633, f1_501=12299, f1_847=15137,
           f1_961=16069, f2_053=16819, f2_562=20995, f3_072=25172)


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _idct_1d(s0, s1, s2, s3, s4, s5, s6, s7):
    """jpeg_idct_islow's butterfly on int64 arrays; returns the 8 undescaled outputs."""
    z1 = (s2 + s6) * FIX["f0_541"]
    tmp2 = z1 + s6 * -FIX["f1_847"]
    tmp3 = z1 + s2 * FIX["f0_765"]
    tmp0 = (s0 + s4) << C13
    tmp1 = (s0 - s4) << C13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    tmp0, tmp1, tmp2, tmp3 = s7, s5, s3, s1
    z1, z2, z3, z4 = tmp0 + tmp3, tmp1 + tmp2, tmp0 + tmp2, tmp1 + tmp3
    z5 = (z3 + z4) * FIX["f1_175"]
    tmp0 = tmp0 * FIX["f0_298"]
    tmp1 = tmp1 * FIX["f2_053"]
    tmp2 = tmp2 * FIX["f3_072"]
    tmp3 = tmp3 * FIX["f1_501"]
    z1 = z1 * -FIX["f0_899"]
    z2 = z2 * -FIX["f2_562"]
    z3 = z3 * -FIX["f1_961"] + z5
    z4 = z4 * -FIX["f0_390"] + z5
    tmp0 += z1 + z3
    tmp1 += z2 + z4
    tmp2 += z2 + z3
    tmp3 += z1 + z4
    return [t10 + tmp3, t11 + tmp2, t12 + tmp1, t13 + tmp0, t13 - tmp0, t12 - tmp1, t11 - tmp2, t10 - tmp3]


def idct_islow(coef, q):
    """int16 [..., 64] natural-order coefficients, quant table [64] -> uint8 [..., 8, 8] samples."""
    c = coef.astype(np.int64).reshape(-1, 8, 8) * q.reshape(8, 8)
    # pass 1: columns -> int32 workspace (the C code casts the descaled value to int)
    cols = _idct_1d(*[c[:, k, :] for k in range(8)])
    ws = np.stack([_descale(v, C13 - P2).astype(np.int32).astype(np.int64) for v in cols], axis=1)   # [n, row, col]
    rows = _idct_1d(*[ws[:, :, k] for k in range(8)])
    out = np.stack([_descale(v, C13 + P2 + 3) for v in rows], axis=2)                                # [n, row, col]
    x = (out & 1023).astype(np.int64)
    x = np.where(x < 512, x, x - 1024) + 128
    return np.clip(x, 0, 255).astype(np.uint8).reshape(coef.shape[:-1] + (8, 8))


def planes(hdr, coef):
    """IDCT of every block -> one uint8 sample plane per component, [bh*8, bw*8]."""
    out = []
    for ci, c in enumerate(hdr["comps"]):
        px = idct_islow(coef[ci], c["q"])                       # [bh, bw, 8, 8]
        bh, bw = px.shape[:2]
        out.append(px.transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8))
    return out


def _fancy_h2v1(p, cw):
    p = p[:, :cw].astype(np.int32)
    out = np.empty((p.shape[0], 2 * cw), np.int32)
    if cw <= 2:
        return np.repeat(p, 2, axis=1)
    left = np.concatenate([p[:, :1], p[:, :-1]], axis=1)
    right = np.concatenate([p[:, 1:], p[:, -1:]], axis=1)
    out[:, 0::2] = (3 * p + left + 1) >> 2
    out[:, 1::2] = (3 * p + right + 2) >> 2
    out[:, 0] = p[:, 0]
    out[:, -1] = p[:, -1]
    return out


def _fancy_h2v2(p, cw, ch):
    p = p[:ch, :cw].astype(np.int32)
    if cw <= 2:
        return np.repeat(np.repeat(p, 2, axis=0), 2, axis=1)
    up = np.concatenate([p[:1], p[:-1]], axis=0)
    down = np.concatenate([p[1:], p[-1:]], axis=0)
    out = np.empty((2 * ch, 2 * cw), np.int32)
    for r0, nb in ((0, up), (1, down)):
        cs = 3 * p + nb                                          # column sums with the nearer neighbour row
        left = np.concatenate([cs[:, :1], cs[:, :-1]], axis=1)
        right = np.concatenate([cs[:, 1:], cs[:, -1:]], axis=1)
        rows = np.empty((ch, 2 * cw), np.int32)
        rows[:, 0::2] = (3 * cs + left + 8) >> 4
        rows[:, 1::2] = (3 * cs + right + 7) >> 4
        rows[:, 0] = (4 * cs[:, 0] + 8) >> 4
        rows[:, -1] = (4 * cs[:, -1] + 7) >> 4
        out[r0::2] = rows
    return out


def _tables():
    x = np.arange(256, dtype=np.int64) - 128
    one_half = 1 << 15

    def fix(v):
        return int(v * 65536 + 0.5)
    cr_r = (fix(1.40200) * x + one_half) >> 16
    cb_b = (fix(1.77200) * x + one_half) >> 16
    cr_g = -fix(0.71414) * x
    cb_g = -fix(0.34414) * x + one_half
    return cr_r, cb_b, cr_g, cb_g


def color(hdr, pl):
    """Sample planes -> uint8 [H, W, 3]."""
    h, w, comps = hdr["h"], hdr["w"], hdr["comps"]
    y = pl[0][:h, :w].astype(np.int64)
    if len(comps) == 1:
        return np.repeat(y[:, :, None].astype(np.uint8), 3, axis=2)
    hm, vm = comps[0]["h"], comps[0]["v"]
    cw, ch = -(-w // hm), -(-h // vm)
    if hm == 1:
        cb, cr = pl[1][:h, :w], pl[2][:h, :w]
    elif vm == 1:
        cb, cr = (_fancy_h2v1(p[:h], cw)[:, :w] for p in pl[1:])
    else:
        cb, cr = (_fancy_h2v2(p, cw, ch)[:h, :w] for p in pl[1:])
    cb, cr = cb.astype(np.int64), cr.astype(np.int64)
    cr_r, cb_b, cr_g, cb_g = _tables()
    r = y + cr_r[cr]
    g = y + ((cb_g[cb] + cr_g[cr]) >> 16)
    b = y + cb_b[cb]
    return np.clip(np.stack([r, g, b], axis=2), 0, 255).astype(np.uint8)


def decode(data: bytes) -> np.ndarray:
    """A JPEG in the GPU subset -> uint8 [H, W, 3], equal to ``PIL.Image.open(f).convert("RGB")``."""
    hdr = parse(data)
    return color(hdr, planes(hdr, entropy_decode(hdr)))
