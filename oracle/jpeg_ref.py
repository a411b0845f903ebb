"""Reference baseline JPEG decoder in numpy / pure Python: what cv2.imdecode(buf, cv2.IMREAD_COLOR) computes for the streams
that csrc/jpeg.cu decodes on the device (SOF0/SOF1, 8-bit, gray or YCbCr 4:4:4 / 4:2:2 / 4:2:0, one interleaved scan).

It restates, step for step, the published libjpeg(-turbo) algorithms the kernels follow:
  * Huffman decoding with 0xFF00 unstuffing, DC prediction and restart intervals (ITU T.81 F.2.2, jdhuff.c);
  * jpeg_idct_islow (jidctint.c): 13-bit constants, PASS1_BITS 2, DESCALE, and the post-IDCT range-limit table
    (idct_range_limit below);
  * h2v1 / h2v2 "fancy" (triangle) upsampling with edge replication (jdsample.c; the first / last row context of
    jdmainct.c), box replication when the downsampled width is 2 or less;
  * ycc_rgb_convert's fixed-point tables (jdcolor.c build_ycc_rgb_table), BGR output; gray replicated to B = G = R.
Slow (pure Python bit reader): for small test images only.
"""
import struct

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                   60, 61, 54, 47, 55, 62, 63], np.int64)       # zigzag index -> natural (row-major) index


class JpegRefError(ValueError):
    pass


def _segments(data):
    """(marker, payload offset, payload bytes) up to and including SOS, then the entropy-coded range."""
    if data[:2] != b"\xff\xd8":
        raise JpegRefError("no SOI")
    pos, out = 2, []
    while True:
        while pos < len(data) and data[pos] == 0xFF and pos + 1 < len(data) and data[pos + 1] == 0xFF:
            pos += 1
        if pos + 4 > len(data) or data[pos] != 0xFF:
            raise JpegRefError("bad marker at %d" % pos)
        m = data[pos + 1]
        L = struct.unpack(">H", data[pos + 2:pos + 4])[0]
        out.append((m, pos + 4, L - 2))
        pos += 2 + L
        if m == 0xDA:
            return out, pos


def parse(data):
    data = bytes(data)
    segs, scan = _segments(data)
    q, huff, ri, sof, sos = {}, {}, 0, None, None
    for m, o, n in segs:
        p = data[o:o + n]
        if m == 0xDB:
            i = 0
            while i < n:
                pq, tq = p[i] >> 4, p[i] & 15
                if pq:
                    vals = struct.unpack(">64H", p[i + 1:i + 129]); i += 129
                else:
                    vals = tuple(p[i + 1:i + 65]); i += 65
                t = np.zeros(64, np.int64)
                t[ZIGZAG] = vals
                q[tq] = t
        elif m == 0xC4:
            i = 0
            while i < n:
                tc, th = p[i] >> 4, p[i] & 15
                counts = list(p[i + 1:i + 17])
                vals = list(p[i + 17:i + 17 + sum(counts)])
                i += 17 + sum(counts)
                huff[(tc, th)] = _derive(counts, vals)
        elif m == 0xDD:
            ri = struct.unpack(">H", p[:2])[0]
        elif m in (0xC0, 0xC1):
            H, W = struct.unpack(">HH", p[1:5])
            comps = [(p[6 + 3 * k], p[7 + 3 * k] >> 4, p[7 + 3 * k] & 15, p[8 + 3 * k]) for k in range(p[5])]
            sof = (H, W, comps)
        elif m == 0xDA:
            sos = [(p[1 + 2 * k], p[2 + 2 * k] >> 4, p[2 + 2 * k] & 15) for k in range(p[0])]
    if sof is None or sos is None:
        raise JpegRefError("no SOF0/SOF1 or SOS")
    return data, q, huff, ri, sof, sos, scan


def _derive(counts, vals):
    """{(length, code): symbol} of a canonical Huffman table (T.81 Annex C)."""
    table, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(counts[length - 1]):
            table[(length, code)] = vals[k]
            code += 1; k += 1
        code <<= 1
    return table


class _Bits:
    """MSB-first bit reader over the entropy-coded bytes; 0xFF00 -> 0xFF; a marker or the end yields zero bits (and is
    remembered: the device flags a frame that consumes them)."""

    def __init__(self, data, pos):
        self.data, self.pos, self.acc, self.n, self.past_end = data, pos, 0, 0, False

    def bit(self):
        if self.n == 0:
            b = 0
            if self.pos < len(self.data) and not self.past_end:
                b = self.data[self.pos]
                if b == 0xFF:
                    if self.pos + 1 < len(self.data) and self.data[self.pos + 1] == 0:
                        self.pos += 2
                    else:
                        b, self.past_end = 0, True
                else:
                    self.pos += 1
            else:
                self.past_end = True
            self.acc, self.n = b, 8
        self.n -= 1
        return (self.acc >> self.n) & 1

    def bits(self, k):
        v = 0
        for _ in range(k):
            v = (v << 1) | self.bit()
        return v

    def restart(self):
        """Discards the partial byte and expects RSTn."""
        self.n = 0
        if self.data[self.pos] != 0xFF or not (0xD0 <= self.data[self.pos + 1] <= 0xD7):
            raise JpegRefError("missing restart marker")
        self.pos += 2


def _huff(bits, table):
    code = 0
    for length in range(1, 17):
        code = (code << 1) | bits.bit()
        s = table.get((length, code))
        if s is not None:
            return s
    raise JpegRefError("bad Huffman code")


def _extend(v, s):
    return v - (1 << s) + 1 if s and v < (1 << (s - 1)) else v


def entropy_decode(parsed):
    """Quantised coefficients in natural order: one int64 array [rows, cols, 64] of blocks per component."""
    data, q, huff, ri, (H, W, comps), sos, pos = parsed
    if len(comps) == 1:
        hs, vs = [1], [1]
        mcux, mcuy = -(-W // 8), -(-H // 8)
    else:
        hs, vs = [c[1] for c in comps], [c[2] for c in comps]
        hmax, vmax = max(hs), max(vs)
        mcux, mcuy = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    coefs = [np.zeros((mcuy * v, mcux * h, 64), np.int64) for h, v in zip(hs, vs)]
    tables = {cid: (huff[(0, td)], huff[(1, ta)]) for cid, td, ta in sos}
    bits = _Bits(data, pos)
    pred = [0] * len(comps)
    for m in range(mcux * mcuy):
        if ri and m and m % ri == 0:
            bits.restart()
            pred = [0] * len(comps)
        my, mx = divmod(m, mcux)
        for ci, (cid, _, _, _) in enumerate(comps):
            dc_t, ac_t = tables[cid]
            for v in range(vs[ci]):
                for h in range(hs[ci]):
                    blk = coefs[ci][my * vs[ci] + v, mx * hs[ci] + h]
                    s = _huff(bits, dc_t)
                    pred[ci] += _extend(bits.bits(s), s)
                    blk[0] = pred[ci]
                    k = 1
                    while k < 64:
                        rs = _huff(bits, ac_t)
                        r, s = rs >> 4, rs & 15
                        if s:
                            k += r
                            if k > 63:
                                raise JpegRefError("coefficient index past 63")
                            blk[ZIGZAG[k]] = _extend(bits.bits(s), s)
                            k += 1
                        elif r == 15:
                            k += 16
                        else:
                            break
    if bits.past_end:
        raise JpegRefError("entropy-coded data ends before the last MCU")
    return coefs


# ---- jpeg_idct_islow ----------------------------------------------------------------------------------------------------
CONST_BITS, PASS1_BITS = 13, 2
F = dict(c0_298631336=2446, c0_390180644=3196, c0_541196100=4433, c0_765366865=6270, c0_899976223=7373, c1_175875602=9633,
         c1_501321110=12299, c1_847759065=15137, c1_961570560=16069, c2_053119869=16819, c2_562915447=20995,
         c3_072711026=25172)


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _idct_1d(s0, s1, s2, s3, s4, s5, s6, s7):
    """The even / odd butterfly of jpeg_idct_islow, on int64 arrays; returns the 8 outputs before descaling."""
    z1 = (s2 + s6) * F["c0_541196100"]
    tmp2 = z1 + s6 * -F["c1_847759065"]
    tmp3 = z1 + s2 * F["c0_765366865"]
    tmp0 = (s0 + s4) << CONST_BITS
    tmp1 = (s0 - s4) << CONST_BITS
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    t0, t1, t2, t3 = s7, s5, s3, s1
    z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
    z5 = (z3 + z4) * F["c1_175875602"]
    t0 = t0 * F["c0_298631336"]; t1 = t1 * F["c2_053119869"]; t2 = t2 * F["c3_072711026"]; t3 = t3 * F["c1_501321110"]
    z1 = z1 * -F["c0_899976223"]; z2 = z2 * -F["c2_562915447"]; z3 = z3 * -F["c1_961570560"]; z4 = z4 * -F["c0_390180644"]
    z3 = z3 + z5; z4 = z4 + z5
    t0 = t0 + z1 + z3; t1 = t1 + z2 + z4; t2 = t2 + z2 + z3; t3 = t3 + z1 + z4
    return [tmp10 + t3, tmp11 + t2, tmp12 + t1, tmp13 + t0, tmp13 - t0, tmp12 - t1, tmp11 - t2, tmp10 - t3]


def idct_range_limit(x):
    """libjpeg's post-IDCT table lookup range_limit[x & 1023] (jdmaster.c prepare_range_limit_table), x the descaled output:
    x + 128 clamped to 0..255 for x in [-512, 511], wrapping outside.  csrc/jpeg.cu flags a frame whose output leaves that
    window (DESIGN.md section 9)."""
    u = (x + 128) & 1023
    return np.where(u < 256, u, np.where(u < 640, 255, 0))


def idct_islow(coef, qt):
    """coef [..., 64] quantised coefficients, qt [64] (natural order) -> uint8 [..., 8, 8] samples."""
    d = (coef.astype(np.int64) * qt.astype(np.int64)).reshape(coef.shape[:-1] + (8, 8))
    # pass 1: columns (the all-zero-AC shortcut of jidctint.c gives the same values as the general formula)
    cols = _idct_1d(*[d[..., k, :] for k in range(8)])
    ws = np.stack([_descale(c, CONST_BITS - PASS1_BITS) for c in cols], -2)
    rows = _idct_1d(*[ws[..., :, k] for k in range(8)])
    out = np.stack([_descale(r, CONST_BITS + PASS1_BITS + 3) for r in rows], -1)
    return idct_range_limit(out).astype(np.uint8)


def component_planes(parsed, coefs):
    data, q, huff, ri, (H, W, comps), sos, pos = parsed
    planes = []
    for (cid, h, v, tq), c in zip(comps, coefs):
        blocks = idct_islow(c, q[tq])                           # [rows, cols, 8, 8]
        r, k = blocks.shape[:2]
        planes.append(blocks.transpose(0, 2, 1, 3).reshape(r * 8, k * 8))
    return planes


def _fancy_h2(rowsum, dw, scale, bias_even, bias_odd, shift):
    """Horizontal triangle filter of jdsample.c over the first dw columns (edge columns replicated)."""
    c = rowsum[:, :dw]
    left = np.concatenate([c[:, :1], c[:, :-1]], 1)
    right = np.concatenate([c[:, 1:], c[:, -1:]], 1)
    out = np.empty((c.shape[0], 2 * dw), np.int64)
    out[:, 0::2] = (c * 3 + left + bias_even) >> shift
    out[:, 1::2] = (c * 3 + right + bias_odd) >> shift
    return out


def upsample(plane, dw, dh, h, v, W, H):
    """A downsampled chroma plane (valid dw x dh) to the full W x H grid: h2v1_fancy_upsample / h2v2_fancy_upsample, or box
    replication when dw <= 2 (jinit_upsampler)."""
    p = plane[:dh, :dw].astype(np.int64)
    if h == 1 and v == 1:
        return p[:H, :W]
    if dw <= 2:
        return np.repeat(np.repeat(p, v, 0), h, 1)[:H, :W]
    if v == 1:
        return _fancy_h2(p, dw, 3, 1, 2, 2)[:H, :W]
    above = np.concatenate([p[:1], p[:-1]], 0)
    below = np.concatenate([p[1:], p[-1:]], 0)
    out = np.empty((2 * dh, 2 * dw), np.int64)
    out[0::2] = _fancy_h2(3 * p + above, dw, 3, 8, 7, 4)
    out[1::2] = _fancy_h2(3 * p + below, dw, 3, 8, 7, 4)
    return out[:H, :W]


def ycc_to_bgr(y, cb, cr):
    """ycc_rgb_convert with build_ycc_rgb_table's fixed-point tables (SCALEBITS 16)."""
    fix = lambda x: int(x * 65536 + 0.5)
    cb = cb.astype(np.int64) - 128
    cr = cr.astype(np.int64) - 128
    y = y.astype(np.int64)
    r = y + ((fix(1.40200) * cr + 32768) >> 16)
    g = y + ((-fix(0.34414) * cb + 32768 - fix(0.71414) * cr) >> 16)
    b = y + ((fix(1.77200) * cb + 32768) >> 16)
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def decode(buf):
    """cv2.imdecode(buf, cv2.IMREAD_COLOR) for an accepted baseline stream: uint8 [H, W, 3] BGR."""
    parsed = parse(buf)
    data, q, huff, ri, (H, W, comps), sos, pos = parsed
    planes = component_planes(parsed, entropy_decode(parsed))
    if len(comps) == 1:
        g = planes[0][:H, :W]
        return np.repeat(g[..., None], 3, -1)
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    full = [planes[0][:H, :W]]
    for (cid, h, v, tq), p in zip(comps[1:], planes[1:]):
        dw, dh = -(-W * h // hmax), -(-H * v // vmax)
        full.append(upsample(p, dw, dh, hmax // h, vmax // v, W, H))
    return ycc_to_bgr(*full)
