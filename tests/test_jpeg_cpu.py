"""Baseline JPEG decoding, host side: the descriptor layout, cdn_jpeg_parse's classification of cv2.imencode outputs and of
malformed input (every header truncation, seeded byte mutations: each returns a status), the argument checks of
cdn_jpeg_decode_batch, and the numpy restatement oracle.jpeg_ref against cv2.imdecode."""
import ctypes as C
import re
import struct

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from codenet_b200 import _lib, jpeg
from oracle import jpeg_ref

SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411,
            "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440}


def _image(h, w, seed, noisy=True):
    rng = np.random.default_rng(seed)
    if noisy:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[:h, :w]
    return np.stack([x * 255 // max(w, 1), y * 255 // max(h, 1), (x + 2 * y) * 5 % 256], -1).astype(np.uint8)


def _encode(img, **kw):
    params = []
    for k, v in kw.items():
        params += [getattr(cv2, "IMWRITE_JPEG_" + k.upper()), v]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return buf.tobytes()


def test_struct_layout_matches_the_header():
    src = open(__file__.rsplit("/tests/", 1)[0] + "/include/codenet_b200.h").read()
    body = src[src.index("typedef struct cdn_jpeg_frame {"):src.index("} cdn_jpeg_frame;")]
    names = [n for n in re.findall(r"(?:int32_t|int64_t|uint16_t|cdn_jpeg_huff)\s+([^;]+);", body)]
    fields = [f.strip().split("[")[0] for n in names for f in n.split(",")]
    assert fields == list(jpeg.JPEG_FRAME.names)
    assert jpeg.JPEG_FRAME.itemsize == 4256 and jpeg.JPEG_HUFF.itemsize == 912
    assert jpeg.JPEG_FRAME.fields["huff"][1] == 584 and jpeg.JPEG_FRAME.fields["data_offset"][1] == 4232


@pytest.mark.parametrize("sampling,want", [("444", 0), ("422", 0), ("420", 0), ("411", 4), ("440", 4)])
def test_parse_classifies_sampling(sampling, want):
    for q in (10, 50, 75, 95, 100):
        buf = _encode(_image(37, 53, q), quality=q, sampling_factor=SAMPLING[sampling])
        rc, d = jpeg.parse(buf)
        assert rc == want, (sampling, q)
        if rc == 0:
            d = d[0]
            hv = {"444": (1, 1), "422": (2, 1), "420": (2, 2)}[sampling]
            assert (d["width"], d["height"], d["ncomp"], d["hmax"], d["vmax"]) == (53, 37, 3) + hv
            assert (d["mcux"], d["mcuy"]) == (-(-53 // (8 * hv[0])), -(-37 // (8 * hv[1])))
            assert d["scan_end"] == len(buf) - 2 and d["nbytes"] == len(buf)


def test_parse_accepts_gray_optimized_restart_and_separate_chroma_quality():
    img = _image(40, 41, 1)
    assert jpeg.parse(_encode(img[..., 0]))[0] == 0
    assert jpeg.parse(_encode(img, optimize=1))[0] == 0
    for ri in (1, 7):
        rc, d = jpeg.parse(_encode(img, rst_interval=ri))
        assert rc == 0 and d[0]["restart_interval"] == ri
        assert d[0]["nsegments"] == -(-(d[0]["mcux"] * d[0]["mcuy"]) // ri)
    rc, d = jpeg.parse(_encode(img, luma_quality=90, chroma_quality=20))
    assert rc == 0 and not np.array_equal(d[0]["qt"][0], d[0]["qt"][1])
    assert np.array_equal(d[0]["qt"][1], d[0]["qt"][2])


def test_parse_sends_progressive_and_png_to_the_host():
    img = _image(20, 30, 2)
    assert jpeg.parse(_encode(img, progressive=1))[0] == 1
    assert jpeg.parse(cv2.imencode(".png", img)[1])[0] == -1
    assert jpeg.parse(b"")[0] == -1


def _splice_app1(buf, payload):
    return buf[:2] + b"\xff\xe1" + struct.pack(">H", len(payload) + 2) + payload + buf[2:]


def _exif(orientation, little=True):
    e = "<" if little else ">"
    tiff = (b"II" if little else b"MM") + struct.pack(e + "HI", 42, 8) + struct.pack(e + "H", 1)
    tiff += struct.pack(e + "HHI", 0x0112, 3, 1) + struct.pack(e + "HH", orientation, 0) + struct.pack(e + "I", 0)
    return b"Exif\x00\x00" + tiff


@pytest.mark.parametrize("little", [True, False])
def test_parse_exif_orientation(little):
    buf = _encode(_image(24, 40, 3))
    assert jpeg.parse(_splice_app1(buf, _exif(1, little)))[0] == 0
    for o in (2, 3, 6, 8):
        assert jpeg.parse(_splice_app1(buf, _exif(o, little)))[0] == 6
    assert jpeg.parse(_splice_app1(buf, b"Exif\x00\x00XX"))[0] == 6          # unreadable Exif: the host decides
    # cv2 rotates: the host path is the one that returns what cv2 returns
    rotated = _splice_app1(buf, _exif(6, little))
    assert cv2.imdecode(np.frombuffer(rotated, np.uint8), cv2.IMREAD_COLOR).shape[:2] == (40, 24)


def test_parse_every_header_truncation_returns_a_status():
    buf = _encode(_image(16, 24, 4), rst_interval=2)
    scan = jpeg.parse(buf)[1][0]["scan_offset"]
    for n in range(len(buf) + 1):
        rc, d = jpeg.parse(buf[:n])
        if n < scan:
            assert rc < 0, n
        else:
            assert rc == 0 and d[0]["scan_end"] <= n


def test_parse_survives_seeded_mutations():
    """A few thousand byte mutations of small streams (header bytes included): every call returns a status, and what it accepts
    describes a frame inside the stream."""
    rng = np.random.default_rng(5)
    bases = [_encode(_image(13, 21, 6), sampling_factor=SAMPLING[s], rst_interval=r) for s in ("444", "420") for r in (0, 3)]
    bases.append(_encode(_image(13, 21, 7)[..., 0]))
    seen = set()
    for t in range(3000):
        b = bytearray(bases[t % len(bases)])
        head = jpeg.parse(bytes(b))[1][0]["scan_offset"]
        for _ in range(rng.integers(1, 4)):
            pos = int(rng.integers(0, head + 8 if rng.random() < 0.8 else len(b)))
            b[min(pos, len(b) - 1)] = int(rng.integers(0, 256))
        rc, d = jpeg.parse(bytes(b))
        seen.add(rc)
        if rc == 0:
            d = d[0]
            assert 0 < d["scan_offset"] <= d["scan_end"] <= len(b) and d["ncomp"] in (1, 3)
            assert d["ws_bytes"] >= d["plane_rel"][d["ncomp"] - 1] and d["ws_bytes"] % 256 == 0
    assert 0 in seen and any(c < 0 for c in seen)


def test_decode_batch_argument_checks():
    """Rejected on the host before anything is launched.  Every device pointer is null: the device-pointer check comes after
    the descriptor checks, so no call here can reach a launch, and the message shows which check rejected it."""
    L = _lib.load()
    buf = np.frombuffer(_encode(_image(16, 16, 8)), np.uint8)
    rc, d = jpeg.parse(buf)
    assert rc == 0

    def call(desc, n=1, pool=4096, ws=1 << 20, out=1 << 20, frames=True):
        rc = L.cdn_jpeg_decode_batch(None, pool, C.c_void_p(desc.ctypes.data) if frames else None, None, n, None, ws, None, out,
                                     None, None)
        return rc, L.cdn_last_error().decode()

    ok = d.copy()
    cases = [(dict(n=-1), "outside [0, 65535]"), (dict(n=70000), "outside [0, 65535]"), (dict(frames=False), "null descriptor"),
             (dict(pool=len(buf) - 1), "outside the pool"), (dict(ws=int(ok[0]["ws_bytes"]) - 1), "workspace"),
             (dict(out=16 * 16 * 3 - 1), "output outside")]
    for kw, msg in cases:
        rc, err = call(ok, **kw)
        assert rc != 0 and msg in err, (kw, err)
    for field, v, msg in (("data_offset", 4096 - len(buf) + 1, "outside the pool"), ("ws_offset", 128, "not 256-byte aligned"),
                          ("width", 17, "geometry"), ("mcux", 3, "geometry"), ("ncomp", 2, "components"),
                          ("nsegments", 2, "geometry"), ("plane_rel", 0, "geometry"), ("scan_end", 1 << 20, "scan range"),
                          ("comp_h", 3, "sampling"), ("comp_dc", 2, "Huffman table slots")):
        bad = ok.copy()
        bad[0][field] = v
        rc, err = call(bad)
        assert rc != 0 and msg in err, (field, err)
    rc, err = call(ok)                                  # a valid descriptor: only the device pointers are missing
    assert rc != 0 and "null device pointer" in err


def _dht(tc, th, counts, symbols):
    body = bytes([(tc << 4) | th]) + bytes(counts) + bytes(symbols)
    return b"\xff\xc4" + struct.pack(">H", len(body) + 2) + body


@pytest.mark.parametrize("tc", [0, 1])
def test_parse_rejects_oversubscribed_huffman_tables(tc):
    """Code lengths 1-8 with more codes than the code space leaves them (codes that would index past the 8-bit lookahead table,
    up to 200 one-bit codes) and all-ones codes: CDN_JPEG_ERR_TABLE, for every table id, in a stream that is otherwise
    valid.  A full code space without the all-ones code is accepted."""
    good = _encode(_image(16, 16, 11))
    for th in range(4):
        for length in range(1, 8):
            for extra in (0, 1, 3):
                counts = [0] * 16
                counts[length - 1] = (1 << length) + extra    # 2^l codes include the all-ones one: rejected as libjpeg does
                stream = good[:2] + _dht(tc, th, counts, [k % 16 for k in range(sum(counts))]) + good[2:]
                assert jpeg.parse(stream)[0] == -4, (tc, th, length, counts)
        for short in range(1, 8):                             # length 8 (a count is one byte: at most 255 codes) after a shorter one
            counts = [0] * 16
            counts[short - 1], counts[7] = 1, 255
            stream = good[:2] + _dht(tc, th, counts, [k % 16 for k in range(sum(counts))]) + good[2:]
            assert jpeg.parse(stream)[0] == -4, (tc, th, short)
        counts = [0] * 16
        counts[0], counts[1], counts[2] = 1, 1, 1             # 0, 10, 110: 111 stays free
        assert jpeg.parse(good[:2] + _dht(tc, th, counts, [1, 2, 3]) + good[2:])[0] == 0
    counts = [0] * 16
    counts[0] = 200
    assert jpeg.parse(good[:2] + _dht(tc, 0, counts, [0] * 200) + good[2:])[0] == -4


@pytest.mark.parametrize("sampling", ["444", "422", "420", "gray"])
def test_oracle_equals_cv2(sampling):
    shapes = [(1, 1), (5, 7), (9, 17), (16, 16), (23, 31), (3, 4), (2, 5), (8, 3), (33, 40)]
    for i, (h, w) in enumerate(shapes):
        for noisy in (False, True):
            img = _image(h, w, 10 + i, noisy)
            for q, extra in ((10, {}), (75, {"rst_interval": 1}), (95, {"optimize": 1}), (100, {"rst_interval": 7})):
                if sampling == "gray":
                    buf = _encode(img[..., 1], quality=q, **extra)
                else:
                    buf = _encode(img, quality=q, sampling_factor=SAMPLING[sampling], **extra)
                want = cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR)
                np.testing.assert_array_equal(jpeg_ref.decode(buf), want, err_msg="%s %dx%d q%d %s" % (sampling, h, w, q, extra))


def test_oracle_range_limit_is_libjpeg_table():
    """idct_range_limit is jdmaster.c's post-IDCT table (x + 128 clamped, wrapping modulo 1024), which equals the clamp the
    kernel applies inside the window [-512, 511] the device accepts."""
    x = np.arange(-2048, 2048)
    table = np.concatenate([np.arange(128, 256), np.full(384, 255), np.zeros(384, int), np.arange(0, 128)])
    np.testing.assert_array_equal(jpeg_ref.idct_range_limit(x), table[x & 1023])
    inside = (x >= -512) & (x <= 511)
    np.testing.assert_array_equal(jpeg_ref.idct_range_limit(x)[inside], np.clip(x + 128, 0, 255)[inside])


def test_run_batch_decodes_jpeg_on_the_device_from_enough_frames_per_step(tmp_path):
    """run_batch keeps a JPEG compressed for the device only at test scale 1 with at least JPEG_DEVICE_MIN_FRAMES frames per
    engine step (and in the call); otherwise cv2 decodes it on the host, as it does every stream the parser refuses."""
    from codenet_b200.compat.detector import CtdetDetector, JPEG_DEVICE_MIN_FRAMES, default_opt
    jpg, prog = _encode(_image(30, 40, 9)), _encode(_image(30, 40, 9), progressive=1)
    p = tmp_path / "a.jpg"
    p.write_bytes(jpg)
    n = JPEG_DEVICE_MIN_FRAMES

    def items(frames, **kw):
        det = CtdetDetector.__new__(CtdetDetector)
        det.opt = default_opt(**kw)
        return det._batch_frames(frames)
    many = [str(p), jpg, bytearray(jpg), memoryview(jpg), np.frombuffer(jpg, np.uint8), prog] * n
    got = items(many, max_batch=n)
    assert all(g[0] is None and g[2][0]["width"] == 40 for g in got[:5]) and got[5][0] is not None
    want = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR)
    for kw in ({"max_batch": n - 1}, {"max_batch": n, "flip_test": True}, {"max_batch": 5 * n, "test_scales": [1.0, 0.5]},
               {"max_batch": 2 * n, "test_scales": [1.0, 1.0]}, {"max_batch": n, "resume_quantize": False}):
        got = items(many, **kw)
        assert all(np.array_equal(g[0], want) for g in got[:5]), kw
    assert items(many[:n - 1], max_batch=n)[0][0] is not None
