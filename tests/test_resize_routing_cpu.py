"""run_batch's device resize without a GPU: the cdn_warp_rs_desc layout and the host checks of
cdn_warp_affine_resize_u8[_f32]_batch, which inputs run_batch resizes inside the warp at scale lists other than [1] and which keep
the host cv2.resize, and the bytes it stages for each."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from codenet_b200 import _lib
from codenet_b200.compat import detector as D
from codenet_b200.compat.detector import CtdetDetector, JPEG_DEVICE_MIN_FRAMES, default_opt, _rs_descs, _staged_sources
from codenet_b200.frames import YUV420, to_bgr

cv2 = pytest.importorskip("cv2")

INVALID = -1
FAKE = 16                            # a device address never dereferenced: every call below is rejected on the host
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_rs_descriptor_layout_matches_the_header():
    d = _lib.WARP_RS_DESC
    assert d.itemsize == 136
    names = ("plane", "pitch", "kind", "chroma_step", "src_h", "src_w", "rs_h", "rs_w", "inv_scale", "M", "dst_slot", "mirror_slot")
    assert [d.fields[k][1] for k in names] == [0, 24, 40, 44, 48, 52, 56, 60, 64, 80, 128, 132]
    header = open(os.path.join(ROOT, "include", "codenet_b200.h")).read()
    define = lambda name: int(re.search(r"#define %s (\d+)" % name, header).group(1))
    assert define("CDN_WARP_RS_DESC_PER_LAUNCH") == _lib.WARP_RS_DESC_PER_LAUNCH
    assert define("CDN_WARP_RS_F32_DESC_PER_LAUNCH") == _lib.WARP_RS_F32_DESC_PER_LAUNCH
    body = re.search(r"typedef struct cdn_warp_rs_desc \{(.*?)\} cdn_warp_rs_desc;", header, re.S).group(1)
    assert [m for m in re.findall(r"(\w+)(?:\[\d\])?[,;]", re.sub(r"/\*.*?\*/", "", body))] == list(names)


def _rs(n, kind=0, **kw):
    """n valid-looking descriptors: a 10 x 12 frame resized to 15 x 9."""
    d = np.zeros(n, _lib.WARP_RS_DESC)
    d["plane"] = FAKE
    d["kind"], d["chroma_step"], d["src_h"], d["src_w"], d["M"] = kind, 1, 10, 12, [1, 0, 0, 0, 1, 0]
    d["rs_h"], d["rs_w"] = 15, 9
    d["pitch"] = np.where(d["kind"][:, None] == 0, [36, 6], [12, 6])
    d["dst_slot"], d["mirror_slot"] = np.arange(n), -1
    for k, v in kw.items():
        d[k] = v
    with np.errstate(divide="ignore"):                     # the descriptors with a resized side of 0
        d["inv_scale"][:, 0] = 1.0 / (d["rs_w"] / d["src_w"])
        d["inv_scale"][:, 1] = 1.0 / (d["rs_h"] / d["src_h"])
    return d


@pytest.mark.parametrize("form", ["u8", "f32"])
def test_resize_warp_argument_checks_run_on_the_host(form):
    lib = _lib.load()
    keep = []

    def call(desc, n=None, dst=FAKE, slots=4, h=8, w=8, table=None, n_tables=2, tables=FAKE):
        keep.append(desc)
        p = C.c_void_p(desc.ctypes.data) if desc is not None else None
        n = len(desc) if n is None else n
        if form == "u8":
            return lib.cdn_warp_affine_resize_u8_batch(p, n, C.c_void_p(dst) if dst else None, slots, h, w, None)
        table = np.zeros(max(n, 1), np.int32) if table is None else np.asarray(table, np.int32)
        keep.append(table)
        return lib.cdn_warp_affine_resize_u8_f32_batch(p, C.c_void_p(table.ctypes.data), n, C.c_void_p(tables) if tables else None,
                                                       n_tables, C.c_void_p(dst) if dst else None, slots, h, w, None)

    def rejects(desc, what, **kw):
        assert call(desc, **kw) == INVALID, what
        assert what.encode() in lib.cdn_last_error(), (what, lib.cdn_last_error())

    ok = _rs(4)
    rejects(ok, "null pointer", dst=0)
    rejects(None, "null pointer", n=1)
    rejects(ok, "n = -1", n=-1)
    rejects(ok, "bad destination", slots=0)
    rejects(_rs(4, kind=[0, 1, 2, 0]), "descriptor 2: unknown source kind 2")
    rejects(_rs(4, src_h=[5, 0, 5, 5]), "descriptor 1: bad source size")
    rejects(_rs(4, rs_h=[5, 5, 0, 5]), "descriptor 2: bad resized size")
    rejects(_rs(4, rs_w=[5, 5, 5, -1]), "descriptor 3: bad resized size")
    null = _rs(4)
    null["plane"][1, 0] = 0
    rejects(null, "descriptor 1: null plane")
    for k in range(3):                                       # every plane of a YUV source is read
        d = _rs(4, kind=1)
        d["plane"][2, k] = 0
        rejects(d, "descriptor 2: null plane")
    rejects(_rs(4, pitch=[(36, 0), (36, 0), (35, 0), (36, 0)]), "descriptor 2: pitch 35 below the row's 36")
    rejects(_rs(4, kind=1, src_w=[12, 11, 12, 12]), "descriptor 1: odd YUV 4:2:0 size")
    rejects(_rs(4, kind=1, chroma_step=[1, 3, 1, 1]), "descriptor 1: chroma step 3")
    # the scales must be the frame's and the resized size's, bit for bit
    bad = _rs(4)
    bad["inv_scale"][3, 0] = np.nextafter(bad["inv_scale"][3, 0], 2.0)
    rejects(bad, "descriptor 3: scales")
    bad = _rs(4)
    bad["rs_h"][0] = 16                                      # a resized size the scales do not describe
    rejects(bad, "descriptor 0: scales")
    rejects(_rs(4, dst_slot=[0, 1, 2, 4]), "outside [0, 4)")
    rejects(_rs(4, mirror_slot=[1, -2, -1, -1]), "descriptor 1: slot")
    per = _lib.WARP_RS_DESC_PER_LAUNCH if form == "u8" else _lib.WARP_RS_F32_DESC_PER_LAUNCH
    many = _rs(2 * per + 3, dst_slot=0)
    many["rs_w"][-1] = 0
    rejects(many, "descriptor %d: bad resized size" % (len(many) - 1), slots=1)
    assert call(ok, n=0) == 0 and call(_rs(4, kind=1), n=0) == 0              # nothing to launch
    if form == "f32":
        rejects(ok, "table 2 outside [0, 2)", table=[0, 1, 2, 0])
        rejects(ok, "n_tables = 0", n_tables=0)
        rejects(ok, "null pointer", tables=0)
        rejects(ok, "4-byte aligned", dst=FAKE + 2)


def test_rs_descs_from_general_source_descriptors():
    s = np.zeros(3, _lib.WARP_SRC_DESC)
    s["plane"][:, 0] = [100, 200, 300]
    s["pitch"][:, 0] = [1500, 4000, 96]
    s["kind"], s["chroma_step"] = [0, 1, 0], [1, 2, 1]
    s["src_h"], s["src_w"] = [375, 480, 20], [500, 640, 32]
    s["M"] = np.arange(18).reshape(3, 6)
    s["dst_slot"], s["mirror_slot"] = [0, 2, 4], [1, 3, -1]
    d = _rs_descs(s, [(187, 250), (720, 960), (20, 32)])
    for k in ("plane", "pitch", "kind", "chroma_step", "src_h", "src_w", "M", "dst_slot", "mirror_slot"):
        np.testing.assert_array_equal(d[k], s[k])
    assert d["rs_h"].tolist() == [187, 720, 20] and d["rs_w"].tolist() == [250, 960, 32]
    assert d["inv_scale"].tolist() == [[1 / (250 / 500), 1 / (187 / 375)], [1 / (960 / 640), 1 / (720 / 480)], [1.0, 1.0]]


# ---- run_batch's routing --------------------------------------------------------------------------------------------------
def _bare(**kw):
    """A detector shell with opt.device_resize on unless kw says otherwise."""
    det = CtdetDetector.__new__(CtdetDetector)
    det.opt = default_opt(**dict({"device_resize": True}, **kw))
    det.scales = det.opt.test_scales
    return det


FIVE = [0.5, 0.75, 1.0, 1.25, 1.5]


def test_device_resize_reads_yuv_frames_in_the_warp():
    """With opt.device_resize, host YUV420 frames stay YUV420 items at scale 1 (the general-source warp) and, at other scale lists,
    whenever the device resize reproduces every scale's cv2.resize of them; only a frame outside device_resize_exact goes through
    to_bgr."""
    rng = np.random.default_rng(10)
    bgr = rng.integers(0, 256, (30, 40, 3), dtype=np.uint8)
    nv12 = rng.integers(0, 256, (45, 40), dtype=np.uint8)
    yuv = YUV420(nv12[:30], nv12[30:, 0::2], nv12[30:, 1::2])
    for kw in ({}, {"flip_test": True}, {"test_scales": [1.0, 1.0]}, {"resume_quantize": False}, {"test_scales": [1.0, 0.5]},
               {"test_scales": [0.75], "flip_test": True}, {"test_scales": FIVE, "resume_quantize": False}):
        det = _bare(**kw)
        items = det._batch_frames([bgr, yuv])
        assert items[0][0] is bgr and items[0][1:] == (None, None)
        assert items[1][:2] == (None, None) and items[1][2] is yuv, kw
        multi = any(s != 1 for s in det.scales)
        assert [det._resized_on_device(it) for it in items] == [multi, multi], kw
    # at scale 0.15 both frames' resized sides fall below a fifth of theirs: cv2 resizes them on the host
    det = _bare(test_scales=[0.15, 1.0])
    tall = YUV420(np.zeros((40, 8), np.uint8), np.zeros((20, 4), np.uint8), np.zeros((20, 4), np.uint8))
    items = det._batch_frames([bgr, tall])
    assert not det._resized_on_device(items[0]) and items[1][1:] == (None, None)
    np.testing.assert_array_equal(items[1][0], to_bgr(tall))


def test_device_resize_is_off_by_default():
    """Without opt.device_resize every scale list other than [1] keeps the host path: YUV420 frames through to_bgr, JPEGs decoded
    by cv2, host arrays resized by cv2; scale 1 reads YUV420 frames in the warp as before."""
    rng = np.random.default_rng(12)
    bgr = rng.integers(0, 256, (30, 40, 3), dtype=np.uint8)
    nv12 = rng.integers(0, 256, (45, 40), dtype=np.uint8)
    yuv = YUV420(nv12[:30], nv12[30:, 0::2], nv12[30:, 1::2])
    for kw in ({"device_resize": False}, {"device_resize": None}):
        det = _bare(test_scales=FIVE, **kw)
        if kw["device_resize"] is None:
            del det.opt.device_resize                          # an opt namespace without the field
        items = det._batch_frames([bgr, yuv])
        assert items[1][1:] == (None, None)
        np.testing.assert_array_equal(items[1][0], to_bgr(yuv))
        assert not det._device_resize() and not any(det._resized_on_device(it) for it in items)
    assert _bare(device_resize=False)._batch_frames([yuv])[0][2] is yuv


def test_run_batch_sends_frames_outside_the_predicate_to_the_host(monkeypatch):
    """With device_resize_exact refusing everything, every scale list other than [1] takes today's host path: YUV420 frames
    through to_bgr, host arrays resized by cv2 (none resized on the device)."""
    rng = np.random.default_rng(11)
    bgr = rng.integers(0, 256, (30, 40, 3), dtype=np.uint8)
    nv12 = rng.integers(0, 256, (45, 40), dtype=np.uint8)
    yuv = YUV420(nv12[:30], nv12[30:, 0::2], nv12[30:, 1::2])
    monkeypatch.setattr(D, "device_resize_exact", lambda *a: False)
    det = _bare(test_scales=FIVE)
    items = det._batch_frames([bgr, yuv])
    assert items[1][1:] == (None, None)
    np.testing.assert_array_equal(items[1][0], to_bgr(yuv))
    assert not any(det._resized_on_device(it) for it in items)
    det = _bare()                                             # scale 1 needs no resize
    assert det._batch_frames([yuv])[0][2] is yuv


def test_run_batch_stages_each_frame_once_when_the_device_resizes_it():
    """Bytes staged per input kind at five scales: a host array once at 1x (3 bytes a pixel) when the device resizes it, each
    scale's cv2.resize copy when not; a host YUV420 frame at 1.5 bytes a pixel; nothing for CUDA frames or device-decoded JPEGs."""
    det = _bare(test_scales=FIVE, flip_test=True)
    H, W = 375, 500
    layout = det._frame_layout(H, W, det.scales)
    img = np.zeros((H, W, 3), np.uint8)
    item = (img, None, None)
    assert det._resized_on_device(item)
    assert _staged_sources(item, layout, True) == [H * W * 3]
    host = _staged_sources(item, layout)
    assert host == [int(H * s) * int(W * s) * 3 for s in FIVE] and sum(host) > 5.5 * H * W * 3
    y = np.zeros((H + 1, W), np.uint8)
    c = np.zeros(((H + 1) // 2, W // 2), np.uint8)
    yuv = (None, None, YUV420(y, c, c))
    assert _staged_sources(yuv, layout, True) == [(H + 1) * W, (H + 1) * W // 4, (H + 1) * W // 4]
    assert _staged_sources((None, np.zeros(100, np.uint8), None), layout, True) == [0]
    (_, offsets, nbytes), = D.plan_frame_steps([_staged_sources(item, layout, True)], 10, 10)
    assert offsets == [[0]] and nbytes == -(-H * W * 3 // 16) * 16


def _encode(img):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90])
    assert ok
    return buf.tobytes()


def test_device_resize_decodes_jpeg_on_the_device_from_enough_frames_per_step(tmp_path):
    """With opt.device_resize the quantised model keeps a JPEG compressed for the device with at least JPEG_DEVICE_MIN_FRAMES frames
    per engine step (and in the call), at [1] and at any scale list with a scale other than 1 whose resizes of it the device
    reproduces; otherwise cv2 decodes it on the host, as it does every stream the parser refuses, every JPEG of the unquantised
    model and every JPEG without the option at such scale lists."""
    img = np.random.default_rng(9).integers(0, 256, (30, 40, 3), dtype=np.uint8)
    jpg = _encode(img)
    _, prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    prog = prog.tobytes()
    p = tmp_path / "a.jpg"
    p.write_bytes(jpg)
    n = JPEG_DEVICE_MIN_FRAMES

    def items(frames, **kw):
        det = CtdetDetector.__new__(CtdetDetector)
        det.opt = default_opt(**dict({"device_resize": True}, **kw))
        return det._batch_frames(frames)
    many = [str(p), jpg, bytearray(jpg), memoryview(jpg), np.frombuffer(jpg, np.uint8), prog] * n
    for kw in ({"max_batch": n}, {"max_batch": 5 * n, "test_scales": [1.0, 0.5]}, {"max_batch": 10 * n, "test_scales": FIVE, "flip_test": True}):
        got = items(many, **kw)
        assert all(g[0] is None and g[2][0]["width"] == 40 for g in got[:5]) and got[5][0] is not None, kw
    want = cv2.imdecode(np.frombuffer(jpg, np.uint8), cv2.IMREAD_COLOR)
    for kw in ({"max_batch": n - 1}, {"max_batch": n, "flip_test": True}, {"max_batch": 5 * n - 1, "test_scales": FIVE},
               {"max_batch": n, "resume_quantize": False}, {"max_batch": 10 * n, "test_scales": [1.0, 0.15]},
               {"max_batch": 2 * n, "test_scales": [1.0, 1.0]}, {"max_batch": 5 * n, "test_scales": [1.0, 0.5], "device_resize": False}):
        got = items(many, **kw)
        assert all(np.array_equal(g[0], want) for g in got[:5]), kw
    assert items(many[:n - 1], max_batch=n)[0][0] is not None
