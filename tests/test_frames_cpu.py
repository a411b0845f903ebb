"""CUDA and YUV 4:2:0 frames for run_batch without a GPU: the general-source descriptor of cdn_warp_affine_src_u8[_f32]_batch and
its host checks, oracle.yuv_ref against cv2.cvtColor (and composed with oracle.warp_ref against cv2.warpAffine), the YUV420 type,
to_bgr, and which inputs run_batch reads in place and which it sends down the host path."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from codenet_b200 import _lib
from codenet_b200.compat.detector import CtdetDetector, default_opt, _staged_sources
from codenet_b200.frames import YUV420, to_bgr

cv2 = pytest.importorskip("cv2")
from oracle import warp_ref, yuv_ref  # noqa: E402

INVALID = -1
FAKE = 16                            # a device address never dereferenced: every call below is rejected on the host
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_src_descriptor_layout_matches_the_header():
    d = _lib.WARP_SRC_DESC
    assert d.itemsize == 112
    names = ("plane", "pitch", "kind", "chroma_step", "src_h", "src_w", "M", "dst_slot", "mirror_slot")
    assert [d.fields[k][1] for k in names] == [0, 24, 40, 44, 48, 52, 56, 104, 108]
    header = open(os.path.join(ROOT, "include", "codenet_b200.h")).read()
    define = lambda name: int(re.search(r"#define %s (\d+)" % name, header).group(1))
    assert define("CDN_WARP_SRC_DESC_PER_LAUNCH") == _lib.WARP_SRC_DESC_PER_LAUNCH
    assert define("CDN_WARP_SRC_F32_DESC_PER_LAUNCH") == _lib.WARP_SRC_F32_DESC_PER_LAUNCH
    assert (define("CDN_WARP_SRC_BGR"), define("CDN_WARP_SRC_YUV420")) == (_lib.WARP_SRC_BGR, _lib.WARP_SRC_YUV420)


def _src_descs(n, kind=0, **kw):
    d = np.zeros(n, _lib.WARP_SRC_DESC)
    d["plane"] = FAKE
    d["kind"], d["chroma_step"], d["src_h"], d["src_w"], d["M"] = kind, 1, 10, 12, [1, 0, 0, 0, 1, 0]
    d["pitch"] = np.where(d["kind"][:, None] == 0, [36, 6], [12, 6])
    d["dst_slot"], d["mirror_slot"] = np.arange(n), -1
    for k, v in kw.items():
        d[k] = v
    return d


@pytest.mark.parametrize("form", ["u8", "f32"])
def test_src_warp_argument_checks_run_on_the_host(form):
    lib = _lib.load()
    keep = []

    def call(desc, n=None, dst=FAKE, slots=4, h=8, w=8, table=None, n_tables=2, tables=FAKE):
        keep.append(desc)
        p = C.c_void_p(desc.ctypes.data) if desc is not None else None
        n = len(desc) if n is None else n
        if form == "u8":
            return lib.cdn_warp_affine_src_u8_batch(p, n, C.c_void_p(dst) if dst else None, slots, h, w, None)
        table = np.zeros(max(n, 1), np.int32) if table is None else np.asarray(table, np.int32)
        keep.append(table)
        return lib.cdn_warp_affine_src_u8_f32_batch(p, C.c_void_p(table.ctypes.data), n, C.c_void_p(tables) if tables else None,
                                                    n_tables, C.c_void_p(dst) if dst else None, slots, h, w, None)

    def rejects(desc, what, **kw):
        assert call(desc, **kw) == INVALID, what
        assert what.encode() in lib.cdn_last_error(), (what, lib.cdn_last_error())

    ok, yuv = _src_descs(4), _src_descs(4, kind=1)
    rejects(ok, "null pointer", dst=0)
    rejects(None, "null pointer", n=1)
    rejects(ok, "n = -1", n=-1)
    rejects(ok, "bad destination", slots=0)
    rejects(_src_descs(4, kind=[0, 1, 2, 0]), "descriptor 2: unknown source kind 2")
    rejects(_src_descs(4, src_h=[5, 0, 5, 5]), "descriptor 1: bad source size")
    rejects(_src_descs(4, src_w=[5, 5, 5, -2]), "descriptor 3: bad source size")
    bgr_null = _src_descs(4)
    bgr_null["plane"][2, 0] = 0
    rejects(bgr_null, "descriptor 2: null plane")
    for k in range(3):                                       # every plane of a YUV source is read
        d = _src_descs(4, kind=1)
        d["plane"][1, k] = 0
        rejects(d, "descriptor 1: null plane")
    bgr_only = _src_descs(4)
    bgr_only["plane"][:, 1:] = 0                             # BGR reads plane 0 only
    assert call(bgr_only, n=0) == 0
    rejects(_src_descs(4, pitch=[(36, 0), (35, 0), (36, 0), (36, 0)]), "descriptor 1: pitch 35 below the row's 36")
    rejects(_src_descs(4, kind=1, src_h=[10, 10, 9, 10]), "descriptor 2: odd YUV 4:2:0 size")
    rejects(_src_descs(4, kind=1, src_w=[10, 11, 10, 10]), "descriptor 1: odd YUV 4:2:0 size")
    rejects(_src_descs(4, kind=1, chroma_step=[1, 1, 1, 3]), "descriptor 3: chroma step 3")
    rejects(_src_descs(4, kind=1, chroma_step=[0, 1, 1, 1]), "descriptor 0: chroma step 0")
    rejects(_src_descs(4, kind=1, pitch=[(12, 6), (11, 6), (12, 6), (12, 6)]), "descriptor 1: pitch 11 / 6")
    rejects(_src_descs(4, kind=1, pitch=[(12, 6), (12, 6), (12, 5), (12, 6)]), "descriptor 2: pitch 12 / 5")
    # interleaved chroma: (W/2 - 1) * 2 + 1 = 11 bytes a row for W = 12
    rejects(_src_descs(4, kind=1, chroma_step=2, pitch=[(12, 12), (12, 12), (12, 12), (12, 10)]), "descriptor 3: pitch 12 / 10")
    assert call(_src_descs(4, kind=1, chroma_step=2, pitch=(12, 11)), n=0) == 0
    rejects(_src_descs(4, dst_slot=[0, 1, 2, 4]), "outside [0, 4)")
    rejects(_src_descs(4, kind=1, mirror_slot=[1, -2, -1, -1]), "descriptor 1: slot")
    # a bad descriptor past the first launch's worth is still caught before anything is launched
    per = _lib.WARP_SRC_DESC_PER_LAUNCH if form == "u8" else _lib.WARP_SRC_F32_DESC_PER_LAUNCH
    many = _src_descs(2 * per + 3, kind=1, dst_slot=0)
    many["chroma_step"][-1] = 4
    rejects(many, "descriptor %d: chroma step 4" % (len(many) - 1), slots=1)
    assert call(ok, n=0) == 0 and call(yuv, n=0) == 0                           # nothing to launch
    if form == "f32":
        rejects(ok, "table 2 outside [0, 2)", table=[0, 1, 2, 0])
        rejects(ok, "n_tables = 3", n_tables=3)
        rejects(ok, "null pointer", tables=0)
        rejects(ok, "4-byte aligned", dst=FAKE + 2)
        many = _src_descs(2 * per + 3, dst_slot=0)
        table = np.zeros(len(many), np.int32)
        table[-1] = -1
        rejects(many, "descriptor %d: table -1" % (len(many) - 1), slots=1, table=table)


# ---- oracle.yuv_ref against cv2 -------------------------------------------------------------------------------------------
CODES = {"I420": cv2.COLOR_YUV2BGR_I420, "YV12": cv2.COLOR_YUV2BGR_YV12, "NV12": cv2.COLOR_YUV2BGR_NV12,
         "NV21": cv2.COLOR_YUV2BGR_NV21}


def _surface(Y, U, V, layout):
    """The (3H/2, W) buffer cv2 converts with CODES[layout], and (y, u, v) as strided views into it."""
    H, W = Y.shape
    if layout in ("I420", "YV12"):
        first, second = (U, V) if layout == "I420" else (V, U)
        s = np.concatenate([Y.reshape(-1), first.reshape(-1), second.reshape(-1)]).reshape(H * 3 // 2, W)
        flat = s.reshape(-1)
        a = flat[H * W:H * W * 5 // 4].reshape(H // 2, W // 2)
        b = flat[H * W * 5 // 4:].reshape(H // 2, W // 2)
        return s, (s[:H], a, b) if layout == "I420" else (s[:H], b, a)
    first, second = (U, V) if layout == "NV12" else (V, U)
    s = np.concatenate([Y.reshape(-1), np.stack([first, second], -1).reshape(-1)]).reshape(H * 3 // 2, W)
    a, b = s[H:, 0::2], s[H:, 1::2]
    return s, (s[:H], a, b) if layout == "NV12" else (s[:H], b, a)


def test_yuv_oracle_equals_cv2_on_every_triple():
    """All 2^24 (Y, U, V) triples in one 4096 x 4096 frame: chroma sample (i, j) carries the pair c = 2048 i + j modulo 2^16 and
    the four Y values 4 (c >> 16) + {0, 1, 2, 3} in its 2 x 2 block, so every pair meets every Y once."""
    c = np.arange(1 << 22, dtype=np.int64).reshape(2048, 2048)
    U, V = (c & 255).astype(np.uint8), ((c >> 8) & 255).astype(np.uint8)
    g = (c >> 16) * 4
    Y = np.empty((4096, 4096), np.uint8)
    for dy in (0, 1):
        for dx in (0, 1):
            Y[dy::2, dx::2] = g + 2 * dy + dx
    triples = (Y.astype(np.int64) << 16) | (np.repeat(np.repeat(U, 2, 0), 2, 1).astype(np.int64) << 8) | np.repeat(np.repeat(V, 2, 0), 2, 1)
    assert np.unique(triples).size == 1 << 24
    del triples
    want = None
    for layout, code in CODES.items():
        s, (y, u, v) = _surface(Y, U, V, layout)
        got = yuv_ref.yuv420_to_bgr(y, u, v)
        want = cv2.cvtColor(s, code) if want is None else want
        np.testing.assert_array_equal(got, want, err_msg=layout)
        np.testing.assert_array_equal(cv2.cvtColor(s, code), want, err_msg=layout)


def test_yuv_oracle_equals_cv2_on_every_width():
    """Seeded frames of every even width from 2 to 258 (every SIMD tail of cv2's row loop), in all four layouts."""
    rng = np.random.default_rng(7)
    for W in range(2, 260, 2):
        H = 2 * int(rng.integers(1, 9))
        Y = rng.integers(0, 256, (H, W), dtype=np.uint8)
        U, V = (rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8) for _ in range(2))
        for layout, code in CODES.items():
            s, (y, u, v) = _surface(Y, U, V, layout)
            np.testing.assert_array_equal(yuv_ref.yuv420_to_bgr(y, u, v), cv2.cvtColor(s, code), err_msg="%s W=%d" % (layout, W))


def test_yuv_oracle_then_warp_ref_equals_cv2_warp_of_the_conversion():
    """oracle.warp_ref of the converted frame is cv2.warpAffine(cv2.cvtColor(...)) for the detector's matrices (landscape,
    portrait, scale 1 and other scales) at its usual input size and a dst_w % 4 != 0 one."""
    det = _bare(test_scales=[1.0, 0.75, 1.25])
    rng = np.random.default_rng(8)
    for H, W in ((38, 50), (50, 38), (20, 34)):
        Y = rng.integers(0, 256, (H, W), dtype=np.uint8)
        U, V = (rng.integers(0, 256, (H // 2, W // 2), dtype=np.uint8) for _ in range(2))
        s, (y, u, v) = _surface(Y, U, V, "NV12")
        bgr = cv2.cvtColor(s, cv2.COLOR_YUV2BGR_NV12)
        for ih, iw in ((64, 64), (30, 45)):
            det.opt.input_h, det.opt.input_w = ih, iw
            for _, _, M, _ in det._frame_layout(H, W, det.scales):
                want = cv2.warpAffine(bgr, M, (iw, ih), flags=cv2.INTER_LINEAR)
                np.testing.assert_array_equal(warp_ref.warp_affine(yuv_ref.yuv420_to_bgr(y, u, v), M, (iw, ih)), want)


# ---- YUV420 and to_bgr ----------------------------------------------------------------------------------------------------
def test_yuv420_validation():
    y, c = np.zeros((4, 6), np.uint8), np.zeros((2, 3), np.uint8)
    YUV420(y, c, c)
    nv12 = np.zeros((6, 6), np.uint8)
    f = YUV420(nv12[:4], nv12[4:, 0::2], nv12[4:, 1::2])
    assert f.shape == (4, 6) and not f.is_cuda
    with pytest.raises(ValueError, match="positive even"):
        YUV420(np.zeros((3, 6), np.uint8), c, c)
    with pytest.raises(ValueError, match="positive even"):
        YUV420(np.zeros((4, 5), np.uint8), np.zeros((2, 2), np.uint8), np.zeros((2, 2), np.uint8))
    with pytest.raises(ValueError, match="must be"):
        YUV420(y, np.zeros((2, 2), np.uint8), c)
    with pytest.raises(ValueError, match="must be"):
        YUV420(y, c, np.zeros((3, 3), np.uint8))
    with pytest.raises(ValueError, match="2-D uint8"):
        YUV420(y.astype(np.int16), c, c)
    with pytest.raises(ValueError, match="2-D uint8"):
        YUV420(y, c.astype(np.float32), c)
    with pytest.raises(ValueError, match="2-D uint8"):
        YUV420(y[..., None], c, c)
    wide = np.zeros((2, 9), np.uint8)
    with pytest.raises(ValueError, match="column strides"):
        YUV420(y, wide[:, 0::3], wide[:, 1::3])                      # column stride 3
    with pytest.raises(ValueError, match="column strides"):
        YUV420(y, nv12[4:, 0::2], c)                                  # 2 and 1
    with pytest.raises(ValueError, match="Y column stride"):
        YUV420(np.zeros((4, 12), np.uint8)[:, ::2], c, c)
    with pytest.raises(ValueError, match="row strides"):
        YUV420(y, c, np.zeros((2, 4), np.uint8)[:, :3])              # U and V rows differ
    with pytest.raises(ValueError, match="row strides"):
        YUV420(np.lib.stride_tricks.as_strided(y, (4, 6), (3, 1)), c, c)
    with pytest.raises(ValueError, match="CPU tensor"):
        YUV420(torch.zeros((4, 6), dtype=torch.uint8), c, c)
    with pytest.raises(ValueError, match="not a numpy array"):
        YUV420([[0] * 6] * 4, c, c)


def test_to_bgr_is_cv2_i420():
    rng = np.random.default_rng(9)
    Y = rng.integers(0, 256, (10, 14), dtype=np.uint8)
    U, V = (rng.integers(0, 256, (5, 7), dtype=np.uint8) for _ in range(2))
    for layout, code in CODES.items():
        s, planes = _surface(Y, U, V, layout)
        np.testing.assert_array_equal(to_bgr(YUV420(*planes)), cv2.cvtColor(s, code), err_msg=layout)


# ---- run_batch's routing --------------------------------------------------------------------------------------------------
def _bare(**kw):
    det = CtdetDetector.__new__(CtdetDetector)
    det.opt = default_opt(**kw)
    det.scales = det.opt.test_scales
    return det


def test_run_batch_reads_yuv_frames_in_the_warp_at_scale_1_and_on_the_host_otherwise():
    rng = np.random.default_rng(10)
    bgr = rng.integers(0, 256, (30, 40, 3), dtype=np.uint8)
    nv12 = rng.integers(0, 256, (45, 40), dtype=np.uint8)
    yuv = YUV420(nv12[:30], nv12[30:, 0::2], nv12[30:, 1::2])
    for kw in ({}, {"flip_test": True}, {"test_scales": [1.0, 1.0]}, {"resume_quantize": False}):
        det = _bare(**kw)
        items = det._batch_frames([bgr, yuv])
        assert items[0][0] is bgr and items[0][1:] == (None, None)
        assert items[1][:2] == (None, None) and items[1][2] is yuv, kw
        layouts = [det._frame_layout(30, 40, det.scales)] * 2
        # host BGR: every scale's source; host YUV420: Y, U and V once, 1.5 bytes per pixel
        assert _staged_sources(items[0], layouts[0]) == [30 * 40 * 3] * len(det.scales)
        assert _staged_sources(items[1], layouts[1]) == [1200, 300, 300]
    for kw in ({"test_scales": [1.0, 0.5]}, {"test_scales": [0.75], "flip_test": True}):
        det = _bare(**kw)
        items = det._batch_frames([bgr, yuv])
        assert items[0][0] is bgr
        assert items[1][1:] == (None, None)
        np.testing.assert_array_equal(items[1][0], to_bgr(yuv))


def test_run_batch_rejects_what_it_does_not_take():
    det = _bare()
    img = np.zeros((20, 30, 3), np.uint8)
    with pytest.raises(ValueError, match="CUDA tensors only"):
        det.run_batch([img, torch.zeros((20, 30, 3), dtype=torch.uint8)])
    with pytest.raises(ValueError, match="prefetched dicts"):
        det.run_batch([img, (np.zeros((4, 6), np.uint8),) * 3])
