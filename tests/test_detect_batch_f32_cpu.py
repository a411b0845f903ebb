"""Host side of the unquantised model's batched pre-process without a GPU: the argument checks of cdn_warp_affine_u8_f32_batch,
the host normalisation table against pre_process, and which table each test scale gets."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200 import _lib
from codenet_b200.compat.detector import CtdetDetector, default_opt

INVALID = -1
FAKE = C.c_void_p(16)               # never dereferenced: every call below is rejected before anything touches the device


def _descs(n, **kw):
    d = np.zeros(n, _lib.WARP_DESC)
    d["src_h"], d["src_w"], d["M"] = 10, 12, [1, 0, 0, 0, 1, 0]
    d["dst_slot"], d["mirror_slot"] = np.arange(n), -1
    for k, v in kw.items():
        d[k] = v
    return d


def _bare(**kw):
    det = CtdetDetector.__new__(CtdetDetector)
    det.opt = default_opt(resume_quantize=False, **kw)
    det.mean = np.array(det.opt.mean, dtype=np.float32).reshape(1, 1, 3)
    det.std = np.array(det.opt.std, dtype=np.float32).reshape(1, 1, 3)
    return det


def test_warp_f32_batch_argument_checks_run_on_the_host():
    lib = _lib.load()
    keep = []

    def call(desc, table=None, n=None, pool=FAKE, tables=FAKE, n_tables=2, dst=FAKE, slots=4, h=8, w=8):
        if table is None and desc is not None:
            table = np.zeros(len(desc), np.int32)
        keep.extend([desc, table])
        p = C.c_void_p(desc.ctypes.data) if desc is not None else None
        t = C.c_void_p(table.ctypes.data) if table is not None else None
        return lib.cdn_warp_affine_u8_f32_batch(pool, p, t, len(desc) if n is None else n, tables, n_tables, dst, slots, h, w, None)

    ok = _descs(4)
    assert call(ok, pool=None) == INVALID and b"null pointer" in lib.cdn_last_error()
    assert call(ok, tables=None) == INVALID and b"null pointer" in lib.cdn_last_error()
    assert call(ok, dst=None) == INVALID and b"null pointer" in lib.cdn_last_error()
    assert call(None, n=1) == INVALID
    assert lib.cdn_warp_affine_u8_f32_batch(FAKE, C.c_void_p(ok.ctypes.data), None, 4, FAKE, 2, FAKE, 4, 8, 8, None) == INVALID
    assert call(ok, dst=C.c_void_p(18)) == INVALID and b"aligned" in lib.cdn_last_error()
    assert call(ok, n=-1) == INVALID
    assert call(ok, n_tables=0) == INVALID and b"n_tables = 0" in lib.cdn_last_error()
    assert call(ok, n_tables=3) == INVALID and b"n_tables = 3" in lib.cdn_last_error()
    assert call(ok, slots=0) == INVALID and call(ok, h=0) == INVALID and call(ok, w=-3) == INVALID
    assert call(_descs(4, src_offset=[0, 16, -1, 32])) == INVALID and b"descriptor 2" in lib.cdn_last_error()
    assert call(_descs(4, src_h=[5, 0, 5, 5])) == INVALID and b"descriptor 1" in lib.cdn_last_error()
    assert call(_descs(4, src_w=[5, 5, 5, -2])) == INVALID
    assert call(_descs(4, dst_slot=[0, 1, 2, 4])) == INVALID and b"outside [0, 4)" in lib.cdn_last_error()
    assert call(_descs(4, mirror_slot=[1, -2, -1, -1])) == INVALID
    assert call(ok, table=np.array([0, 1, 2, 0], np.int32)) == INVALID and b"descriptor 2: table 2" in lib.cdn_last_error()
    assert call(ok, table=np.array([0, -1, 0, 0], np.int32)) == INVALID and b"descriptor 1" in lib.cdn_last_error()
    assert call(ok, table=np.array([0, 0, 0, 1], np.int32), n_tables=1) == INVALID and b"outside [0, 1)" in lib.cdn_last_error()
    # a bad descriptor or table index past the first launch's worth is still caught before anything is launched
    many = _descs(2 * _lib.WARP_F32_DESC_PER_LAUNCH + 3, dst_slot=0)
    many["src_h"][-1] = 0
    assert call(many, slots=1) == INVALID and b"descriptor %d" % (len(many) - 1) in lib.cdn_last_error()
    many = _descs(_lib.WARP_F32_DESC_PER_LAUNCH + 5, dst_slot=0)
    table = np.zeros(len(many), np.int32)
    table[_lib.WARP_F32_DESC_PER_LAUNCH + 2] = 2
    assert call(many, table=table, slots=1) == INVALID
    assert b"descriptor %d: table 2" % (_lib.WARP_F32_DESC_PER_LAUNCH + 2) in lib.cdn_last_error()
    assert call(ok, n=0) == 0                                                  # nothing to launch
    assert call(ok, n=0, n_tables=1) == 0


def _lookup(table, u8_hwc):
    """table [3][256] applied to a uint8 HWC image -> fp32 CHW"""
    return np.stack([table[c][u8_hwc[..., c]] for c in range(3)])


@pytest.mark.parametrize("shape", [(3, 2), (31, 17), (375, 500), (500, 333), (512, 512)])
def test_host_table_equals_pre_process(shape):
    """The host table run_batch uses for scales other than 1 (and for scale 1 without device_pre_process), looked up at the
    bytes cv2.warpAffine writes, equals pre_process's float64 normalisation, mirror included, bit for bit."""
    cv2 = pytest.importorskip("cv2")
    from codenet_b200.compat.detector import get_affine_transform
    det = _bare(input_h=128, input_w=160, flip_test=True)
    table = det._host_table()
    assert table.shape == (3, 256) and table.dtype == np.float32
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    img = rng.integers(0, 256, shape + (3,), dtype=np.uint8)
    for scale in (0.5, 1.0, 1.5):
        got, meta = det.pre_process(img, scale)
        got = got.numpy()
        (sh, sw), (ih, iw), c, s = det.input_geometry(shape[0], shape[1], scale)
        warped = cv2.warpAffine(cv2.resize(img, (sw, sh)), get_affine_transform(c, s, 0, [iw, ih]), (iw, ih), flags=cv2.INTER_LINEAR)
        assert got.shape == (2, 3, ih, iw)
        np.testing.assert_array_equal(got[0], _lookup(table, warped))
        np.testing.assert_array_equal(got[1], _lookup(table, warped[:, ::-1]))
    # the table is the helper's value at every byte: the normalisation of a 256 x 3 ramp image
    ramp = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, 1)[None]
    np.testing.assert_array_equal(det._normalize_host(ramp)[0].T, table)


def test_table_choice_per_scale():
    """Scale 1 with device_pre_process (the default) is normalised as _process_float does on the device (table 0); every other
    scale, and scale 1 without device_pre_process, as pre_process does on the host (table 1)."""
    det = _bare()
    assert not hasattr(det.opt, "device_pre_process")
    assert [det._device_table(s) for s in (0.5, 1, 1.0, 1.5)] == [False, True, True, False]
    for on in (True, False):
        det = _bare(device_pre_process=on)
        assert [det._device_table(s) for s in (0.5, 0.75, 1.0, 1.25, 1.5)] == [False, False, on, False, False]
        assert list(det._table_index([0.5, 1.0, 1.5], 3)) == [1, int(not on), 1] * 3
