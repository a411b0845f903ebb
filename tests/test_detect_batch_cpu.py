"""Host side of the batched detector without a GPU: the argument checks of cdn_warp_affine_u8_batch, the step / slot planner
of CtdetDetector.run_batch and the inputs run_batch rejects."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200 import _lib
from codenet_b200.compat.detector import CtdetDetector, default_opt, plan_frame_steps

INVALID = -1
FAKE = C.c_void_p(16)               # never dereferenced: every call below is rejected before anything touches the device


def _descs(n, **kw):
    d = np.zeros(n, _lib.WARP_DESC)
    d["src_h"], d["src_w"], d["M"] = 10, 12, [1, 0, 0, 0, 1, 0]
    d["dst_slot"], d["mirror_slot"] = np.arange(n), -1
    for k, v in kw.items():
        d[k] = v
    return d


def test_descriptor_layout_matches_the_header():
    assert _lib.WARP_DESC.itemsize == 72
    assert [_lib.WARP_DESC.fields[k][1] for k in ("src_offset", "src_h", "src_w", "M", "dst_slot", "mirror_slot")] == [0, 8, 12, 16, 64, 68]


def test_warp_batch_argument_checks_run_on_the_host():
    lib = _lib.load()
    keep = []

    def call(desc, n=None, pool=FAKE, dst=FAKE, slots=4, h=8, w=8):
        keep.append(desc)
        p = C.c_void_p(desc.ctypes.data) if desc is not None else None
        return lib.cdn_warp_affine_u8_batch(pool, p, len(desc) if n is None else n, dst, slots, h, w, None)

    ok = _descs(4)
    assert call(ok, pool=None) == INVALID and b"null pointer" in lib.cdn_last_error()
    assert call(ok, dst=None) == INVALID
    assert call(None, n=1) == INVALID
    assert call(ok, n=-1) == INVALID
    assert call(ok, slots=0) == INVALID and call(ok, h=0) == INVALID and call(ok, w=-3) == INVALID
    assert call(_descs(4, src_offset=[0, 16, -1, 32])) == INVALID and b"descriptor 2" in lib.cdn_last_error()
    assert call(_descs(4, src_h=[5, 0, 5, 5])) == INVALID and b"descriptor 1" in lib.cdn_last_error()
    assert call(_descs(4, src_w=[5, 5, 5, -2])) == INVALID
    assert call(_descs(4, dst_slot=[0, 1, 2, 4])) == INVALID and b"outside [0, 4)" in lib.cdn_last_error()
    assert call(_descs(4, dst_slot=[0, -1, 2, 3])) == INVALID
    assert call(_descs(4, mirror_slot=[1, -2, -1, -1])) == INVALID
    assert call(_descs(4, mirror_slot=[4, -1, -1, -1])) == INVALID
    # a bad descriptor past the first launch's worth is still caught before anything is launched
    many = _descs(2 * _lib.WARP_DESC_PER_LAUNCH + 3, dst_slot=0)
    many["src_h"][-1] = 0
    assert call(many, slots=1) == INVALID and b"descriptor %d" % (len(many) - 1) in lib.cdn_last_error()
    assert call(ok, n=0) == 0                                                  # nothing to launch
    # the one-descriptor entry point keeps its checks
    M = np.array([1, 0, 0, 0, 1, 0], np.float64)
    assert lib.cdn_warp_affine_u8(FAKE, 0, 5, C.c_void_p(M.ctypes.data), FAKE, 8, 8, 0, None) == INVALID
    assert lib.cdn_warp_affine_u8(FAKE, 5, 5, None, FAKE, 8, 8, 0, None) == INVALID


def test_step_planner():
    """Whole frames per step in frame order, at most max(max_batch, slots per frame) slots, 16-byte-aligned pool offsets."""
    rng = np.random.default_rng(0)
    sizes = [[int(v) for v in rng.integers(1, 5000, 3)] for _ in range(11)]
    for spf, max_batch in ((3, 1), (3, 8), (6, 6), (6, 13), (6, 64), (2, 3)):
        steps = plan_frame_steps(sizes, spf, max_batch)
        frames = [f for fr, _, _ in steps for f in fr]
        assert frames == list(range(len(sizes)))
        for fr, offsets, nbytes in steps:
            assert 1 <= len(fr) and len(fr) * spf <= max(max_batch, spf)
            assert len(offsets) == len(fr)
            flat = [(o, sizes[f][j]) for f, offs in zip(fr, offsets) for j, o in enumerate(offs)]
            assert [len(o) for o in offsets] == [len(sizes[f]) for f in fr]
            assert all(o % 16 == 0 for o, _ in flat)
            assert all(a + na <= b for (a, na), (b, _) in zip(flat, flat[1:]))      # in order, no overlap
            assert flat[-1][0] + flat[-1][1] <= nbytes and nbytes % 16 == 0
        # every step but the last is full
        per = max(max_batch, spf) // spf
        assert [len(fr) for fr, _, _ in steps][:-1] == [per] * (len(steps) - 1)
    assert plan_frame_steps([], 2, 8) == []
    (fr, offsets, nbytes), = plan_frame_steps([[375 * 500 * 3, 100, 17]], 3, 1)
    assert list(fr) == [0] and offsets == [[0, 562512, 562624]] and nbytes == 562656


def _bare(**kw):
    det = CtdetDetector.__new__(CtdetDetector)
    det.opt = default_opt(**kw)
    return det


def test_run_batch_rejects_what_it_does_not_take(tmp_path):
    img = np.zeros((20, 30, 3), np.uint8)
    with pytest.raises(ValueError, match="fix_res"):
        _bare(fix_res=False).run_batch([img])
    det = _bare()
    for bad in (img.astype(np.float32), img[..., :2], img[..., 0], np.zeros((20, 30, 4), np.uint8)):
        with pytest.raises(ValueError, match="uint8 HWC 3-channel"):
            det.run_batch([img, bad])
    with pytest.raises(ValueError, match="prefetched dicts"):
        det.run_batch([{"image": img, "images": {}, "meta": {}}])
    with pytest.raises(ValueError, match="prefetched dicts"):
        det.run_batch([img, 3])
    pytest.importorskip("cv2")
    with pytest.raises(ValueError, match="cannot read"):
        det.run_batch([str(tmp_path / "missing.jpg")])
    assert det.run_batch([]) == []
