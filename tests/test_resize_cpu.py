"""oracle.resize_ref, the reference of the device resize inside cdn_warp_affine_resize_u8[_f32]_batch, against this machine's
cv2.resize (INTER_LINEAR, uint8, 3 channels): zero mismatched bytes wherever device_resize_exact says the device path may run."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")
from oracle import resize_ref  # noqa: E402
from oracle.resize_ref import device_resize_exact  # noqa: E402

SCALES = (0.5, 0.75, 1.0, 1.25, 1.5)
# the VOC / COCO frame shapes (H, W) and their transposes
SHAPES = [(375, 500), (500, 375), (333, 500), (500, 333), (480, 640), (640, 480), (427, 640), (640, 427)]


def _mismatch(src, sh, sw):
    return int(np.count_nonzero(cv2.resize(src, (sw, sh)) != resize_ref.resize(src, (sw, sh))))


def test_dense_small_grid_at_the_standard_scales():
    """Every H x W from 1 x 1 to 64 x 64 at the five standard scales (the detector's int(side * scale))."""
    rng = np.random.default_rng(0)
    checked = 0
    for H in range(1, 65):
        for W in range(1, 65):
            src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
            for s in SCALES:
                sh, sw = int(H * s), int(W * s)
                if not device_resize_exact(H, W, sh, sw):
                    assert min(sh, sw) == 0, (H, W, s)              # only the empty resizes of 1-pixel sides are left out
                    continue
                assert _mismatch(src, sh, sw) == 0, (H, W, s)
                checked += 1
    assert checked == 5 * 64 * 64 - 2 * (2 * 64 - 1)                # a side of 1 at scales 0.5 and 0.75


@pytest.mark.parametrize("shape", SHAPES)
def test_voc_coco_shapes(shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    H, W = shape
    src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    for s in SCALES:
        sh, sw = int(H * s), int(W * s)
        assert device_resize_exact(H, W, sh, sw), (shape, s)
        assert _mismatch(src, sh, sw) == 0, (shape, s)


def test_upscale_border_rows_read_row_zero_twice():
    """The first row of an upscale has source row -1 with an unclamped fraction: both of its taps read row 0, and the two
    truncating vertical products can lose one unit.  A fully clamped restatement (weights 2048, 0) differs there."""
    rng = np.random.default_rng(5)
    src = rng.integers(0, 256, (375, 500, 3), dtype=np.uint8)
    want = cv2.resize(src, (625, 468))
    np.testing.assert_array_equal(resize_ref.resize(src, (625, 468)), want)
    sy, b0, b1 = resize_ref.coefficients(375, 468, False)
    assert sy[0] == -1 and b1[0] > 0 and sy[-1] == 374 and b1[-1] > 0
    sx, a0, a1 = resize_ref.coefficients(500, 625, True)
    row0 = src[0].astype(np.int64)
    S = row0[sx] * a0[:, None] + row0[np.minimum(sx + 1, 499)] * a1[:, None]
    clamped = (((2048 * (S >> 4)) >> 16) + 2) >> 2           # row 0 at weights (2048, 0)
    assert np.count_nonzero(clamped != want[0]) > 0


def test_random_sweep():
    """Seeded sizes up to 1920 per side (and a few up to RESIZE_MAX_SIDE) at random scales in [0.15, 3.2], per axis: every
    geometry the predicate accepts matches cv2 exactly; the sweep also reaches geometries it rejects."""
    from codenet_b200.compat.detector import RESIZE_MAX_SIDE
    rng = np.random.default_rng(1)
    accepted = rejected = 0
    for i in range(160):
        top = RESIZE_MAX_SIDE if i % 40 == 0 else 1920
        H, W = (int(v) for v in rng.integers(1, top + 1, 2))
        sy, sx = rng.uniform(0.15, 3.2, 2) if i % 2 else (rng.uniform(0.15, 3.2),) * 2
        sh, sw = max(int(H * sy), 1), max(int(W * sx), 1)
        if not device_resize_exact(H, W, sh, sw):
            rejected += 1
            continue
        accepted += 1
        src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        assert _mismatch(src, sh, sw) == 0, (H, W, sh, sw)
    assert accepted >= 100 and rejected >= 5


def test_predicate_says_yes_only_where_the_oracle_holds():
    """The predicate against a brute-force check over a grid of odd geometries: whatever it accepts must match cv2, and it
    rejects empty, oversized and out-of-ratio resizes."""
    rng = np.random.default_rng(2)
    for H, W, sh, sw in [(1, 1, 1, 3), (1, 5, 3, 1), (2, 2, 1, 1), (5, 3, 15, 9), (7, 9, 2, 2), (640, 2, 128, 6), (3, 640, 9, 128),
                         (99, 101, 297, 303), (100, 100, 20, 20), (1080, 1920, 1620, 2880)]:
        assert device_resize_exact(H, W, sh, sw), (H, W, sh, sw)
        src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        assert _mismatch(src, sh, sw) == 0, (H, W, sh, sw)
    for H, W, sh, sw in [(10, 10, 0, 5), (10, 10, 5, 0), (0, 10, 1, 1), (4097, 10, 4097, 10), (10, 10, 31, 10), (100, 100, 19, 50),
                         (4000, 4000, 4097, 4000)]:
        assert not device_resize_exact(H, W, sh, sw), (H, W, sh, sw)


def test_identity_copies():
    rng = np.random.default_rng(3)
    src = rng.integers(0, 256, (17, 23, 3), dtype=np.uint8)
    out = resize_ref.resize(src, (23, 17))
    np.testing.assert_array_equal(out, src)
    assert out is not src
