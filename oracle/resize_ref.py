"""TEST INFRASTRUCTURE ONLY.  numpy restatement of cv2.resize(src, (sw, sh)) with the default INTER_LINEAR for uint8 HWC images --
the resize of BaseDetector.pre_process (lib/detectors/base_detector.py:48-60) in front of the warpAffine of oracle.warp_ref.

OpenCV (resize.cpp / resize.simd.hpp, third-party; this container has cv2 4.13) resizes 8-bit images in fixed point with 11-bit
coefficients (INTER_RESIZE_COEF_SCALE = 2048):
  * per destination column dx: fx = float((dx + 0.5) * (1 / (sw / W)) - 0.5), the scale and the products in double, rounded once
    to float; sx = floor(fx), fx -= sx.  A column left of the frame (sx < 0) becomes sx = 0, fx = 0, one past its last pixel
    (sx >= W - 1) becomes sx = W - 1, fx = 0.  Weights a0 = rint(float(1 - fx) * 2048), a1 = rint(fx * 2048) (saturate_cast<short>
    rounds half to even);
  * per destination row the same with H, sh, EXCEPT that the row fraction is never clamped: an upscale's first row has sy = -1
    and a fraction near 1, and reads the frame's row 0 twice (the source row index is clipped, the weights are not).  This is
    why upscales differed from a fully clamped restatement on their first and last rows only;
  * horizontal pass: the exact int S = p[sx] * a0 + p[sx + 1] * a1 (< 2^20) per channel;
  * vertical pass, the one rounding of the SIMD and the scalar code alike: (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16)
    + 2) >> 2, saturated to 8 bits;
  * sh == H and sw == W copies the frame.  The exact-2x downscale OpenCV hands to INTER_AREA, (a + b + c + d + 2) >> 2, is this
    formula with a0 = a1 = b0 = b1 = 1024, so it needs no case of its own.
Pinned against cv2 itself by tests/test_resize_cpu.py over the geometry device_resize_exact accepts."""
import numpy as np

from codenet_b200.compat.detector import device_resize_exact  # noqa: F401  (the geometry the tests pin, re-exported)

COEF_SCALE = 2048


def coefficients(n_src, n_dst, clamp):
    """(first source index, weight of it, weight of the next) of every destination index, int64 arrays of n_dst."""
    scale = 1.0 / (n_dst / n_src)
    f = ((np.arange(n_dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    s = s.astype(np.int64)
    if clamp:
        out = (s < 0) | (s >= n_src - 1)
        s = np.clip(s, 0, n_src - 1)
        f[out] = 0
    w0 = np.rint((np.float32(1) - f) * np.float32(COEF_SCALE)).astype(np.int64)
    w1 = np.rint(f * np.float32(COEF_SCALE)).astype(np.int64)
    return s, w0, w1


def resize(src, dsize):
    """cv2.resize(src, dsize) for uint8 (H, W, C) src, dsize = (sw, sh)."""
    sw, sh = dsize
    H, W = src.shape[:2]
    if (sh, sw) == (H, W):
        return src.copy()
    sx, a0, a1 = coefficients(W, sw, True)
    sy, b0, b1 = coefficients(H, sh, False)
    p = src.astype(np.int64)
    S = p[:, sx] * a0[None, :, None] + p[:, np.minimum(sx + 1, W - 1)] * a1[None, :, None]
    S0, S1 = S[np.clip(sy, 0, H - 1)], S[np.clip(sy + 1, 0, H - 1)]
    out = (((b0[:, None, None] * (S0 >> 4)) >> 16) + ((b1[:, None, None] * (S1 >> 4)) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8)
