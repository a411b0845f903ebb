"""TEST INFRASTRUCTURE ONLY.  numpy restatement of OpenCV's YUV 4:2:0 -> BGR conversion, cv2.cvtColor(frame,
COLOR_YUV2BGR_I420 | _YV12 | _NV12 | _NV21), for planes given as arrays of any strides.

OpenCV (color_yuv.simd.hpp, third-party; this container has cv2 4.13) converts every pixel with one fixed-point function of its
Y and of the U, V samples of its 2x2 block: BT.601 video range with a 20-bit shift, y' = max(Y - 16, 0) * CY and
channel = saturate((y' + 2^19 + C_u * (U - 128) + C_v * (V - 128)) >> 20).  The four layouts differ only in where U and V sit,
which the caller expresses as views (I420: planar U then V; YV12: V then U; NV12: interleaved UV; NV21: VU).  Composed with
oracle.warp_ref it is the reference of cdn_warp_affine_src_u8_batch's YUV sources (tests/test_frames_cpu.py pins it against cv2)."""
import numpy as np

SHIFT = 20
CY, CUB, CUG, CVG, CVR = 1220542, 2116026, -409993, -852492, 1673527


def yuv420_to_bgr(y, u, v):
    """y: uint8 (H, W), H and W even; u, v: uint8 (H/2, W/2) -> uint8 BGR (H, W, 3)."""
    y, u, v = (np.asarray(p) for p in (y, u, v))
    H, W = y.shape
    assert H % 2 == 0 and W % 2 == 0 and u.shape == v.shape == (H // 2, W // 2)
    uu = np.repeat(np.repeat(u.astype(np.int32) - 128, 2, 0), 2, 1)
    vv = np.repeat(np.repeat(v.astype(np.int32) - 128, 2, 0), 2, 1)
    yy = np.maximum(y.astype(np.int32) - 16, 0) * CY + (1 << (SHIFT - 1))
    out = np.empty((H, W, 3), np.uint8)
    out[..., 0] = np.clip((yy + CUB * uu) >> SHIFT, 0, 255)
    out[..., 1] = np.clip((yy + CVG * vv + CUG * uu) >> SHIFT, 0, 255)
    out[..., 2] = np.clip((yy + CVR * vv) >> SHIFT, 0, 255)
    return out
