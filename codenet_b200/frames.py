"""Frame types CtdetDetector.run_batch takes besides uint8 BGR arrays, image paths and encoded images."""
import numpy as np
import torch


def _strides(p):
    """(row, column) strides in bytes of a 2-D uint8 array or tensor."""
    return tuple(p.strides) if isinstance(p, np.ndarray) else tuple(p.stride())


class YUV420:
    """One YUV 4:2:0 video frame (BT.601 video range, what decoders emit and OpenCV's COLOR_YUV2BGR_* converts) as three uint8
    planes: y (H, W) with H and W even, u and v (H/2, W/2).  The planes are 2-D numpy arrays, all on the host, or CUDA tensors,
    all on one device; they may be views: the Y column stride is 1, the U and V column strides are 1 or 2 and equal, the U and V
    row strides are equal, and every row stride is positive and at least the row it holds.  The usual layouts are one slicing away:

        NV12 surface s, shape (3H/2, W):  YUV420(s[:H], s[H:, 0::2], s[H:, 1::2])
        NV21 surface s:                   YUV420(s[:H], s[H:, 1::2], s[H:, 0::2])
        I420 buffer b, H*W*3/2 bytes:     YUV420(b[:H*W].reshape(H, W), b[H*W:H*W*5//4].reshape(H//2, W//2),
                                                 b[H*W*5//4:].reshape(H//2, W//2))

    to_bgr(frame) defines what the frame is: cv2.cvtColor(..., COLOR_YUV2BGR_I420) of its planes."""
    __slots__ = ("y", "u", "v")

    def __init__(self, y, u, v):
        planes = (y, u, v)
        for name, p in zip("yuv", planes):
            if isinstance(p, torch.Tensor):
                if not p.is_cuda:
                    raise ValueError("YUV420: plane %s is a CPU tensor; host planes are numpy arrays" % name)
                ok = p.dtype == torch.uint8
            elif isinstance(p, np.ndarray):
                ok = p.dtype == np.uint8
            else:
                raise ValueError("YUV420: plane %s is a %s, not a numpy array or CUDA tensor" % (name, type(p).__name__))
            if not ok or p.ndim != 2:
                raise ValueError("YUV420: plane %s must be 2-D uint8, got %s %s" % (name, p.dtype, tuple(p.shape)))
        cuda = {isinstance(p, torch.Tensor) for p in planes}
        if len(cuda) != 1:
            raise ValueError("YUV420: planes must be all on the host or all on the device, not mixed")
        if cuda == {True} and len({p.device for p in planes}) != 1:
            raise ValueError("YUV420: planes on different devices")
        H, W = (int(s) for s in y.shape)
        if H <= 0 or W <= 0 or H % 2 or W % 2:
            raise ValueError("YUV420: Y is %d x %d; 4:2:0 needs a positive even height and width" % (H, W))
        if tuple(u.shape) != (H // 2, W // 2) or tuple(v.shape) != (H // 2, W // 2):
            raise ValueError("YUV420: U %s and V %s must be (%d, %d) for Y (%d, %d)"
                             % (tuple(u.shape), tuple(v.shape), H // 2, W // 2, H, W))
        (ys, yc), (us, uc), (vs, vc) = _strides(y), _strides(u), _strides(v)
        if yc != 1:
            raise ValueError("YUV420: the Y column stride must be 1, got %d" % yc)
        if uc not in (1, 2) or vc != uc:
            raise ValueError("YUV420: the U and V column strides must be equal and 1 or 2, got %d and %d" % (uc, vc))
        if us != vs or ys < W or us < (W // 2 - 1) * uc + 1:
            raise ValueError("YUV420: row strides Y %d, U %d, V %d: U and V must be equal and every row must fit its stride"
                             % (ys, us, vs))
        self.y, self.u, self.v = y, u, v

    @property
    def shape(self):
        """(H, W) of the frame."""
        return tuple(int(s) for s in self.y.shape)

    @property
    def is_cuda(self):
        return isinstance(self.y, torch.Tensor)


def to_bgr(frame):
    """The uint8 BGR (H, W, 3) host image a YUV420 frame stands for: cv2.cvtColor(i420, COLOR_YUV2BGR_I420) of its planes copied
    to the host."""
    import cv2
    y, u, v = (p.cpu().numpy() if isinstance(p, torch.Tensor) else p for p in (frame.y, frame.u, frame.v))
    H, W = frame.shape
    i420 = np.concatenate([y.reshape(-1), u.reshape(-1), v.reshape(-1)]).reshape(H * 3 // 2, W)
    return cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420)
