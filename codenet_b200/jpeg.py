"""Baseline JPEG decoding on the device (csrc/jpeg.cu): cdn_jpeg_parse on the host, cdn_jpeg_decode_batch on the GPU.

decode_jpeg(buffers) returns what cv2.imdecode(buf, cv2.IMREAD_COLOR) returns for every buffer, as uint8 CUDA tensors
[H, W, 3] (BGR).  Streams the parser accepts are decoded on the device in one call; the others, and the frames the device
flags (corrupt data), are decoded by cv2 on the host, frame by frame.
"""
import ctypes as C

import numpy as np

from . import _lib

# cdn_jpeg_huff / cdn_jpeg_frame (include/codenet_b200.h); sizes asserted here and in csrc/jpeg.cu
JPEG_HUFF = np.dtype([("maxcode", np.int32, (18,)), ("valoffset", np.int32, (18,)), ("look", np.uint16, (256,)),
                      ("huffval", np.uint8, (256,))], align=True)
JPEG_FRAME = np.dtype([("width", np.int32), ("height", np.int32), ("ncomp", np.int32), ("hmax", np.int32), ("vmax", np.int32),
                       ("mcux", np.int32), ("mcuy", np.int32), ("restart_interval", np.int32), ("nsegments", np.int32),
                       ("pad0", np.int32), ("nbytes", np.int64), ("scan_offset", np.int64), ("scan_end", np.int64),
                       ("comp_h", np.int32, (3,)), ("comp_v", np.int32, (3,)), ("comp_bw", np.int32, (3,)),
                       ("comp_bh", np.int32, (3,)), ("comp_dw", np.int32, (3,)), ("comp_dh", np.int32, (3,)),
                       ("comp_dc", np.int32, (3,)), ("comp_ac", np.int32, (3,)), ("ws_bytes", np.int64), ("coef_rel", np.int64),
                       ("plane_rel", np.int64, (3,)), ("qt", np.uint16, (3, 64)), ("huff", JPEG_HUFF, (4,)),
                       ("data_offset", np.int64), ("out_offset", np.int64), ("ws_offset", np.int64)], align=True)
assert JPEG_HUFF.itemsize == 912 and JPEG_FRAME.itemsize == 4256

HOST_REASONS = {1: "process", 2: "precision", 3: "color", 4: "sampling", 5: "scan", 6: "orientation", 7: "size"}
ERRORS = {-1: "not a JPEG", -2: "truncated", -3: "bad segment", -4: "bad table"}
BAD_CODE, BAD_END, BAD_RESTART, BAD_RANGE = 1, 2, 4, 8          # CDN_JPEG_BAD_*
ALIGN = 16                      # streams and decoded frames in a pool start at multiples of ALIGN bytes
WS_ALIGN = 256


def as_bytes(buf):
    """bytes | bytearray | memoryview | 1-D uint8 array -> 1-D uint8 array over the same bytes (no copy where possible)."""
    if isinstance(buf, np.ndarray):
        if buf.dtype != np.uint8 or buf.ndim != 1:
            raise ValueError("an encoded image is a 1-D uint8 array, got %s %s" % (buf.dtype, buf.shape))
        return np.ascontiguousarray(buf)
    if isinstance(buf, (bytes, bytearray, memoryview)):
        return np.frombuffer(buf, np.uint8)
    raise ValueError("an encoded image is bytes, bytearray, memoryview or a 1-D uint8 array, not %s" % type(buf).__name__)


def parse(buf, out=None):
    """cdn_jpeg_parse of one encoded image -> (status, descriptor): 0 = the device decodes it, > 0 = a host reason
    (HOST_REASONS), < 0 = not a parseable JPEG.  `out` (a JPEG_FRAME record view, e.g. one row of a staging table) is filled
    in place when given."""
    data = as_bytes(buf)
    desc = np.zeros(1, JPEG_FRAME) if out is None else out
    rc = _lib.load().cdn_jpeg_parse(C.c_void_p(data.ctypes.data), data.size, C.c_void_p(desc.ctypes.data))
    return rc, desc


def imdecode_host(buf):
    """cv2.imdecode(buf, cv2.IMREAD_COLOR) or ValueError when cv2 cannot read it."""
    import cv2
    img = cv2.imdecode(as_bytes(buf), cv2.IMREAD_COLOR)
    if img is None:
        raise ValueError("cannot decode image (%d bytes)" % as_bytes(buf).size)
    return img


def layout(desc, base, stream_sizes, out_base):
    """Places n parsed frames: streams back to back from byte `base` of a pool, decoded frames from `out_base` of the output
    buffer, workspaces back to back.  Fills data_offset, out_offset, ws_offset of `desc` and returns
    (stream offsets, end of the streams, end of the outputs, workspace bytes)."""
    offs, end = [], base
    for nb in stream_sizes:
        offs.append(end)
        end += -(-int(nb) // ALIGN) * ALIGN
    out = out_base
    ws = 0
    for i in range(len(desc)):
        desc[i]["data_offset"] = offs[i]
        desc[i]["out_offset"] = out
        desc[i]["ws_offset"] = ws
        out += -(-int(desc[i]["width"]) * int(desc[i]["height"]) * 3 // ALIGN) * ALIGN
        ws += int(desc[i]["ws_bytes"])
    return offs, end, out, ws


def decode_batch(d_pool, pool_bytes, desc, d_desc, d_ws, ws_bytes, d_out, out_bytes, d_status, stream):
    """cdn_jpeg_decode_batch on raw device pointers (ints), desc the host JPEG_FRAME array."""
    _lib.check(_lib.load().cdn_jpeg_decode_batch(C.c_void_p(d_pool), int(pool_bytes), C.c_void_p(desc.ctypes.data), C.c_void_p(d_desc),
                                                 len(desc), C.c_void_p(d_ws), int(ws_bytes), C.c_void_p(d_out), int(out_bytes),
                                                 C.c_void_p(d_status), C.c_void_p(stream)))


def decode_jpeg(buffers, device=None, return_status=False):
    """cv2.imdecode(buf, cv2.IMREAD_COLOR) of every encoded image in `buffers` as uint8 CUDA tensors [H, W, 3] on `device`.
    Accepted streams go to the device in one host-to-device copy (descriptor table, then the streams) and are decoded by one
    cdn_jpeg_decode_batch call; the rest, and frames the device flags, are decoded by cv2 on the host.  Raises ValueError
    for an input neither can read.  With return_status, also returns [(parse status, device status or None)] per buffer."""
    import torch
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    datas = [as_bytes(b) for b in buffers]
    table = np.zeros(len(datas), JPEG_FRAME)
    codes = [parse(d, table[i:i + 1])[0] for i, d in enumerate(datas)]
    on_dev = [i for i, c in enumerate(codes) if c == 0]
    out = [None] * len(datas)
    dstat = [None] * len(datas)
    if on_dev:
        desc = np.ascontiguousarray(table[on_dev])
        head = -(-desc.nbytes // ALIGN) * ALIGN
        offs, end, out_end, ws_bytes = layout(desc, head, [datas[i].size for i in on_dev], 0)
        host = np.zeros(end, np.uint8)
        for k, i in enumerate(on_dev):
            host[offs[k]:offs[k] + datas[i].size] = datas[i]
        host[:desc.nbytes] = desc.view(np.uint8)
        with torch.cuda.device(dev):
            pool = torch.from_numpy(host).to(dev)
            ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
            pix = torch.empty(max(out_end, 1), dtype=torch.uint8, device=dev)
            status = torch.empty(len(on_dev), dtype=torch.int32, device=dev)
            decode_batch(pool.data_ptr(), end, desc, pool.data_ptr(), ws.data_ptr(), ws.numel(), pix.data_ptr(), pix.numel(),
                         status.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
            st = status.cpu().numpy()
        for k, i in enumerate(on_dev):
            dstat[i] = int(st[k])
            if st[k] == 0:
                h, w, o = int(desc[k]["height"]), int(desc[k]["width"]), int(desc[k]["out_offset"])
                out[i] = pix[o:o + h * w * 3].view(h, w, 3)
    for i, d in enumerate(datas):
        if out[i] is None:
            out[i] = torch.from_numpy(imdecode_host(d)).to(dev)
    return (out, list(zip(codes, dstat))) if return_status else out
