"""Host-side mirror of the reference's `soft_nms` (lib/models/external/nms.pyx:77-170), used by
`CtdetDetector.merge_outputs` for multi-scale testing and `--nms` (lib/detectors/ctdet.py:59-74), and its device form
`soft_nms_device` (cdn_soft_nms, many segments in one launch), which CtdetDetector.run() reaches through cdn_ctdet_merge.

The reference runs this on the CPU (compiled Cython).  The restatement keeps the reference's in-place semantics and its single-precision arithmetic (`cdef float` temporaries; `np.exp` evaluated
in double and rounded to float), so results are bit-identical to the compiled reference (tests/golden/soft_nms_kat.npz):

  * `boxes` [N, 5] float32 (x1, y1, x2, y2, score) is modified IN PLACE: selection-sorts by score, decays the scores of
    overlapping boxes, and overwrites a box whose score falls below `threshold` with a COPY of the last box (the discarded
    box is lost; rows past the final N keep stale copies with their scores from before that pass);
  * the outer loop runs over the ORIGINAL N (Cython evaluates `range(N)` once) while the inner loops use the shrinking N;
  * returns `list(range(N_final))`, which `merge_outputs` ignores -- it keeps every row of the modified array.
"""
import numpy as np

F = np.float32
D = np.float64


def soft_nms(boxes, sigma=0.5, Nt=0.3, threshold=0.001, method=0):
    assert boxes.ndim == 2 and boxes.dtype == np.float32 and boxes.shape[1] >= 5
    n0 = N = boxes.shape[0]
    sigma, Nt, threshold, one = F(sigma), F(Nt), F(threshold), F(1)
    for i in range(n0):
        maxscore, maxpos = boxes[i, 4], i
        tx1, ty1, tx2, ty2, ts = (F(v) for v in boxes[i, :5])
        pos = i + 1
        while pos < N:                                   # get max box
            if maxscore < boxes[pos, 4]:
                maxscore, maxpos = boxes[pos, 4], pos
            pos += 1
        boxes[i, :5] = boxes[maxpos, :5]                 # add max box as a detection
        boxes[maxpos, :5] = (tx1, ty1, tx2, ty2, ts)     # swap ith box with position of max box
        tx1, ty1, tx2, ty2, ts = (F(v) for v in boxes[i, :5])
        pos = i + 1
        while pos < N:                                   # N shrinks when a box falls below the threshold
            x1, y1, x2, y2 = (F(v) for v in boxes[pos, :4])
            # Differences of two floats are single precision; the `+ 1` is a double addition (Cython types the literal as
            # 1.0), so the products / sums that follow run in double and are rounded once on assignment to the
            # `cdef float` (checked against the compiled reference, Cython 3.x: tests/golden/soft_nms_kat.npz).
            area = F((D(F(x2 - x1)) + 1.0) * (D(F(y2 - y1)) + 1.0))
            iw = F(D(F(min(tx2, x2) - max(tx1, x1))) + 1.0)
            if iw > 0:
                ih = F(D(F(min(ty2, y2) - max(ty1, y1))) + 1.0)
                if ih > 0:
                    ua = F((D(F(tx2 - tx1)) + 1.0) * (D(F(ty2 - ty1)) + 1.0) + D(area) - D(F(iw * ih)))
                    ov = F(F(iw * ih) / ua)              # iou between max box and detection box
                    if method == 1:                      # linear
                        weight = F(1.0 - D(ov)) if ov > Nt else one
                    elif method == 2:                    # gaussian
                        weight = F(np.exp(D(F(F(-F(ov * ov)) / sigma))))
                    else:                                # original NMS
                        weight = F(0) if ov > Nt else one
                    boxes[pos, 4] = F(weight * boxes[pos, 4])
                    if boxes[pos, 4] < threshold:        # discard the box by swapping with the last box
                        boxes[pos, :5] = boxes[N - 1, :5]
                        N -= 1
                        pos -= 1
            pos += 1
    return list(range(N))


def soft_nms_device(boxes, seg_off, sigma=0.5, Nt=0.3, threshold=0.001, method=0):
    """soft_nms on the device over independent segments: `boxes` CUDA float32 [rows, 5] (contiguous), segment g = rows
    seg_off[g] .. seg_off[g+1] (host sequence of n_seg + 1 non-decreasing offsets), each modified in place exactly as
    soft_nms(boxes[seg], sigma, Nt, threshold, method) modifies its array.  Returns the keep counts (len of soft_nms's
    result) as an int32 CUDA tensor [n_seg]; asynchronous on the current stream.  A segment longer than
    CDN_SOFT_NMS_MAX_LEN (1024) rows raises CdnError before anything is launched."""
    import ctypes as C
    import torch
    from .. import _lib
    if not (torch.is_tensor(boxes) and boxes.is_cuda and boxes.dtype == torch.float32 and boxes.dim() == 2 and boxes.shape[1] == 5
            and boxes.is_contiguous()):
        raise ValueError("soft_nms_device takes a contiguous CUDA float32 [rows, 5] tensor")
    off = np.asarray(seg_off, dtype=np.int64).reshape(-1)
    if off.size < 1 or off[0] < 0 or off[-1] > boxes.shape[0] or (np.diff(off) < 0).any():
        raise ValueError("seg_off must be non-decreasing offsets into the rows of boxes")
    n_seg = off.size - 1
    max_len = int(np.diff(off).max()) if n_seg else 0
    keep = torch.empty(n_seg, dtype=torch.int32, device=boxes.device)
    d_off = torch.from_numpy(off.astype(np.int32)).to(boxes.device)
    with torch.cuda.device(boxes.device):
        _lib.check(_lib.load().cdn_soft_nms(C.c_void_p(boxes.data_ptr()), C.c_void_p(d_off.data_ptr()), n_seg, max_len, float(sigma),
                                            float(Nt), float(threshold), int(method), C.c_void_p(keep.data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream(boxes.device).cuda_stream)))
    return keep
