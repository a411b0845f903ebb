"""TEST INFRASTRUCTURE (never imported by the product): numpy restatement of the parallel form of soft-NMS that
codenet_b200/csrc/merge.cu runs, checked against the sequential mirror compat.soft_nms (lib/models/external/nms.pyx:77-170).

Within one outer iteration i of the mirror, every row examined by the inner loop is decayed by the same max row (row i after
the swap), and every row of [i+1, N) is examined exactly once: a discarded row is overwritten by a copy of row N-1, which has
not been examined yet.  So the decayed score and the discard flag of each row depend on that row alone and can be computed in
parallel.  What stays sequential in the mirror is where the rows land, and that depends on the flags alone:

  * F = number of flagged rows, N' = N - F.  Front region [i+1, N'), back region [N', N).
  * Unflagged front rows stay where they are (with their decayed score).
  * The flagged front rows are holes.  The k-th hole (ascending) receives the k-th unflagged back row counted from the top
    (descending), with its decayed score.  There are as many unflagged back rows as holes.
  * Back-region rows keep their content from before the pass (stale copies), except in one case: when the back region has
    flagged rows below its lowest unflagged row (R = that row, or N if there is none, and R > N'), the mirror's last step
    discards the row at slot N' = N - 1 onto itself.  Slot N' then holds the decayed row N' + 1 if R - N' >= 2 (it was
    copied into slot N' before), else the decayed row N'.
"""
import numpy as np

F = np.float32
D = np.float64


def decay(t, r, sigma, Nt, method):
    """(decayed score, flag-eligible) of row r against the max row t, compat.soft_nms's float/double sequence."""
    tx1, ty1, tx2, ty2 = (F(v) for v in t[:4])
    x1, y1, x2, y2 = (F(v) for v in r[:4])
    area = F((D(F(x2 - x1)) + 1.0) * (D(F(y2 - y1)) + 1.0))
    iw = F(D(F(min(tx2, x2) - max(tx1, x1))) + 1.0)
    if not iw > 0:
        return r[4], False
    ih = F(D(F(min(ty2, y2) - max(ty1, y1))) + 1.0)
    if not ih > 0:
        return r[4], False
    ua = F((D(F(tx2 - tx1)) + 1.0) * (D(F(ty2 - ty1)) + 1.0) + D(area) - D(F(iw * ih)))
    ov = F(F(iw * ih) / ua)
    if method == 1:
        weight = F(1.0 - D(ov)) if ov > Nt else F(1)
    elif method == 2:
        weight = F(np.exp(D(F(F(-F(ov * ov)) / sigma))))
    else:
        weight = F(0) if ov > Nt else F(1)
    return F(weight * r[4]), True


def place(flags):
    """flags [n] bool for rows A..A+n-1 (relative indices) -> (n_kept, moves) with moves = list of (dst, src) relative
    indices: dst receives the decayed src row.  Rows neither a dst nor moved keep their own decayed (front) or stale (back)
    content; see the module docstring."""
    flags = np.asarray(flags, bool)
    n = flags.size
    nk = n - int(flags.sum())
    holes = np.nonzero(flags[:nk])[0]
    back = np.arange(nk, n)
    up = back[~flags[nk:]][::-1]                       # unflagged back rows, descending
    assert holes.size == up.size
    moves = list(zip(holes.tolist(), up.tolist()))
    R = int(up[-1]) if up.size else n
    if R > nk:                                         # flagged rows under the lowest unflagged back row: self-copy at nk
        moves.append((nk, nk + 1 if R - nk >= 2 else nk))
    return nk, moves


def soft_nms_parallel(boxes, sigma=0.5, Nt=0.3, threshold=0.001, method=0):
    """compat.soft_nms computed in the parallel form: same in-place result, returns the final N."""
    assert boxes.ndim == 2 and boxes.dtype == np.float32 and boxes.shape[1] >= 5
    sigma, Nt, threshold = F(sigma), F(Nt), F(threshold)
    N = boxes.shape[0]
    i = 0
    while i < N:
        s = boxes[i:N, 4]
        m = i + int(np.argmax(s == s.max())) if not np.isnan(s).any() else i     # first maximum, row i wins ties
        t = boxes[m, :5].copy()
        boxes[m, :5] = boxes[i, :5]
        boxes[i, :5] = t
        A = i + 1
        dec = np.empty(N - A, np.float32)
        flags = np.zeros(N - A, bool)
        for k in range(N - A):
            dec[k], hit = decay(t, boxes[A + k], sigma, Nt, method)
            flags[k] = hit and dec[k] < threshold
        nk, moves = place(flags)
        old = boxes[A:N, :5].copy()
        for k in range(nk):                            # front rows in place
            boxes[A + k, 4] = dec[k]
        for dst, src in moves:
            boxes[A + dst, :4] = old[src, :4]
            boxes[A + dst, 4] = dec[src]
        N = A + nk
        i += 1
    return N
