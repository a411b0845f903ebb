"""Host side of the device merge (codenet_b200/csrc/merge.cu) without a GPU: the argument checks of the C ABI, the numpy
restatement of soft-NMS's parallel placement against the sequential mirror, and the scale-batch planning of run()."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200 import _lib
from codenet_b200.compat import soft_nms
from codenet_b200.compat.detector import plan_scale_batches, MERGE_MAX_ROWS
from oracle.soft_nms_place import place, soft_nms_parallel

INVALID = -1
FAKE = C.c_void_p(16)               # never dereferenced: every call below is rejected before anything touches the device


def test_argument_checks_run_on_the_host():
    lib = _lib.load()
    one = np.ones(5, np.float32)
    sp = C.c_void_p(one.ctypes.data)
    assert lib.cdn_soft_nms(FAKE, FAKE, 4, MERGE_MAX_ROWS + 1, 0.5, 0.5, 0.001, 2, FAKE, None) == INVALID
    assert b"up to 1024 rows" in lib.cdn_last_error()
    assert lib.cdn_soft_nms(FAKE, FAKE, 4, 10, 0.5, 0.5, 0.001, 3, FAKE, None) == INVALID          # method
    assert lib.cdn_soft_nms(None, FAKE, 4, 10, 0.5, 0.5, 0.001, 2, FAKE, None) == INVALID
    assert lib.cdn_soft_nms(FAKE, FAKE, -1, 10, 0.5, 0.5, 0.001, 2, FAKE, None) == INVALID
    assert lib.cdn_soft_nms(FAKE, FAKE, 0, 10, 0.5, 0.5, 0.001, 2, FAKE, None) == 0                # nothing to launch
    merge = lambda S, K, nc, scales=sp, mpi=100: lib.cdn_ctdet_merge(FAKE, FAKE, 1, S, K, nc, scales, 1, mpi, FAKE, FAKE, None)
    assert merge(11, 100, 20) == INVALID and b"scales x K" in lib.cdn_last_error()
    assert merge(17, 10, 20) == INVALID                                                            # CDN_MERGE_MAX_SCALES
    assert merge(2, 100, 1025) == INVALID and merge(2, 100, 0) == INVALID                           # CDN_MERGE_MAX_CLASSES
    assert merge(2, 100, 20, mpi=0) == INVALID
    assert merge(1, 100, 20, scales=None) == INVALID
    bad = np.array([1.0, 0.0], np.float32)
    assert lib.cdn_ctdet_merge(FAKE, FAKE, 1, 2, 100, 20, C.c_void_p(bad.ctypes.data), 0, 100, FAKE, FAKE, None) == INVALID
    assert b"scale 1" in lib.cdn_last_error()
    assert lib.cdn_ctdet_merge(FAKE, FAKE, 0, 5, 100, 20, sp, 0, 100, FAKE, FAKE, None) == 0          # empty batch: no launch


def _boxes(rng, n, spread=60.0, size=(-3.0, 40.0), scores=None):
    c = rng.uniform(0, spread, (n, 2)); wh = rng.uniform(size[0], size[1], (n, 2))
    s = rng.uniform(0, 1, (n, 1)) ** 3 if scores is None else rng.choice(scores, (n, 1))
    return np.concatenate([c - wh / 2, c + wh / 2, s], 1).astype(np.float32)


def test_parallel_placement_restates_the_mirror(golden):
    """oracle/soft_nms_place.py (the placement cdn_soft_nms computes from the discard flags alone) against compat.soft_nms:
    the reference's own vectors, then dense clusters (long discard chains, copies from the tail, a discarded last row), exact
    ties, zero- and negative-width boxes and scores just above the threshold, for the three methods and three Nt."""
    g = golden("soft_nms_kat.npz")
    for key in g.files:
        if key.endswith("_in"):
            tag = key[:-3]
            a = g[key].copy()
            assert soft_nms_parallel(a, Nt=0.5, method=int(tag.split("_m")[1])) == int(g[tag + "_keep"])
            np.testing.assert_array_equal(a, g[tag + "_out"], err_msg=tag)
    rng = np.random.default_rng(11)
    cases = [_boxes(rng, n) for n in (0, 1, 2, 31, 33, 70)]
    cases += [_boxes(rng, 60, spread=4.0, size=(20.0, 24.0)), _boxes(rng, 50, spread=3.0, size=(10.0, 12.0), scores=[0.0012, 0.002, 0.9])]
    cases += [_boxes(rng, 40, scores=[0.25, 0.5, 0.5, 0.75]), _boxes(rng, 40, size=(-6.0, 1.0))]
    for b in cases:
        for method in (0, 1, 2):
            for Nt in (0.3, 0.5, 0.7):
                for thr in (0.001, 0.3):
                    a, r = b.copy(), b.copy()
                    n = soft_nms_parallel(a, sigma=0.5, Nt=Nt, threshold=thr, method=method)
                    keep = soft_nms(r, sigma=0.5, Nt=Nt, threshold=thr, method=method)
                    np.testing.assert_array_equal(a, r)
                    assert n == len(keep)


def test_placement_cases():
    """The placement rule by hand: holes filled from the top of the back region, and the mirror's last self-copy."""
    assert place([False] * 4) == (4, [])
    assert place([True, False, False, False]) == (3, [(0, 3)])                  # row 3 moves into hole 0
    assert place([True, False, True, False]) == (2, [(0, 3), (2, 2)])           # back: 3 unflagged fills hole 0, 2 self-copies
    assert place([False, False, True, True]) == (2, [(2, 3)])                   # back rows 2, 3 flagged: slot 2 ends as row 3
    assert place([False, False, False, True]) == (3, [(3, 3)])                  # last row discarded onto itself
    assert place([True]) == (0, [(0, 0)])
    assert place([True, True, True]) == (0, [(0, 1)])


def test_scale_batch_planning():
    """run()'s batches: one per distinct network input size in order of first appearance, scales in order inside one."""
    assert plan_scale_batches([(512, 512)] * 5) == [((512, 512), [0, 1, 2, 3, 4])]
    assert plan_scale_batches([]) == []
    assert plan_scale_batches([(256, 384), (512, 512), (256, 384), (128, 128)]) == [((256, 384), [0, 2]), ((512, 512), [1]),
                                                                                   ((128, 128), [3])]


def test_scale_batch_planning_of_the_detector():
    """Under fix_res every test scale has the network's input size, so all scales of an image go into one engine batch;
    without it (keep_res) every scale has its own padded size."""
    from codenet_b200.compat.detector import CtdetDetector, default_opt
    det = CtdetDetector.__new__(CtdetDetector)
    det.opt = default_opt(test_scales=[0.5, 0.75, 1.0, 1.25, 1.5])
    for h, w in ((300, 400), (400, 300)):
        sizes = [det.input_geometry(h, w, s)[1] for s in det.opt.test_scales]
        assert plan_scale_batches(sizes) == [((512, 512), [0, 1, 2, 3, 4])]
    det.opt.fix_res = False
    sizes = [det.input_geometry(300, 400, s)[1] for s in det.opt.test_scales]
    assert [hw for hw, _ in plan_scale_batches(sizes)] == [(160, 224), (256, 320), (320, 416), (384, 512), (480, 608)]
