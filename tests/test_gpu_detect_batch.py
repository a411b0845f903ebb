"""The batched detector (CtdetDetector.run_batch) and its ragged pre-process (cdn_warp_affine_u8_batch): the ragged warp against
the one-frame cdn_warp_affine_u8 and the OpenCV restatement oracle.warp_ref, and run_batch against run() frame for frame."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200.arch import NetConfig
from codenet_b200.synth import make_quant_state

pytestmark = pytest.mark.gpu
CFG = NetConfig(num_classes=20)


def _ragged(frames, jobs, dst_slots, dh, dw, gap=lambda i: 0, fill=77):
    """jobs: [(frame index, M, dst slot, mirror slot)].  Frames go into one pool at offsets shifted by gap(i) bytes (odd ones
    included).  Returns the destination batch as numpy."""
    import torch
    from codenet_b200 import _lib
    offs, end = [], 0
    for i, f in enumerate(frames):
        end += gap(i)
        offs.append(end)
        end += f.nbytes
    pool = np.zeros(end, np.uint8)
    for o, f in zip(offs, frames):
        pool[o:o + f.nbytes] = f.reshape(-1)
    desc = np.zeros(len(jobs), _lib.WARP_DESC)
    for k, (i, M, slot, mirror) in enumerate(jobs):
        desc[k] = (offs[i], frames[i].shape[0], frames[i].shape[1], np.asarray(M, np.float64).reshape(6), slot, mirror)
    d_pool = torch.from_numpy(pool).cuda()
    dst = torch.full((dst_slots, dh, dw, 3), fill, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_u8_batch(C.c_void_p(d_pool.data_ptr()), C.c_void_p(desc.ctypes.data), len(desc),
                                                     C.c_void_p(dst.data_ptr()), dst_slots, dh, dw,
                                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst.cpu().numpy()


def _single(frame, M, dh, dw, flip):
    import torch
    from codenet_b200 import _lib
    src = torch.from_numpy(np.ascontiguousarray(frame)).cuda()
    M = np.ascontiguousarray(M, np.float64)
    dst = torch.empty((2 if flip else 1, dh, dw, 3), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_u8(C.c_void_p(src.data_ptr()), frame.shape[0], frame.shape[1], C.c_void_p(M.ctypes.data),
                                               C.c_void_p(dst.data_ptr()), dh, dw, int(flip),
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst.cpu().numpy()


@pytest.mark.parametrize("dh,dw", [(256, 256), (70, 99), (33, 6)])
def test_ragged_warp_equals_single_warp_and_oracle(dh, dw):
    """1x1, 31x17, 97x203, landscape, portrait, input-sized and larger-than-input frames, plain, rotated and scaled matrices,
    mirrors on some slots only, odd pool offsets, dst_w a multiple of 4 or not; slots no descriptor names stay untouched."""
    from oracle import warp_ref
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(50 + dw)
    shapes = [(1, 1), (31, 17), (97, 203), (300, 400), (400, 300), (dh, dw), (2 * dh + 5, 3 * dw + 1)]
    frames = [rng.integers(0, 256, s + (3,), dtype=np.uint8) for s in shapes]
    jobs, slot = [], 0
    for i, (h, w) in enumerate(shapes):
        c = np.array([w / 2., h / 2.], np.float32)
        for k, (rot, sc) in enumerate(((0, 1.0), (17, 0.8), (-40, 1.3))):
            M = get_affine_transform(c, max(h, w) * sc, rot, [dw, dh])
            mirror = (i + k) % 2 == 0
            jobs.append((i, M, slot, slot + 1 if mirror else -1))
            slot += 3 if mirror else 2                       # one slot between images stays unwritten
    got = _ragged(frames, jobs, slot, dh, dw, gap=lambda i: 2 * i + 1)
    written = set()
    for i, M, s, m in jobs:
        want = warp_ref.warp_affine(frames[i], M, (dw, dh))
        np.testing.assert_array_equal(got[s], want, err_msg="frame %s slot %d" % (shapes[i], s))
        one = _single(frames[i], M, dh, dw, m >= 0)
        np.testing.assert_array_equal(one[0], want)
        written.add(s)
        if m >= 0:
            np.testing.assert_array_equal(got[m], want[:, ::-1])
            np.testing.assert_array_equal(one[1], want[:, ::-1])
            written.add(m)
    for s in set(range(slot)) - written:
        assert (got[s] == 77).all()


def test_ragged_warp_more_descriptors_than_one_launch():
    """2.5 launches' worth of descriptors (CDN_WARP_DESC_PER_LAUNCH each) over 40 small frames, every third mirrored."""
    from oracle import warp_ref
    from codenet_b200 import _lib
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(60)
    dh, dw = 9, 14
    frames = [rng.integers(0, 256, (int(rng.integers(1, 40)), int(rng.integers(1, 40)), 3), dtype=np.uint8) for _ in range(40)]
    n = _lib.WARP_DESC_PER_LAUNCH * 5 // 2
    jobs, slot = [], 0
    for k in range(n):
        i = k % len(frames)
        h, w = frames[i].shape[:2]
        M = get_affine_transform(np.array([w / 2., h / 2.], np.float32), max(h, w) * (0.6 + 0.01 * (k % 70)), (k * 7) % 90 - 45, [dw, dh])
        mirror = k % 3 == 0
        jobs.append((i, M, slot, slot + 1 if mirror else -1))
        slot += 2 if mirror else 1
    got = _ragged(frames, jobs, slot, dh, dw, gap=lambda i: i % 5)
    for i, M, s, m in jobs:
        want = warp_ref.warp_affine(frames[i], M, (dw, dh))
        np.testing.assert_array_equal(got[s], want, err_msg="slot %d" % s)
        if m >= 0:
            np.testing.assert_array_equal(got[m], want[:, ::-1])


def _detector(calib, res, **kw):
    from codenet_b200 import compat
    from codenet_b200.compat.detector import default_opt
    st = make_quant_state(CFG, calib, "round", res)
    opt = default_opt(state_dict=st, offset_mode="round", input_h=res, input_w=res, **kw)
    return compat.CtdetDetector(opt)


def _frames(seed, n=11):
    rng = np.random.default_rng(seed)
    shapes = [(300, 400), (400, 300), (256, 256), (97, 203), (375, 500), (500, 333), (40, 31), (256, 300), (600, 700),
              (333, 500), (128, 64)]
    return [rng.integers(0, 256, shapes[i % len(shapes)] + (3,), dtype=np.uint8) for i in range(n)]


def _count_engine_runs(monkeypatch):
    from codenet_b200.engine import Engine
    calls = []
    orig = Engine.run

    def counted(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    monkeypatch.setattr(Engine, "run", counted)
    return calls


def _assert_same(got, want, nc=20, tag=""):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert set(g) == {"results", "tot", "load", "pre", "net", "dec", "post", "merge"}
        for j in range(1, nc + 1):
            np.testing.assert_array_equal(g["results"][j], w[j], err_msg="%s frame %d class %d" % (tag, i, j))


@pytest.mark.parametrize("scales,max_batch", [([1.0], 3), ([0.5, 1.0, 1.5], 6)])
def test_run_batch_equals_run(calib, monkeypatch, scales, max_batch):
    """11 mixed raw frames at 256^2, steps small enough that both staging buffers are reused: run_batch's results equal run()'s
    frame for frame, x flip, x nms, with ceil(frames / frames per step) engine calls."""
    pytest.importorskip("cv2")
    det = _detector(calib, 256, max_batch=max_batch, test_scales=scales)
    frames = _frames(70)
    for flip in (False, True):
        for nms in (False, True):
            det.opt.flip_test, det.opt.nms = flip, nms
            want = [det.run(f)["results"] for f in frames]
            calls = _count_engine_runs(monkeypatch)
            got = det.run_batch(frames)
            spf = len(scales) * (2 if flip else 1)
            per_step = max(max_batch, spf) // spf
            assert len(calls) == -(-len(frames) // per_step) and len(calls) >= 4
            monkeypatch.undo()
            _assert_same(got, want, tag="flip %s nms %s" % (flip, nms))
            again = det.run_batch(frames[3:5])                     # a later call on the same buffers, a partial step
            _assert_same(again, want[3:5], tag="second call")
    det.opt.flip_test = det.opt.nms = False


def test_run_batch_timers_sum_to_the_call(calib):
    import time
    det = _detector(calib, 256, max_batch=4, test_scales=[1.0])
    frames = _frames(71, 6)
    det.run_batch(frames)
    t0 = time.time()
    got = det.run_batch(frames)
    wall = time.time() - t0
    tot = sum(g["tot"] for g in got)
    assert 0 < tot <= wall + 1e-6
    parts = sum(g[k] for g in got for k in ("load", "pre", "net", "dec", "post", "merge"))
    assert parts <= tot + 1e-6 and len({g["tot"] for g in got}) == 1


def test_run_batch_paths_equal_arrays(calib, tmp_path):
    cv2 = pytest.importorskip("cv2")
    det = _detector(calib, 256, max_batch=4, test_scales=[1.0], flip_test=True)
    frames = _frames(72, 5)
    paths = []
    for i, f in enumerate(frames):
        p = str(tmp_path / ("f%d.png" % i))
        assert cv2.imwrite(p, f)
        paths.append(p)
    want = [det.run(f)["results"] for f in frames]
    _assert_same(det.run_batch(paths), want, tag="paths")
    _assert_same(det.run_batch([paths[0], frames[1], paths[2], frames[3], paths[4]]), want, tag="mixed")


def test_run_batch_host_merge_beyond_the_limit(calib, monkeypatch):
    """11 scales x K = 100 rows exceed the device merge's 1024: every frame is merged on the host, same results as run()."""
    pytest.importorskip("cv2")
    from codenet_b200.compat import detector as D
    det = _detector(calib, 256, max_batch=11, test_scales=[0.5 + 0.1 * i for i in range(11)])
    frames = _frames(73, 3)
    want = [det.run(f)["results"] for f in frames]
    used = []
    orig = D.CtdetDetector.merge_outputs
    monkeypatch.setattr(D.CtdetDetector, "merge_outputs", lambda self, d: used.append(1) or orig(self, d))
    got = det.run_batch(frames)
    assert used == [1, 1, 1]
    _assert_same(got, want, tag="host merge")


def test_float_model_run_batch_equals_run(golden):
    import torch
    pytest.importorskip("cv2")
    from codenet_b200 import compat
    from codenet_b200.compat.detector import default_opt
    from codenet_b200.synth import make_raw_state
    g = golden("codenet_float_1x_256.npz")
    raw = make_raw_state(CFG, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    opt = default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()}, input_h=256,
                      input_w=256, test_scales=[1.0, 1.5], nms=True)
    det = compat.CtdetDetector(opt)
    frames = _frames(74, 3)
    want = [det.run(f)["results"] for f in frames]
    _assert_same(det.run_batch(frames), want, tag="float")
