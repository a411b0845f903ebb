"""The multi-scale merge on the device (codenet_b200/csrc/merge.cu): cdn_soft_nms against the compiled reference's vectors and
the host mirror compat.soft_nms, cdn_ctdet_merge against CtdetDetector.merge_outputs, and CtdetDetector.run() (all test scales
in one engine batch + the device merge) against the host composition pre_process -> process -> post_process -> merge_outputs."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200.arch import NetConfig
from codenet_b200.synth import make_quant_state

pytestmark = pytest.mark.gpu
CFG = NetConfig(num_classes=20)
LIMIT = 1024


def _device_nms(segs, **kw):
    import torch
    from codenet_b200.compat.nms import soft_nms_device
    off = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int64)
    rows = np.concatenate([s.reshape(-1, 5) for s in segs], 0).astype(np.float32) if segs else np.zeros((0, 5), np.float32)
    d = torch.from_numpy(rows).cuda().contiguous()
    keep = soft_nms_device(d, off, **kw).cpu().numpy()
    out = d.cpu().numpy()
    return [out[off[g]:off[g + 1]] for g in range(len(segs))], keep


def test_soft_nms_golden_cases_in_one_launch(golden):
    """All 36 cases of the compiled reference's soft_nms (tests/golden/soft_nms_kat.npz), one segment each, one launch per
    method (the method is a launch argument): rows and keep counts equal to the reference's."""
    g = golden("soft_nms_kat.npz")
    tags = sorted(k[:-3] for k in g.files if k.endswith("_in"))
    assert len(tags) == 36
    for method in (0, 1, 2):
        mine = [t for t in tags if t.endswith("_m%d" % method)]
        out, keep = _device_nms([g[t + "_in"] for t in mine], Nt=0.5, method=method)
        for t, o, k in zip(mine, out, keep):
            np.testing.assert_array_equal(o, g[t + "_out"], err_msg=t)
            assert k == int(g[t + "_keep"]), t


def _case(rng, n, kind):
    if kind == "cluster":                            # dense: long discard chains, copies from the tail, discarded last rows
        c = rng.uniform(0, 6, (n, 2)); wh = rng.uniform(30, 34, (n, 2)); s = rng.uniform(0.0005, 0.05, (n, 1))
    elif kind == "ties":                             # exact score ties for the max rule
        c = rng.uniform(0, 80, (n, 2)); wh = rng.uniform(5, 40, (n, 2)); s = rng.choice([0.125, 0.25, 0.5, 0.75], (n, 1))
    elif kind == "degenerate":                       # zero- and negative-width boxes: iw <= 0 and ih <= 0 branches
        c = rng.uniform(0, 30, (n, 2)); wh = rng.choice([-3.0, -1.0, -0.5, 0.0, 2.0, 10.0], (n, 2)); s = rng.uniform(0, 1, (n, 1))
    else:                                            # scores just above the threshold
        c = rng.uniform(0, 40, (n, 2)); wh = rng.uniform(8, 30, (n, 2))
        s = np.float32(0.001) * (1 + rng.integers(0, 64, (n, 1)) * np.float32(2 ** -10))
    return np.concatenate([c - wh / 2, c + wh / 2, s], 1).astype(np.float32)


def test_soft_nms_random_segments_equal_the_mirror():
    """Segment lengths 0 ... the limit in one launch, every method and Nt, against compat.soft_nms row for row."""
    from codenet_b200.compat import soft_nms
    rng = np.random.default_rng(21)
    kinds = ("cluster", "ties", "degenerate", "threshold")
    lengths = (0, 1, 2, 31, 32, 33, 127, 500, LIMIT)
    for method in (0, 1, 2):
        for Nt in (0.3, 0.5, 0.7):
            segs = [_case(rng, n, kinds[(i + method) % 4]) for i, n in enumerate(lengths)]
            segs += [_case(rng, 200, k) for k in kinds]
            out, keep = _device_nms(segs, sigma=0.5, Nt=Nt, threshold=0.001, method=method)
            for i, (s, o, k) in enumerate(zip(segs, out, keep)):
                r = s.copy()
                n = len(soft_nms(r, sigma=0.5, Nt=Nt, threshold=0.001, method=method))
                np.testing.assert_array_equal(o, r, err_msg="method %d Nt %g segment %d" % (method, Nt, i))
                assert k == n


def test_oversize_segment_is_rejected_before_launch():
    import torch
    from codenet_b200 import _lib
    from codenet_b200.compat.nms import soft_nms_device
    rows = torch.from_numpy(_case(np.random.default_rng(2), LIMIT + 6, "ties")).cuda()
    before = rows.clone()
    with pytest.raises(_lib.CdnError, match="up to 1024 rows"):
        soft_nms_device(rows, [0, 5, LIMIT + 6], method=2)
    torch.cuda.synchronize()
    assert torch.equal(rows, before)


def _fake_detector(nc, scales, nms):
    from codenet_b200.compat.detector import CtdetDetector
    det = CtdetDetector.__new__(CtdetDetector)
    det.num_classes, det.max_per_image, det.scales = nc, 100, list(scales)
    det.opt = type("O", (), {"nms": nms})()
    return det


def _host_post(dets, nc, scale):
    """What post_process returns for dets already in image space: grouped per class, coordinates / scale in float32."""
    cls = dets[:, 5].astype(np.int64)
    out = {j + 1: np.ascontiguousarray(dets[cls == j, :5], dtype=np.float32).reshape(-1, 5) for j in range(nc)}
    if scale != 1:
        for v in out.values():
            v[:, :4] /= scale
    return out


@pytest.mark.parametrize("S", [1, 2, 5])
@pytest.mark.parametrize("nms", [False, True])
def test_merge_equals_merge_outputs(S, nms):
    """cdn_ctdet_merge for several images per call against merge_outputs on the same per-scale detections: totals below, at
    and above max_per_image, score ties exactly at the cut, empty classes and zero padding rows of class 0."""
    import torch
    from codenet_b200 import _lib
    L = _lib.load()
    nc, rng = 20, np.random.default_rng(30 + S + 10 * nms)
    scales = [0.5, 0.75, 1.0, 1.25, 1.5][:S] if S > 1 else [1.0]
    for K in (60 // S, 100 // S, 100, min(200, LIMIT // S)):
        B = 3
        dets = np.zeros((B * S, K, 6), np.float32)
        for i in range(B * S):
            n = int(rng.integers(K // 2, K + 1))              # the rest stay zero padding rows (class 0, score 0)
            c = rng.uniform(0, 300, (n, 2)); wh = rng.uniform(8, 80, (n, 2))
            dets[i, :n, :4] = np.concatenate([c - wh / 2, c + wh / 2], 1)
            dets[i, :n, 4] = rng.choice(np.float32([0.05, 0.1, 0.2, 0.3, 0.5, 0.9]), n) if i % 2 else np.sort(rng.uniform(0, 1, n))[::-1]
            dets[i, :n, 5] = rng.choice([0, 3, 4, 7, 19], n)    # most classes empty
        d = torch.from_numpy(dets).cuda()
        g = torch.empty_like(d); counts = torch.empty((B * S, nc), dtype=torch.int32, device="cuda")
        rows = torch.full((B, S * K, 5), np.nan, dtype=torch.float32, device="cuda")
        ccnt = torch.empty((B, nc), dtype=torch.int32, device="cuda")
        sc = np.asarray(scales, np.float32)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(L.cdn_ctdet_group_by_class(C.c_void_p(d.data_ptr()), B * S, K, nc, C.c_void_p(g.data_ptr()), C.c_void_p(counts.data_ptr()), st))
        _lib.check(L.cdn_ctdet_merge(C.c_void_p(g.data_ptr()), C.c_void_p(counts.data_ptr()), B, S, K, nc, C.c_void_p(sc.ctypes.data),
                                     int(nms), 100, C.c_void_p(rows.data_ptr()), C.c_void_p(ccnt.data_ptr()), st))
        rows, ccnt = rows.cpu().numpy(), ccnt.cpu().numpy()
        det = _fake_detector(nc, scales, nms)
        for b in range(B):
            want = det.merge_outputs([_host_post(dets[b * S + s], nc, scales[s]) for s in range(S)])
            ends = np.cumsum(ccnt[b])
            for j in range(nc):
                np.testing.assert_array_equal(rows[b, ends[j] - ccnt[b, j]:ends[j]], want[j + 1], err_msg="K %d image %d class %d" % (K, b, j))


def _detector(calib, res, **kw):
    from codenet_b200 import compat
    from codenet_b200.compat.detector import default_opt
    st = make_quant_state(CFG, calib, "round", res)
    opt = default_opt(state_dict=st, offset_mode="round", input_h=res, input_w=res, **kw)
    return compat.CtdetDetector(opt)


def _host_composition(det, img):
    """The reference's run(): per scale pre_process -> process -> post_process, then merge_outputs, all through the host."""
    import torch
    per_scale = []
    for scale in det.scales:
        images, meta = det.pre_process(img, scale)
        _, dets = det.process(images.cuda())
        per_scale.append(det.post_process(dets, meta, scale))
    return det.merge_outputs(per_scale)


def _prefetched(det, img):
    """What test.py's prefetch loader hands to run(): the image plus pre_process's tensors and metas per scale."""
    import torch
    images, metas = {}, {}
    for scale in det.scales:
        x, m = det.pre_process(img, scale)
        images[scale], metas[scale] = x[None], m
    return {"image": torch.from_numpy(img)[None], "images": images, "meta": metas}


def _count_engine_runs(monkeypatch):
    from codenet_b200.engine import Engine
    calls = []
    orig = Engine.run

    def counted(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    monkeypatch.setattr(Engine, "run", counted)
    return calls


def test_run_batches_the_scales_and_merges_on_the_device(calib, monkeypatch):
    """run() with 5 test scales, x flip, x nms, on landscape and portrait raw frames and on prefetched dicts: results per class
    equal to the host composition, with one engine call per image."""
    pytest.importorskip("cv2")
    det = _detector(calib, 256, max_batch=10, test_scales=[0.5, 0.75, 1.0, 1.25, 1.5])
    rng = np.random.default_rng(40)
    frames = [rng.integers(0, 256, (300, 400, 3), dtype=np.uint8), rng.integers(0, 256, (400, 300, 3), dtype=np.uint8)]
    calls = _count_engine_runs(monkeypatch)
    for flip in (False, True):
        for nms in (False, True):
            det.opt.flip_test, det.opt.nms = flip, nms
            for img in frames:
                want = _host_composition(det, img)
                for src in (img, _prefetched(det, img)):
                    del calls[:]
                    ret = det.run(src)
                    assert len(calls) == 1
                    assert set(ret) == {"results", "tot", "load", "pre", "net", "dec", "post", "merge"}
                    for j in range(1, 21):
                        np.testing.assert_array_equal(ret["results"][j], want[j], err_msg="flip %s nms %s class %d" % (flip, nms, j))
    det.opt.flip_test = det.opt.nms = False


def test_run_single_scale_input_sized_and_host_pre_process(calib):
    """Scale 1 with --nms on an input-sized frame (copied as it is) and with device_pre_process off (host pre_process)."""
    pytest.importorskip("cv2")
    det = _detector(calib, 256, max_batch=10, test_scales=[1.0], nms=True)
    rng = np.random.default_rng(41)
    for img in (rng.integers(0, 256, (256, 256, 3), dtype=np.uint8), rng.integers(0, 256, (300, 400, 3), dtype=np.uint8)):
        want = _host_composition(det, img)
        for dpp in (True, False):
            det.opt.device_pre_process = dpp
            got = det.run(img)["results"]
            for j in range(1, 21):
                np.testing.assert_array_equal(got[j], want[j])
    det.opt.device_pre_process = True


def test_run_falls_back_to_the_host_merge_beyond_the_limit(calib, monkeypatch):
    """11 scales x K = 100 rows exceed the device merge's 1024: run() merges that image on the host, same results."""
    pytest.importorskip("cv2")
    from codenet_b200.compat import detector as D
    det = _detector(calib, 256, max_batch=11, test_scales=[0.5 + 0.1 * i for i in range(11)])
    img = np.random.default_rng(42).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    used = []
    orig = D.CtdetDetector.merge_outputs
    monkeypatch.setattr(D.CtdetDetector, "merge_outputs", lambda self, d: used.append(1) or orig(self, d))
    got = det.run(img)["results"]
    assert used == [1]
    want = _host_composition(det, img)
    for j in range(1, 21):
        np.testing.assert_array_equal(got[j], want[j])


def test_float_model_run_with_two_scales_and_nms(golden):
    """The unquantised model keeps one network call per scale and merges on the device: run() equal to the host composition."""
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
                      input_w=256, test_scales=[1.0, 1.5], nms=True, device_pre_process=False)
    det = compat.CtdetDetector(opt)
    img = np.random.default_rng(43).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    got = det.run(img)["results"]
    want = _host_composition(det, img)
    for j in range(1, 21):
        np.testing.assert_array_equal(got[j], want[j])
