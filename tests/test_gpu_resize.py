"""The device resize: cdn_warp_affine_resize_u8[_f32]_batch against oracle.warp_ref of oracle.resize_ref bit for bit over every source
kind, and run_batch with opt.device_resize at scale lists other than [1] against run() frame for frame, for every input kind and
both models."""
import ctypes as C

import numpy as np
import pytest

import test_gpu_frames as F
from codenet_b200.compat.detector import device_resize_exact

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

FIVE = [0.5, 0.75, 1.0, 1.25, 1.5]


def _rs_descs(sources, jobs, keep):
    """jobs: [(source index, (rs_h, rs_w), M, slot, mirror)] -> WARP_RS_DESC array (F._descs' sources, M on the resized image)."""
    from codenet_b200.compat.detector import _rs_descs
    s = F._descs(sources, [(i, M, slot, mirror) for i, _, M, slot, mirror in jobs], keep)
    return _rs_descs(s, [rs for _, rs, _, _, _ in jobs])


def _run(desc, slots, dh, dw, table, tables):
    import torch
    from codenet_b200 import _lib
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    dst = torch.full((slots, dh, dw, 3), 77, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_resize_u8_batch(C.c_void_p(desc.ctypes.data), len(desc), C.c_void_p(dst.data_ptr()), slots,
                                                            dh, dw, st))
    table = np.ascontiguousarray(table, np.int32)
    d_tables = torch.from_numpy(np.ascontiguousarray(tables, np.float32)).cuda()
    dst_f = torch.full((slots, 3, dh, dw), 77.0, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_resize_u8_f32_batch(
        C.c_void_p(desc.ctypes.data), C.c_void_p(table.ctypes.data), len(desc), C.c_void_p(d_tables.data_ptr()), len(tables),
        C.c_void_p(dst_f.data_ptr()), slots, dh, dw, st))
    return dst.cpu().numpy(), dst_f.cpu().numpy()


def _check(sources, jobs, dh, dw, seed):
    """Both entry points on one ragged batch: u8 slot = warp_ref(resize_ref(the source's BGR image)), fp32 slot = that looked up in
    the descriptor's table, mirrors reversed."""
    from oracle import resize_ref, warp_ref
    keep = []
    desc = _rs_descs(sources, jobs, keep)
    slots = max(max(s, m) for _, _, _, s, m in jobs) + 1
    tables = np.random.default_rng(seed).standard_normal((2, 3, 256)).astype(np.float32)
    table = [(k // 3) % 2 for k in range(len(jobs))]
    got, got_f = _run(desc, slots, dh, dw, table, tables)
    for k, (i, (rh, rw), M, s, m) in enumerate(jobs):
        bgr = sources[i][2]
        want = warp_ref.warp_affine(resize_ref.resize(bgr, (rw, rh)), M, (dw, dh))
        tag = "%s %s -> %s slot %d" % (sources[i][0], bgr.shape[:2], (rh, rw), s)
        np.testing.assert_array_equal(got[s], want, err_msg=tag)
        np.testing.assert_array_equal(got_f[s], np.stack([tables[table[k]][c][want[..., c]] for c in range(3)]), err_msg=tag)
        if m >= 0:
            np.testing.assert_array_equal(got[m], want[:, ::-1], err_msg=tag + " mirror")
            np.testing.assert_array_equal(got_f[m], got_f[s][..., ::-1], err_msg=tag + " mirror")


def _jobs(sources, dh, dw, rng, scales):
    """The detector's matrices for every source at every scale (a random one per source among them), every other one mirrored."""
    from codenet_b200.compat.detector import get_affine_transform
    jobs, slot = [], 0
    for i, (_, _, bgr) in enumerate(sources):
        h, w = bgr.shape[:2]
        for sc in list(scales) + [float(rng.uniform(0.3, 2.5))]:
            rh, rw = int(h * sc), int(w * sc)
            if not device_resize_exact(h, w, rh, rw):
                continue
            M = get_affine_transform(np.array([rw / 2., rh / 2.], np.float32), float(max(rh, rw)), 0, [dw, dh])
            mirror = len(jobs) % 2 == 0
            jobs.append((i, (rh, rw), M, slot, slot + 1 if mirror else -1))
            slot += 2 if mirror else 1
    return jobs


@pytest.mark.parametrize("dh,dw,shapes", [(64, 64, [(2, 2), (30, 18), (376, 500), (1080, 1920)]),
                                          (70, 99, [(2, 2), (96, 202), (480, 640), (500, 334)])])
def test_resize_warp_equals_oracle(dh, dw, shapes):
    """Pool BGR, pitched CUDA crops and I420 / NV12 / NV21 views from 2 x 2 to 1920 x 1080 in one ragged batch at the five standard
    scales and a random one, mirrors on some slots, dst_w a multiple of 4 or not."""
    rng = np.random.default_rng(300 + dw)
    sources = F._sources(rng, shapes)
    _check(sources, _jobs(sources, dh, dw, rng, FIVE), dh, dw, dw)


def test_resize_warp_odd_and_tiny_frames():
    """BGR frames of odd sizes down to 1 x 1 (pool sources and pitched CUDA crops) at the standard scales, 2 and 0.3."""
    import torch
    rng = np.random.default_rng(310)
    sources = []
    for h, w in [(1, 1), (3, 5), (7, 2), (33, 47), (375, 500), (333, 500)]:
        bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        big = torch.from_numpy(rng.integers(0, 256, (h + 3, w + 5, 3), dtype=np.uint8)).cuda()
        big[1:1 + h, 2:2 + w] = torch.from_numpy(bgr).cuda()
        sources += [("pool", bgr, bgr), ("crop", big[1:1 + h, 2:2 + w], bgr)]
    _check(sources, _jobs(sources, 40, 52, rng, FIVE + [2.0, 0.3]), 40, 52, 311)


def test_resize_warp_more_descriptors_than_one_launch():
    """2.5 launches' worth of descriptors of either form cycling over every source kind."""
    from codenet_b200 import _lib
    rng = np.random.default_rng(320)
    sources = F._sources(rng, [(2 * int(rng.integers(1, 20)), 2 * int(rng.integers(1, 20))) for _ in range(4)])
    n = max(_lib.WARP_RS_DESC_PER_LAUNCH, _lib.WARP_RS_F32_DESC_PER_LAUNCH) * 5 // 2
    jobs = []
    while len(jobs) < n:
        jobs += _jobs(sources, 9, 14, rng, FIVE)
    slot, out = 0, []
    for i, rs, M, _, m in jobs[:n]:
        out.append((i, rs, M, slot, slot + 1 if m >= 0 else -1))
        slot += 2 if m >= 0 else 1
    _check(sources, out, 9, 14, 321)


# ---- run_batch ------------------------------------------------------------------------------------------------------------
def _scale_cases():
    return [(FIVE, True, True, 10), (FIVE, True, False, 20), ([0.75, 1.25], False, True, 6), ([1.5], False, False, 3),
            ([1.5], True, False, 4)]


@pytest.mark.parametrize("scales,flip,nms,max_batch", _scale_cases())
def test_run_batch_multiscale_equals_run(calib, monkeypatch, tmp_path, scales, flip, nms, max_batch):
    """Host arrays, paths, JPEG bytes (decoded on the device: the threshold is lowered to 1 frame per step), CUDA BGR crops, host
    I420 and CUDA NV12 frames in one call: every result equals run() of the frame's BGR image, with ceil(frames / frames per
    step) engine calls and one warp launch per step, all of them resize launches."""
    from codenet_b200.engine import Engine
    from codenet_b200.compat import detector as D
    det = F._detector(calib, 256, device_resize=True, max_batch=max_batch, test_scales=scales, flip_test=flip, nms=nms)
    frames = F._mixed(np.random.default_rng(330), tmp_path, 12)
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    monkeypatch.setattr(D, "JPEG_DEVICE_MIN_FRAMES", 1)
    items = det._batch_frames([f for f, _, _ in frames])
    assert [it[1] is not None for it in items] == [k in ("path", "jpeg") for _, _, k in frames]
    assert all(det._resized_on_device(it) for it in items)
    engine = F._count(monkeypatch, Engine, ["run"])
    warps = F._count(monkeypatch, D.CtdetDetector, ["_warp", "_warp_src", "_pack_frame"])
    got = det.run_batch([f for f, _, _ in frames])
    spf = len(scales) * (2 if flip else 1)
    steps = -(-len(frames) // (max(max_batch, spf) // spf))
    assert engine["run"] == steps and warps["_warp_src"] == steps and warps["_warp"] == 0 and warps["_pack_frame"] == 0
    monkeypatch.undo()
    F._assert_same(got, want, 20, "scales %s flip %s nms %s" % (scales, flip, nms))


def test_run_batch_multiscale_jpeg_paths_at_48_frames_per_step(calib, tmp_path):
    """JPEG paths at the default threshold: 48 frames a step at three scales, decoded and resized on the device."""
    rng = np.random.default_rng(340)
    det = F._detector(calib, 256, device_resize=True, max_batch=48 * 3, test_scales=[0.75, 1.0, 1.25])
    paths, want = [], []
    for i in range(50):
        bgr = rng.integers(0, 256, F.SHAPES[i % len(F.SHAPES)] + (3,), dtype=np.uint8)
        ok, buf = cv2.imencode(".jpg", bgr, [cv2.IMWRITE_JPEG_QUALITY, 85])
        p = tmp_path / ("p%d.jpg" % i)
        p.write_bytes(buf.tobytes())
        paths.append(str(p))
    assert all(it[1] is not None for it in det._batch_frames(paths))
    want = [det.run(p)["results"] for p in paths]
    F._assert_same(det.run_batch(paths), want, 20, "jpeg paths")


def test_run_batch_of_cuda_frames_at_five_scales_stages_no_bytes(calib, monkeypatch, tmp_path):
    """CUDA BGR crops and NV12 surfaces at five scales with flip: no staging buffer is asked for, results equal run()'s; host
    arrays are staged once at 1x and host I420 frames at 1.5 bytes a pixel."""
    from codenet_b200.compat import detector as D
    det = F._detector(calib, 256, device_resize=True, max_batch=10, test_scales=FIVE, flip_test=True)
    mixed = F._mixed(np.random.default_rng(350), tmp_path, 18)
    frames = [x for x in mixed if x[2] in ("cuda", "cuda_nv12")]
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    staged = []
    orig = D.CtdetDetector._staging
    monkeypatch.setattr(D.CtdetDetector, "_staging", lambda self, st, b, nbytes, pool_bytes=None:
                        staged.append(nbytes) or orig(self, st, b, nbytes, pool_bytes))
    got = det.run_batch([f for f, _, _ in frames])
    assert sum(staged) == 0
    F._assert_same(got, want, 20, "cuda only")
    rnd = lambda nb: -(-nb // 16) * 16
    for kind in ("array", "yuv"):
        staged.clear()
        f, ref, _ = [x for x in mixed if x[2] == kind][0]
        got = det.run_batch([f])
        h, w = ref.shape[:2]
        assert staged == ([rnd(h * w * 3)] if kind == "array" else [sum(rnd(nb) for nb in (h * w, h * w // 4, h * w // 4))])
        F._assert_same(got, [det.run(ref)["results"]], 20, kind)


def test_run_batch_frame_outside_the_predicate_takes_the_host_path(calib, monkeypatch, tmp_path):
    """Frames whose resize device_resize_exact refuses (here: every frame of one shape) are resized by cv2 on the host and their
    copies go into the same pool and the same resize launch as the other frames; every result still equals run()'s."""
    from codenet_b200.compat import detector as D
    det = F._detector(calib, 256, device_resize=True, max_batch=20, test_scales=FIVE, flip_test=True)
    frames = F._mixed(np.random.default_rng(360), tmp_path, 12)
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    refuse = F.SHAPES[0]
    orig = D.device_resize_exact
    monkeypatch.setattr(D, "device_resize_exact", lambda H, W, sh, sw: (H, W) != refuse and orig(H, W, sh, sw))
    items = det._batch_frames([f for f, _, _ in frames])
    on_dev = [det._resized_on_device(it) for it in items]
    assert on_dev == [ref.shape[:2] != refuse for _, ref, _ in frames] and not all(on_dev)
    calls = F._count(monkeypatch, D.CtdetDetector, ["_warp", "_warp_src", "_pack_frame"])
    got = det.run_batch([f for f, _, _ in frames])
    assert calls["_warp"] == 0 and calls["_warp_src"] == 6 and calls["_pack_frame"] == on_dev.count(False)
    monkeypatch.undo()
    F._assert_same(got, want, 20, "outside the predicate")


@pytest.mark.parametrize("scales,flip,nms", [(FIVE, True, True), ([0.75, 1.25], False, False), ([1.5], True, False)])
def test_float_model_run_batch_multiscale_equals_run(golden, monkeypatch, tmp_path, scales, flip, nms):
    """The unquantised model: every input kind through cdn_warp_affine_resize_u8_f32_batch (JPEGs decoded by cv2 on the host),
    results equal run()'s."""
    import torch
    from codenet_b200 import compat
    from codenet_b200.arch import NetConfig
    from codenet_b200.compat import detector as D
    from codenet_b200.compat.detector import default_opt
    from codenet_b200.synth import make_raw_state
    cfg = NetConfig(num_classes=20)
    g = golden("codenet_float_1x_256.npz")
    raw = make_raw_state(cfg, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    opt = default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()}, input_h=256,
                      input_w=256, test_scales=scales, flip_test=flip, nms=nms, max_batch=10, device_resize=True)
    det = compat.CtdetDetector(opt)
    frames = F._mixed(np.random.default_rng(370), tmp_path, 8)
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    warps = F._count(monkeypatch, D.CtdetDetector, ["_warp_f32", "_warp_src_f32"])
    got = det.run_batch([f for f, _, _ in frames])
    spf = len(scales) * (2 if flip else 1)
    assert warps == {"_warp_f32": 0, "_warp_src_f32": -(-len(frames) // (max(10, spf) // spf))}
    monkeypatch.undo()
    F._assert_same(got, want, 20, "float %s" % scales)
