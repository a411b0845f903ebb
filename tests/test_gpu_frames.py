"""run_batch from frames already on the GPU and from YUV 4:2:0 frames: cdn_warp_affine_src_u8[_f32]_batch against oracle.yuv_ref +
oracle.warp_ref bit for bit, and run_batch against run() frame for frame for both models."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200.arch import NetConfig
from codenet_b200.synth import make_quant_state

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _i420(bgr):
    """The I420 buffer (3H/2, W) of a BGR frame, as a video decoder would give it."""
    return cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)


def _nv12(i420):
    H = i420.shape[0] * 2 // 3
    W = i420.shape[1]
    flat = i420.reshape(-1)
    u, v = flat[H * W:H * W * 5 // 4], flat[H * W * 5 // 4:]
    return np.concatenate([flat[:H * W], np.stack([u, v], -1).reshape(-1)]).reshape(H * 3 // 2, W)


def _views(s, layout):
    """(y, u, v) views of a surface s (numpy or torch) of shape (3H/2, W)."""
    H = s.shape[0] * 2 // 3
    W = s.shape[1]
    if layout == "I420":
        flat = s.reshape(-1)
        return s[:H], flat[H * W:H * W * 5 // 4].reshape(H // 2, W // 2), flat[H * W * 5 // 4:].reshape(H // 2, W // 2)
    if layout == "NV12":
        return s[:H], s[H:, 0::2], s[H:, 1::2]
    return s[:H], s[H:, 1::2], s[H:, 0::2]                  # NV21 view of an NV12 surface: U and V swapped


def _sources(rng, shapes):
    """For every shape one source of each kind: [(kind, device object, host BGR it stands for)] with kinds pool (BGR in a shared
    pool at an odd offset), crop (pitched CUDA BGR crop of a larger tensor), I420, NV12, NV21 (views of one CUDA surface)."""
    import torch
    from oracle import yuv_ref
    out = []
    for h, w in shapes:
        bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        out.append(("pool", bgr, bgr))
        big = torch.from_numpy(rng.integers(0, 256, (h + 5, w + 7, 3), dtype=np.uint8)).cuda()
        big[2:2 + h, 3:3 + w] = torch.from_numpy(bgr).cuda()
        out.append(("crop", big[2:2 + h, 3:3 + w], bgr))
        i420 = _i420(bgr)
        d_i420, d_nv12 = torch.from_numpy(i420).cuda(), torch.from_numpy(_nv12(i420)).cuda()
        for layout, surf in (("I420", d_i420), ("NV12", d_nv12), ("NV21", d_nv12)):
            planes = _views(surf, layout)
            out.append((layout, planes, yuv_ref.yuv420_to_bgr(*(p.cpu().numpy() for p in planes))))
    return out


def _descs(sources, jobs, pool_keep):
    """jobs: [(source index, M, slot, mirror)] -> WARP_SRC_DESC array; pool sources go into one CUDA pool at odd offsets."""
    import torch
    from codenet_b200 import _lib
    offs, end = {}, 0
    for i, (kind, obj, _) in enumerate(sources):
        if kind == "pool":
            end += 3
            offs[i] = end
            end += obj.nbytes
    pool = np.zeros(max(end, 1), np.uint8)
    for i, o in offs.items():
        pool[o:o + sources[i][1].nbytes] = sources[i][1].reshape(-1)
    d_pool = torch.from_numpy(pool).cuda()
    pool_keep.append(d_pool)
    d = np.zeros(len(jobs), _lib.WARP_SRC_DESC)
    for k, (i, M, slot, mirror) in enumerate(jobs):
        kind, obj, bgr = sources[i]
        h, w = bgr.shape[:2]
        if kind == "pool":
            row = ((d_pool.data_ptr() + offs[i], 0, 0), (3 * w, 0), _lib.WARP_SRC_BGR, 1)
        elif kind == "crop":
            row = ((obj.data_ptr(), 0, 0), (obj.stride(0), 0), _lib.WARP_SRC_BGR, 1)
        else:
            y, u, v = obj
            row = ((y.data_ptr(), u.data_ptr(), v.data_ptr()), (y.stride(0), u.stride(0)), _lib.WARP_SRC_YUV420, u.stride(1))
        d[k] = row + (h, w, np.asarray(M, np.float64).reshape(6), slot, mirror)
    return d


def _run_u8(desc, slots, dh, dw):
    import torch
    from codenet_b200 import _lib
    dst = torch.full((slots, dh, dw, 3), 77, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_src_u8_batch(C.c_void_p(desc.ctypes.data), len(desc), C.c_void_p(dst.data_ptr()), slots,
                                                         dh, dw, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst.cpu().numpy()


def _run_f32(desc, table, tables, slots, dh, dw):
    import torch
    from codenet_b200 import _lib
    table = np.ascontiguousarray(table, np.int32)
    d_tables = torch.from_numpy(np.ascontiguousarray(tables, np.float32)).cuda()
    dst = torch.full((slots, 3, dh, dw), 77.0, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().cdn_warp_affine_src_u8_f32_batch(
        C.c_void_p(desc.ctypes.data), C.c_void_p(table.ctypes.data), len(desc), C.c_void_p(d_tables.data_ptr()), len(tables),
        C.c_void_p(dst.data_ptr()), slots, dh, dw, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst.cpu().numpy()


def _check(sources, jobs, dh, dw, seed):
    """Both entry points on one ragged batch: u8 slots equal the oracle's warp of the source's BGR image (mirrors reversed), the
    fp32 slots that warp looked up in the descriptor's table."""
    from oracle import warp_ref
    keep = []
    desc = _descs(sources, jobs, keep)
    slots = max(max(s, m) for _, _, s, m in jobs) + 1
    got = _run_u8(desc, slots, dh, dw)
    tables = np.random.default_rng(seed).standard_normal((2, 3, 256)).astype(np.float32)
    table = [(k // 3) % 2 for k in range(len(jobs))]
    got_f = _run_f32(desc, table, tables, slots, dh, dw)
    for k, (i, M, s, m) in enumerate(jobs):
        want = warp_ref.warp_affine(sources[i][2], M, (dw, dh))
        tag = "%s %s slot %d" % (sources[i][0], sources[i][2].shape[:2], s)
        np.testing.assert_array_equal(got[s], want, err_msg=tag)
        np.testing.assert_array_equal(got_f[s], np.stack([tables[table[k]][c][want[..., c]] for c in range(3)]), err_msg=tag)
        if m >= 0:
            np.testing.assert_array_equal(got[m], want[:, ::-1], err_msg=tag + " mirror")
            np.testing.assert_array_equal(got_f[m], got_f[s][..., ::-1], err_msg=tag + " mirror")


@pytest.mark.parametrize("dh,dw", [(64, 64), (70, 99)])
def test_src_warp_equals_oracle(dh, dw):
    """Pool BGR, pitched CUDA crops and I420 / NV12 / NV21 views of one surface from 2x2 to 1920x1080 in one ragged batch, plain,
    rotated and scaled matrices, mirrors on some slots, dst_w a multiple of 4 or not."""
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(200 + dw)
    sources = _sources(rng, [(2, 2), (30, 18), (96, 202), (dh, dw - dw % 2), (1080, 1920)])     # 4:2:0 sizes are even
    jobs, slot = [], 0
    for i, (_, _, bgr) in enumerate(sources):
        h, w = bgr.shape[:2]
        for k, (rot, sc) in enumerate(((0, 1.0), (17, 0.8))):
            M = get_affine_transform(np.array([w / 2., h / 2.], np.float32), max(h, w) * sc, rot, [dw, dh])
            mirror = (i + k) % 2 == 0
            jobs.append((i, M, slot, slot + 1 if mirror else -1))
            slot += 2 if mirror else 1
    _check(sources, jobs, dh, dw, dw)


def test_src_warp_more_descriptors_than_one_launch():
    """2.5 launches' worth of descriptors of either form (CDN_WARP_SRC_DESC_PER_LAUNCH, CDN_WARP_SRC_F32_DESC_PER_LAUNCH) cycling
    over every source kind, every third mirrored."""
    from codenet_b200 import _lib
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(210)
    sources = _sources(rng, [(2 * int(rng.integers(1, 20)), 2 * int(rng.integers(1, 20))) for _ in range(6)])
    dh, dw = 9, 14
    n = max(_lib.WARP_SRC_DESC_PER_LAUNCH, _lib.WARP_SRC_F32_DESC_PER_LAUNCH) * 5 // 2
    jobs, slot = [], 0
    for k in range(n):
        i = k % len(sources)
        h, w = sources[i][2].shape[:2]
        M = get_affine_transform(np.array([w / 2., h / 2.], np.float32), max(h, w) * (0.6 + 0.01 * (k % 70)), (k * 7) % 90 - 45, [dw, dh])
        jobs.append((i, M, slot, slot + 1 if k % 3 == 0 else -1))
        slot += 2 if k % 3 == 0 else 1
    _check(sources, jobs, dh, dw, 211)


# ---- run_batch ------------------------------------------------------------------------------------------------------------
CFG = NetConfig(num_classes=20)


def _detector(calib, res, **kw):
    from codenet_b200 import compat
    from codenet_b200.compat.detector import default_opt
    st = make_quant_state(CFG, calib, "round", res)
    return compat.CtdetDetector(default_opt(state_dict=st, offset_mode="round", input_h=res, input_w=res, **kw))


SHAPES = [(300, 400), (400, 300), (256, 256), (96, 202), (376, 500), (500, 334), (40, 30), (256, 300), (600, 700)]


def _mixed(rng, tmp_path, n):
    """n frames cycling through every input kind: [(frame, what run() is given for it, kind)]."""
    import torch
    from codenet_b200.frames import YUV420, to_bgr
    out = []
    for i in range(n):
        bgr = rng.integers(0, 256, SHAPES[i % len(SHAPES)] + (3,), dtype=np.uint8)
        kind = ("array", "path", "jpeg", "cuda", "yuv", "cuda_nv12")[i % 6]
        if kind == "array":
            out.append((bgr, bgr, kind))
        elif kind in ("path", "jpeg"):
            ok, buf = cv2.imencode(".jpg", bgr, [cv2.IMWRITE_JPEG_QUALITY, 90])
            assert ok
            dec = cv2.imdecode(buf, cv2.IMREAD_COLOR)
            if kind == "path":
                p = tmp_path / ("f%d.jpg" % i)
                p.write_bytes(buf.tobytes())
                out.append((str(p), dec, kind))
            else:
                out.append((buf.tobytes(), dec, kind))
        elif kind == "cuda":
            big = torch.from_numpy(rng.integers(0, 256, (bgr.shape[0] + 4, bgr.shape[1] + 6, 3), dtype=np.uint8)).cuda()
            t = big[1:1 + bgr.shape[0], 5:5 + bgr.shape[1]]
            t.copy_(torch.from_numpy(bgr).cuda())
            out.append((t, t.cpu().numpy(), kind))
        elif kind == "yuv":
            f = YUV420(*_views(_i420(bgr), "I420"))
            out.append((f, to_bgr(f), kind))
        else:
            f = YUV420(*_views(torch.from_numpy(_nv12(_i420(bgr))).cuda(), "NV12"))
            out.append((f, to_bgr(f), kind))
    return out


def _count(monkeypatch, cls, names):
    calls = {k: 0 for k in names}
    for name in names:
        orig = getattr(cls, name)

        def counted(self, *a, _name=name, _orig=orig, **k):
            calls[_name] += 1
            return _orig(self, *a, **k)
        monkeypatch.setattr(cls, name, counted)
    return calls


def _assert_same(got, want, nc, tag):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        for j in range(1, nc + 1):
            np.testing.assert_array_equal(g["results"][j], w[j], err_msg="%s frame %d class %d" % (tag, i, j))


@pytest.mark.parametrize("scales,flip,nms,max_batch", [([1.0], False, False, 4), ([1.0], True, False, 8),
                                                        ([0.5, 0.75, 1.0, 1.25, 1.5], True, True, 10)])
def test_run_batch_mixed_inputs_equal_run(calib, monkeypatch, tmp_path, scales, flip, nms, max_batch):
    """Host arrays, paths, JPEG bytes (decoded on the device at scale 1: the threshold is lowered to 2 frames per step), CUDA BGR
    crops, host I420 and CUDA NV12 frames in one call: every result equals run() of the frame's BGR image, with
    ceil(frames / frames per step) engine calls and one warp launch per step (the general-source one at scale 1)."""
    from codenet_b200.engine import Engine
    from codenet_b200.compat import detector as D
    det = _detector(calib, 256, max_batch=max_batch, test_scales=scales, flip_test=flip, nms=nms)
    frames = _mixed(np.random.default_rng(220), tmp_path, 14)
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    monkeypatch.setattr(D, "JPEG_DEVICE_MIN_FRAMES", 2)
    items = det._batch_frames([f for f, _, _ in frames])
    if scales == [1.0]:
        assert [it[1] is not None for it in items] == [k in ("path", "jpeg") for _, _, k in frames]
    engine = _count(monkeypatch, Engine, ["run"])
    warps = _count(monkeypatch, D.CtdetDetector, ["_warp", "_warp_src"])
    got = det.run_batch([f for f, _, _ in frames])
    spf = len(scales) * (2 if flip else 1)
    per_step = max(max_batch, spf) // spf
    kinds = [k for _, _, k in frames]
    steps = -(-len(frames) // per_step)
    assert engine["run"] == steps and warps["_warp"] + warps["_warp_src"] == steps
    if scales == [1.0]:                                   # the steps holding a CUDA or YUV frame take the general-source warp
        direct = sum(any(k in ("cuda", "yuv", "cuda_nv12") for k in kinds[i:i + per_step]) for i in range(0, len(frames), per_step))
        assert 0 < direct < steps and warps["_warp_src"] == direct
    monkeypatch.undo()
    _assert_same(got, want, 20, "scales %s flip %s" % (scales, flip))


def test_run_batch_of_cuda_frames_stages_no_bytes(calib, monkeypatch, tmp_path):
    """A call of only CUDA frames (BGR crops and NV12 surfaces) stages nothing: no staging buffer is asked for, so no frame byte
    crosses PCIe, and the results equal run()'s."""
    from codenet_b200.compat import detector as D
    det = _detector(calib, 256, max_batch=4, test_scales=[1.0], flip_test=True)
    frames = [x for x in _mixed(np.random.default_rng(230), tmp_path, 18) if x[2] in ("cuda", "cuda_nv12")]
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    staged = []
    orig = D.CtdetDetector._staging
    monkeypatch.setattr(D.CtdetDetector, "_staging", lambda self, st, b, nbytes, pool_bytes=None:
                        staged.append(nbytes) or orig(self, st, b, nbytes, pool_bytes))
    got = det.run_batch([f for f, _, _ in frames])
    assert sum(staged) == 0
    _assert_same(got, want, 20, "cuda only")
    # a host YUV420 frame is staged at 1.5 bytes per pixel (16-byte aligned planes)
    staged.clear()
    yuv = [x for x in _mixed(np.random.default_rng(231), tmp_path, 6) if x[2] == "yuv"][0]
    det.run_batch([yuv[0]])
    h, w = yuv[0].shape
    assert staged == [sum(-(-nb // 16) * 16 for nb in (h * w, h * w // 4, h * w // 4))]


@pytest.mark.parametrize("tag,gemm", [("1x", "fp32"), ("2x_coco", "tf32x3")])
def test_float_model_run_batch_mixed_inputs_equal_run(golden, monkeypatch, tmp_path, tag, gemm):
    import torch
    from codenet_b200 import compat
    from codenet_b200.compat import detector as D
    from codenet_b200.compat.detector import default_opt
    from codenet_b200.synth import make_raw_state
    cfg = NetConfig(num_classes=20) if tag == "1x" else NetConfig(num_classes=80, w2=True)
    g = golden("codenet_float_%s_256.npz" % tag)
    raw = make_raw_state(cfg, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    nc = cfg.num_classes
    opt = default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()}, input_h=256,
                      input_w=256, f32_gemm=gemm, heads={"hm": nc, "wh": 2, "reg": 2}, num_classes=nc, w2=cfg.w2,
                      test_scales=[1.0], flip_test=True, max_batch=6)
    det = compat.CtdetDetector(opt)
    frames = _mixed(np.random.default_rng(240), tmp_path, 8)
    want = [det.run(ref)["results"] for _, ref, _ in frames]
    warps = _count(monkeypatch, D.CtdetDetector, ["_warp_f32", "_warp_src_f32"])
    got = det.run_batch([f for f, _, _ in frames])
    assert warps == {"_warp_f32": 2, "_warp_src_f32": 1}         # steps of 3 frames: only the second holds CUDA or YUV ones
    monkeypatch.undo()
    _assert_same(got, want, nc, "float %s" % tag)


def test_cuda_frame_on_another_device_is_rejected(calib):
    import torch
    from codenet_b200.frames import YUV420
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    det = _detector(calib, 256)
    other = torch.device("cuda", 1 - det.opt.device.index)
    with pytest.raises(ValueError, match="detector runs on"):
        det.run_batch([torch.zeros((8, 8, 3), dtype=torch.uint8, device=other)])
    s = torch.zeros((12, 8), dtype=torch.uint8, device=other)
    with pytest.raises(ValueError, match="detector runs on"):
        det.run_batch([YUV420(*_views(s, "NV12"))])


def test_cuda_frame_checks(calib):
    import torch
    det = _detector(calib, 256)
    t = torch.zeros((8, 10, 3), dtype=torch.uint8, device="cuda")
    for bad, match in ((t.float(), "uint8"), (t[..., :2], "uint8"), (t.permute(1, 0, 2), "strides"),
                       (torch.zeros((8, 10, 4), dtype=torch.uint8, device="cuda")[..., :3], "strides")):
        with pytest.raises(ValueError, match=match):
            det.run_batch([bad])
