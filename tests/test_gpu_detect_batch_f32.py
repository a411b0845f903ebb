"""The unquantised model's batched detector: cdn_warp_affine_u8_f32_batch against the OpenCV restatement oracle.warp_ref looked up
in the tables, and against what run() feeds EngineF32; EngineF32's batch invariance; run_batch against run() frame for frame."""
import ctypes as C

import numpy as np
import pytest

from codenet_b200.arch import NetConfig

pytestmark = pytest.mark.gpu
CFG_1X = NetConfig(num_classes=20)
CFG_2X_COCO = NetConfig(num_classes=80, w2=True)


def _float_state(golden, tag, cfg):
    """The float state dict of tests/test_gpu_f32.py: synthetic weights with the golden file's BatchNorm statistics."""
    from codenet_b200.synth import make_raw_state
    g = golden("codenet_float_%s_256.npz" % tag)
    raw = make_raw_state(cfg, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    return raw


def _detector(golden, tag="1x", gemm="fp32", **kw):
    import torch
    from codenet_b200 import compat
    from codenet_b200.compat.detector import default_opt
    cfg = CFG_1X if tag == "1x" else CFG_2X_COCO
    raw = _float_state(golden, tag, cfg)
    nc = cfg.num_classes
    opt = default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()},
                      input_h=256, input_w=256, f32_gemm=gemm, heads={"hm": nc, "wh": 2, "reg": 2}, num_classes=nc,
                      w2=cfg.w2, **kw)
    return compat.CtdetDetector(opt)


def _warp_f32(frames, jobs, table, tables, dst_slots, dh, dw, gap=lambda i: 0, fill=77.0, dst_offset=0):
    """jobs: [(frame index, M, dst slot, mirror slot)], table[k] the table index of job k, tables fp32 [n][3][256].  Frames go into
    one pool at offsets shifted by gap(i) bytes; the destination starts dst_offset floats into its buffer.  Returns numpy
    [dst_slots][3][dh][dw]."""
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
    table = np.ascontiguousarray(table, np.int32)
    d_pool = torch.from_numpy(pool).cuda()
    d_tables = torch.from_numpy(np.ascontiguousarray(tables, np.float32)).cuda()
    n = dst_slots * 3 * dh * dw
    buf = torch.full((n + dst_offset,), fill, dtype=torch.float32, device="cuda")
    dst = buf[dst_offset:]
    _lib.check(_lib.load().cdn_warp_affine_u8_f32_batch(
        C.c_void_p(d_pool.data_ptr()), C.c_void_p(desc.ctypes.data), C.c_void_p(table.ctypes.data), len(desc),
        C.c_void_p(d_tables.data_ptr()), d_tables.shape[0], C.c_void_p(dst.data_ptr()), dst_slots, dh, dw,
        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst.cpu().numpy().reshape(dst_slots, 3, dh, dw)


def _lookup(table, u8_hwc):
    return np.stack([table[c][u8_hwc[..., c]] for c in range(3)])


def _random_tables(rng, n=2):
    return rng.standard_normal((n, 3, 256)).astype(np.float32)


@pytest.mark.parametrize("dh,dw,dst_offset", [(256, 256, 0), (256, 256, 1), (70, 99, 0), (33, 6, 0)])
def test_f32_warp_equals_oracle_then_table(dh, dw, dst_offset):
    """The ragged shapes of the u8 kernel's test (1x1 up to larger-than-input frames, plain, rotated and scaled matrices,
    mirrors on some slots, odd pool offsets, dst_w a multiple of 4 or not) with mixed table indices: every slot equals the
    oracle's warp looked up in its table, transposed to CHW, bit for bit; unnamed slots stay untouched.  dst_offset = 1 moves
    the destination off 16-byte alignment (scalar stores)."""
    from oracle import warp_ref
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(150 + dw + dst_offset)
    tables = _random_tables(rng)
    shapes = [(1, 1), (31, 17), (97, 203), (300, 400), (400, 300), (dh, dw), (2 * dh + 5, 3 * dw + 1)]
    frames = [rng.integers(0, 256, s + (3,), dtype=np.uint8) for s in shapes]
    jobs, table, slot = [], [], 0
    for i, (h, w) in enumerate(shapes):
        c = np.array([w / 2., h / 2.], np.float32)
        for k, (rot, sc) in enumerate(((0, 1.0), (17, 0.8), (-40, 1.3))):
            M = get_affine_transform(c, max(h, w) * sc, rot, [dw, dh])
            mirror = (i + k) % 2 == 0
            jobs.append((i, M, slot, slot + 1 if mirror else -1))
            table.append((i + 2 * k) % 3 % 2)
            slot += 3 if mirror else 2                       # one slot between images stays unwritten
    got = _warp_f32(frames, jobs, table, tables, slot, dh, dw, gap=lambda i: 2 * i + 1, dst_offset=dst_offset)
    written = set()
    for (i, M, s, m), t in zip(jobs, table):
        want = warp_ref.warp_affine(frames[i], M, (dw, dh))
        np.testing.assert_array_equal(got[s], _lookup(tables[t], want), err_msg="frame %s slot %d" % (shapes[i], s))
        written.add(s)
        if m >= 0:
            np.testing.assert_array_equal(got[m], _lookup(tables[t], want[:, ::-1]))
            written.add(m)
    for s in set(range(slot)) - written:
        assert (got[s] == 77.0).all()


def test_f32_warp_more_descriptors_than_one_launch():
    """2.5 launches' worth of descriptors (CDN_WARP_F32_DESC_PER_LAUNCH each) over 40 small frames, every third mirrored, the
    table index alternating in a pattern that crosses the launch boundaries."""
    from oracle import warp_ref
    from codenet_b200 import _lib
    from codenet_b200.compat.detector import get_affine_transform
    rng = np.random.default_rng(160)
    tables = _random_tables(rng)
    dh, dw = 9, 16
    frames = [rng.integers(0, 256, (int(rng.integers(1, 40)), int(rng.integers(1, 40)), 3), dtype=np.uint8) for _ in range(40)]
    n = _lib.WARP_F32_DESC_PER_LAUNCH * 5 // 2
    jobs, table, slot = [], [], 0
    for k in range(n):
        i = k % len(frames)
        h, w = frames[i].shape[:2]
        M = get_affine_transform(np.array([w / 2., h / 2.], np.float32), max(h, w) * (0.6 + 0.01 * (k % 70)), (k * 7) % 90 - 45, [dw, dh])
        mirror = k % 3 == 0
        jobs.append((i, M, slot, slot + 1 if mirror else -1))
        table.append((k // 5) % 2)
        slot += 2 if mirror else 1
    got = _warp_f32(frames, jobs, table, tables, slot, dh, dw, gap=lambda i: i % 5)
    for (i, M, s, m), t in zip(jobs, table):
        want = warp_ref.warp_affine(frames[i], M, (dw, dh))
        np.testing.assert_array_equal(got[s], _lookup(tables[t], want), err_msg="slot %d" % s)
        if m >= 0:
            np.testing.assert_array_equal(got[m], _lookup(tables[t], want[:, ::-1]))


def _frames(seed, n=11):
    rng = np.random.default_rng(seed)
    shapes = [(300, 400), (400, 300), (256, 256), (97, 203), (375, 500), (500, 333), (40, 31), (256, 300), (600, 700),
              (333, 500), (128, 64)]
    return [rng.integers(0, 256, shapes[i % len(shapes)] + (3,), dtype=np.uint8) for i in range(n)]


def _batched_input(det, frame, scales):
    """run_batch's pre-process of one frame: the fp32 NCHW slots cdn_warp_affine_u8_f32_batch writes (as torch, on the device)."""
    import torch
    from codenet_b200 import _lib
    from codenet_b200.compat.detector import plan_frame_steps
    n = 2 if det.opt.flip_test else 1
    layout = det._frame_layout(frame.shape[0], frame.shape[1], scales)
    (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in layout]], n * len(scales), 1)
    pool = np.empty(nbytes, np.uint8)
    desc = np.empty(len(scales), _lib.WARP_DESC)
    det._pack_frame(frame, layout, scales, pool, offsets[0], desc, 0)
    dst = torch.empty((n * len(scales), 3, det.opt.input_h, det.opt.input_w), dtype=torch.float32, device="cuda")
    det._warp_f32(torch.from_numpy(pool).cuda(), desc, det._table_index(scales, 1), det._norm_tables(0), dst)
    return dst


def test_f32_warp_equals_what_run_feeds_the_engine(golden):
    """Scale 1: pre_process_device + _process_float's normalisation; scales 0.5 and 1.5, and scale 1 without device_pre_process:
    pre_process.  Mirror included, bit for bit."""
    import torch
    det = _detector(golden, flip_test=True)
    for f in _frames(75, 6):
        u8, _ = det.pre_process_device(f, 1)
        want = det._normalize_device(u8).permute(0, 3, 1, 2).contiguous()
        assert torch.equal(_batched_input(det, f, [1.0]), want)
        for scale in (0.5, 1.5):
            want = det.pre_process(f, scale)[0].cuda()
            assert torch.equal(_batched_input(det, f, [scale]), want), scale
        got = _batched_input(det, f, [0.5, 1.0, 1.5])
        assert torch.equal(got[2:4], det._normalize_device(u8).permute(0, 3, 1, 2))
        det.opt.device_pre_process = False
        assert torch.equal(_batched_input(det, f, [1.0]), det.pre_process(f, 1.0)[0].cuda())
        det.opt.device_pre_process = True


@pytest.mark.parametrize("gemm", ["fp32", "tf32x3"])
@pytest.mark.parametrize("tag", ["1x", "2x_coco"])
def test_engine_f32_is_batch_invariant(golden, tag, gemm):
    """A batch of 7 differing images against each image alone: heads and detect()'s detections identical."""
    import torch
    from codenet_b200.engine_f32 import EngineF32
    from codenet_b200.synth import make_images
    cfg = CFG_1X if tag == "1x" else CFG_2X_COCO
    eng = EngineF32(cfg, _float_state(golden, tag, cfg), gemm=gemm)
    x = torch.from_numpy(make_images(7, 256, seed=9)).cuda()
    dets, inds, v = eng.detect(x)
    batch = {k: t.clone() for k, t in v.items()}
    dets, inds = dets.clone(), inds.clone()
    for i in range(7):
        d1, i1, v1 = eng.detect(x[i:i + 1].contiguous())
        for k in batch:
            assert torch.equal(v1[k], batch[k][i:i + 1]), (tag, gemm, i, k)
        assert torch.equal(d1, dets[i:i + 1]) and torch.equal(i1, inds[i:i + 1]), (tag, gemm, i)


def _count_forwards(monkeypatch):
    from codenet_b200.engine_f32 import EngineF32
    calls = []
    orig = EngineF32.forward

    def counted(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    monkeypatch.setattr(EngineF32, "forward", counted)
    return calls


def _assert_same(got, want, nc=20, tag=""):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert set(g) == {"results", "tot", "load", "pre", "net", "dec", "post", "merge"}
        for j in range(1, nc + 1):
            np.testing.assert_array_equal(g["results"][j], w[j], err_msg="%s frame %d class %d" % (tag, i, j))


@pytest.mark.parametrize("device_pre_process", [True, False])
@pytest.mark.parametrize("gemm", ["fp32", "tf32x3"])
@pytest.mark.parametrize("scales,max_batch", [([1.0], 3), ([0.5, 1.0, 1.5], 6)])
def test_float_run_batch_equals_run(golden, monkeypatch, scales, max_batch, gemm, device_pre_process):
    """11 mixed raw frames at 256^2, steps small enough that both staging buffers are reused: run_batch's results equal run()'s
    frame for frame, x flip, x nms, with ceil(frames / frames per step) EngineF32 forwards."""
    pytest.importorskip("cv2")
    det = _detector(golden, gemm=gemm, max_batch=max_batch, test_scales=scales, device_pre_process=device_pre_process)
    frames = _frames(76)
    for flip in (False, True):
        for nms in (False, True):
            det.opt.flip_test, det.opt.nms = flip, nms
            want = [det.run(f)["results"] for f in frames]
            calls = _count_forwards(monkeypatch)
            got = det.run_batch(frames)
            spf = len(scales) * (2 if flip else 1)
            per_step = max(max_batch, spf) // spf
            assert len(calls) == -(-len(frames) // per_step) and len(calls) >= 4
            monkeypatch.undo()
            _assert_same(got, want, tag="flip %s nms %s" % (flip, nms))
            again = det.run_batch(frames[3:5])                     # a later call on the same buffers, a partial step
            _assert_same(again, want[3:5], tag="second call")


def test_float_run_batch_host_merge_beyond_the_limit(golden, monkeypatch):
    """11 scales x K = 100 rows exceed the device merge's 1024: every frame is merged on the host, same results as run()."""
    pytest.importorskip("cv2")
    from codenet_b200.compat import detector as D
    det = _detector(golden, max_batch=11, test_scales=[0.5 + 0.1 * i for i in range(11)])
    frames = _frames(77, 3)
    want = [det.run(f)["results"] for f in frames]
    used = []
    orig = D.CtdetDetector.merge_outputs
    monkeypatch.setattr(D.CtdetDetector, "merge_outputs", lambda self, d: used.append(1) or orig(self, d))
    got = det.run_batch(frames)
    assert used == [1, 1, 1]
    _assert_same(got, want, tag="host merge")


def test_float_run_batch_paths_and_bytes_decode_on_the_host(golden, monkeypatch, tmp_path):
    """JPEG and PNG paths and encoded bytes give run()'s results for the decoded arrays; with 50 frames per step (above
    JPEG_DEVICE_MIN_FRAMES) the unquantised model still decodes every JPEG with cv2 and never calls cdn_jpeg_decode_batch."""
    cv2 = pytest.importorskip("cv2")
    from codenet_b200 import jpeg
    from codenet_b200.compat import detector as D
    n = 50
    assert n >= D.JPEG_DEVICE_MIN_FRAMES
    det = _detector(golden, max_batch=n, test_scales=[1.0])
    frames = _frames(78, n)
    blobs, paths = [], []
    for i, f in enumerate(frames):
        ok, buf = cv2.imencode(".png" if i % 7 == 3 else ".jpg", f)
        assert ok
        blobs.append(buf.tobytes())
        p = tmp_path / ("f%d%s" % (i, ".png" if i % 7 == 3 else ".jpg"))
        p.write_bytes(blobs[-1])
        paths.append(str(p))
    decoded = [cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR) for b in blobs]
    want = [det.run(d)["results"] for d in decoded]
    calls = []
    monkeypatch.setattr(jpeg, "decode_batch", lambda *a, **k: calls.append(1))
    fwd = _count_forwards(monkeypatch)
    _assert_same(det.run_batch(paths), want, tag="paths")
    _assert_same(det.run_batch([b if i % 2 else np.frombuffer(b, np.uint8) for i, b in enumerate(blobs)]), want, tag="bytes")
    _assert_same(det.run_batch(decoded), want, tag="arrays")
    assert calls == [] and len(fwd) == 3


def test_float_run_batch_2x_coco(golden):
    """BASELINE config 5's geometry (2x, 80 COCO classes) at 256^2, tf32x3, scale 1 with flip, 9 frames in steps of 4 slots."""
    pytest.importorskip("cv2")
    det = _detector(golden, tag="2x_coco", gemm="tf32x3", max_batch=4, test_scales=[1.0], flip_test=True)
    frames = _frames(79, 9)
    want = [det.run(f)["results"] for f in frames]
    _assert_same(det.run_batch(frames), want, nc=80, tag="2x coco")
