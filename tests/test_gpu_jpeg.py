"""Baseline JPEG decoding on the device (cdn_jpeg_decode_batch through codenet_b200.jpeg.decode_jpeg) against cv2.imdecode,
element for element, and CtdetDetector.run_batch from JPEG paths and encoded bytes against run() frame for frame."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from codenet_b200 import jpeg

pytestmark = pytest.mark.gpu

SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420}


def _image(h, w, rng, noisy):
    if noisy:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[:h, :w].astype(np.float64)
    a, b, c = rng.uniform(0.01, 0.08, 3)
    img = np.stack([128 + 100 * np.sin(a * x + b * y), 128 + 90 * np.cos(b * x - c * y), 128 + 110 * np.sin(c * (x + y))], -1)
    return np.clip(img, 0, 255).astype(np.uint8)


def _encode(img, q=75, sampling="420", **kw):
    params = [cv2.IMWRITE_JPEG_QUALITY, q]
    if img.ndim == 3:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    for k, v in kw.items():
        params += [getattr(cv2, "IMWRITE_JPEG_" + k.upper()), v]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return buf.tobytes()


def _corpus(seed):
    rng = np.random.default_rng(seed)
    sizes = [(1, 1), (5, 7), (9, 17), (375, 500), (500, 333), (480, 640), (1080, 1920), (3, 4), (16, 16), (31, 33)]
    out = []
    for i, (h, w) in enumerate(sizes):
        for s in ("444", "422", "420", "gray"):
            q = [10, 30, 50, 75, 90, 95, 100][(i + len(out)) % 7]
            kw = [{}, {"optimize": 1}, {"rst_interval": 1}, {"rst_interval": 7}][(i + len(out)) % 4]
            img = _image(h, w, rng, noisy=(i + len(out)) % 2 == 0)
            out.append(((h, w, s, q, kw), _encode(img[..., 0] if s == "gray" else img, q, "420" if s == "gray" else s, **kw)))
    return out


def _want(buf):
    return cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR)


def test_decode_jpeg_equals_cv2_over_a_seeded_corpus():
    """Sizes 1x1 to 1920x1080, every accepted sampling, q10-q100, optimized tables, restart intervals 1 and 7, smooth and noisy
    content: all decoded on the device in one call, each bit-identical to cv2.imdecode."""
    corpus = _corpus(1)
    got, status = jpeg.decode_jpeg([b for _, b in corpus], return_status=True)
    for (tag, buf), g, (rc, ds) in zip(corpus, got, status):
        assert rc == 0 and ds == 0, (tag, rc, ds)
        np.testing.assert_array_equal(g.cpu().numpy(), _want(buf), err_msg=str(tag))


def test_decode_jpeg_many_frames_mixed_with_refused_ones():
    rng = np.random.default_rng(2)
    bufs, kinds = [], []
    for i in range(300):
        h, w = int(rng.integers(1, 90)), int(rng.integers(1, 90))
        img = _image(h, w, rng, noisy=i % 3 == 0)
        k = i % 6
        if k == 4:
            bufs.append(_encode(img, progressive=1))                  # host: progressive
        elif k == 5:
            bufs.append(cv2.imencode(".png", img)[1].tobytes())      # host: not a JPEG
        else:
            bufs.append(_encode(img, int(rng.integers(10, 101)), ("444", "422", "420", "420")[k], rst_interval=int(rng.integers(0, 4))))
        kinds.append(k)
    got, status = jpeg.decode_jpeg(bufs, return_status=True)
    for i, (buf, g, (rc, ds)) in enumerate(zip(bufs, got, status)):
        assert (rc == 0) == (kinds[i] < 4), (i, rc)
        if rc == 0:
            assert ds == 0, (i, ds)
        np.testing.assert_array_equal(g.cpu().numpy(), _want(buf), err_msg=str(i))


def test_decode_jpeg_flipped_scan_bytes_are_flagged_or_equal_cv2():
    """Corrupt entropy-coded data: every frame the device does not flag equals cv2; decode_jpeg's result (host decode for the
    flagged ones) always equals cv2."""
    rng = np.random.default_rng(3)
    bufs = []
    for i in range(240):
        img = _image(int(rng.integers(8, 120)), int(rng.integers(8, 120)), rng, noisy=i % 2 == 0)
        b = bytearray(_encode(img, int(rng.choice([10, 50, 90])), ("444", "422", "420")[i % 3],
                              rst_interval=int(rng.choice([0, 0, 1, 3]))))
        scan = jpeg.parse(bytes(b))[1][0]["scan_offset"]
        for _ in range(int(rng.integers(1, 4))):
            p = int(rng.integers(scan, len(b) - 2))
            b[p] ^= 1 << int(rng.integers(0, 8))
        bufs.append(bytes(b))
    got, status = jpeg.decode_jpeg(bufs, return_status=True)
    flagged = 0
    for buf, g, (rc, ds) in zip(bufs, got, status):
        want = _want(buf)
        if want is None:
            continue
        flagged += ds is not None and ds != 0
        np.testing.assert_array_equal(g.cpu().numpy(), want)
    assert flagged > 0


def test_decode_jpeg_rejects_what_neither_decoder_reads():
    with pytest.raises(ValueError):
        jpeg.decode_jpeg([b"not an image"])
    with pytest.raises(ValueError):
        jpeg.decode_jpeg([np.zeros((4, 4), np.uint8)])


# ---- CtdetDetector.run_batch from JPEG files and bytes ------------------------------------------------------------------
def _detector(calib, res, **kw):
    from codenet_b200 import compat
    from codenet_b200.arch import NetConfig
    from codenet_b200.compat.detector import default_opt
    from codenet_b200.synth import make_quant_state
    st = make_quant_state(NetConfig(num_classes=20), calib, "round", res)
    return compat.CtdetDetector(default_opt(state_dict=st, offset_mode="round", input_h=res, input_w=res, **kw))


def _count_engine_runs(monkeypatch):
    from codenet_b200.engine import Engine
    calls = []
    orig = Engine.run

    def counted(self, *a, **k):
        calls.append(1)
        return orig(self, *a, **k)
    monkeypatch.setattr(Engine, "run", counted)
    return calls


def _device_decode_from(monkeypatch, frames_per_step):
    """Lowers the frames per step from which run_batch decodes JPEGs on the device (the tests' steps are small) and counts
    the cdn_jpeg_decode_batch calls."""
    from codenet_b200.compat import detector as D
    monkeypatch.setattr(D, "JPEG_DEVICE_MIN_FRAMES", frames_per_step)
    calls = []
    orig = jpeg.decode_batch

    def counted(*a, **k):
        calls.append(1)
        return orig(*a, **k)
    monkeypatch.setattr(jpeg, "decode_batch", counted)
    return calls


def _assert_same(got, want, tag=""):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert set(g) == {"results", "tot", "load", "pre", "net", "dec", "post", "merge"}
        for j in range(1, 21):
            np.testing.assert_array_equal(g["results"][j], w[j], err_msg="%s frame %d class %d" % (tag, i, j))


def _files(tmp_path, seed, n=9):
    """VOC-sized JPEG files (4:2:0 q75 / q95, one 4:4:4 with restart markers, one gray) plus a progressive JPEG and a PNG
    that the host decodes."""
    rng = np.random.default_rng(seed)
    shapes = [(375, 500), (500, 333), (256, 256), (97, 203), (480, 640), (333, 500), (40, 31), (300, 400), (600, 700)]
    paths = []
    for i in range(n):
        img = _image(*shapes[i % len(shapes)], rng, noisy=i % 3 == 2)
        if i % 9 == 6:
            buf = _encode(img, 90, "444", rst_interval=5)
        elif i % 9 == 7:
            buf = _encode(img[..., 0], 80)
        elif i % 9 == 8:
            buf = _encode(img, 75, progressive=1)
        else:
            buf = _encode(img, (75, 95)[i % 2])
        p = tmp_path / ("f%d.jpg" % i)
        p.write_bytes(buf)
        paths.append(str(p))
    png = tmp_path / "g.png"
    assert cv2.imwrite(str(png), _image(123, 77, rng, True))
    return paths[:4] + [str(png)] + paths[4:]


def test_run_batch_jpeg_paths_and_bytes_equal_run(calib, monkeypatch, tmp_path):
    """Scale 1 with and without flip: JPEG paths and bytes decoded on the device give run(path)'s results frame for frame, with
    ceil(frames / frames per step) engine calls."""
    det = _detector(calib, 256, max_batch=4, test_scales=[1.0])
    paths = _files(tmp_path, 80)
    blobs = [open(p, "rb").read() for p in paths]
    decodes = _device_decode_from(monkeypatch, 1)
    for flip in (False, True):
        det.opt.flip_test = flip
        want = [det.run(p)["results"] for p in paths]
        per_step = 4 // (2 if flip else 1)
        del decodes[:]
        with monkeypatch.context() as m:
            calls = _count_engine_runs(m)
            got = det.run_batch(paths)
        assert len(calls) == -(-len(paths) // per_step) and len(decodes) == len(calls)
        _assert_same(got, want, tag="paths flip %s" % flip)
        mixed = [blobs[0], bytearray(blobs[1]), memoryview(blobs[2]), np.frombuffer(blobs[3], np.uint8)] + paths[4:]
        _assert_same(det.run_batch(mixed), want, tag="bytes flip %s" % flip)
    det.opt.flip_test = False


def test_run_batch_jpeg_five_scales_flip_nms_decode_on_the_host(calib, monkeypatch, tmp_path):
    det = _detector(calib, 256, max_batch=10, test_scales=[0.5, 0.75, 1.0, 1.25, 1.5], flip_test=True, nms=True)
    from codenet_b200 import jpeg as J
    parsed = []
    monkeypatch.setattr(J, "parse", lambda *a, **k: parsed.append(1))       # never consulted at scales other than 1
    paths = _files(tmp_path, 81, 5)
    want = [det.run(p)["results"] for p in paths]
    _assert_same(det.run_batch(paths), want, tag="five scales")
    assert not parsed


def test_run_batch_jpeg_more_frames_than_one_step(calib, monkeypatch, tmp_path):
    """Small frames first, then larger ones: both staging buffers, their device pools and the decode workspace grow during
    the call; a second call reuses them."""
    decodes = _device_decode_from(monkeypatch, 3)
    det = _detector(calib, 256, max_batch=3, test_scales=[1.0])
    rng = np.random.default_rng(82)
    paths = []
    for i, (h, w) in enumerate([(20, 30)] * 4 + [(375, 500), (500, 375), (720, 1280), (1080, 1920)] * 3):
        p = tmp_path / ("s%d.jpg" % i)
        p.write_bytes(_encode(_image(h, w, rng, noisy=i % 2 == 0), 85, ("420", "422")[i % 2]))
        paths.append(str(p))
    want = [det.run(p)["results"] for p in paths]
    _assert_same(det.run_batch(paths), want, tag="growth")
    _assert_same(det.run_batch(paths[::-1]), want[::-1], tag="again")
    assert len(decodes) == 2 * 6


def test_run_batch_jpeg_small_steps_decode_on_the_host(calib, monkeypatch, tmp_path):
    """Below JPEG_DEVICE_MIN_FRAMES frames per step the host decode is the faster one: no device decode call, same results."""
    decodes = _device_decode_from(monkeypatch, 48)
    det = _detector(calib, 256, max_batch=32, test_scales=[1.0], flip_test=True)
    paths = _files(tmp_path, 84, 5)
    want = [det.run(p)["results"] for p in paths]
    _assert_same(det.run_batch(paths), want, tag="host decode")
    assert not decodes


def test_run_batch_jpeg_corrupt_file_is_rerun_from_the_host_decode(calib, monkeypatch, tmp_path):
    """A stream cut short inside its scan: the device flags it, cv2 decodes what it can (gray fill), run() gives the results."""
    decodes = _device_decode_from(monkeypatch, 1)
    det = _detector(calib, 256, max_batch=4, test_scales=[1.0])
    paths = _files(tmp_path, 83, 6)
    good = open(paths[1], "rb").read()
    scan = int(_scan_offset(good))
    cut = tmp_path / "cut.jpg"
    cut.write_bytes(good[:scan + (len(good) - scan) // 3] + b"\xff\xd9")
    paths.insert(2, str(cut))
    assert cv2.imread(str(cut)) is not None
    want = [det.run(p)["results"] for p in paths]
    with monkeypatch.context() as m:
        calls = _count_engine_runs(m)
        got = det.run_batch(paths)
    assert len(calls) == -(-len(paths) // 4) + 1 and len(decodes) == len(calls) - 1   # the steps + one run() of the flagged frame
    _assert_same(got, want, tag="corrupt")
    with pytest.raises(ValueError, match="cannot read"):
        det.run_batch([paths[0], b"\xff\xd8\xff\xd9 not a jpeg"])


def _scan_offset(buf):
    rc, d = jpeg.parse(buf)
    assert rc == 0
    return d[0]["scan_offset"]
