"""GPU box only: baseline JPEG decoding on the device (cdn_jpeg_decode_batch) against cv2.imdecode on the host, and
CtdetDetector.run_batch from JPEG paths (device decode) against the host cv2.imread path and against pre-decoded arrays.

Seeded 500x375-class mix (500x375, 375x500, 500x333, 333x500) of smooth content with mild noise, written as 4:2:0 JPEG files
at q75 and q95 (--frames each).  Reports, with the card's name and power limit read in the same run:
  * decode time per kernel (torch.profiler, a separate pass) and frames/s of one cdn_jpeg_decode_batch call at 32, 128, 256
    and 1024 frames per call (CUDA events; successive calls decode disjoint frames with disjoint workspaces and outputs, a
    rotating working set of all frames, above the 126 MB L2);
  * the same frames through one-thread cv2.imdecode and a cv2.imdecode thread pool over every host core;
  * run_batch frames/s from paths as the detector chooses (device decode from JPEG_DEVICE_MIN_FRAMES frames per step, host
    decode below: max_batch 32 is on the host side of that choice, 128 and 256 on the device side), from paths with the device
    decode forced at every step size, over cv2.imread'd frames (the host decode path) and over pre-decoded arrays, at max_batch 32, 128 and 256, scale 1 with and without flip,
    512x512 synthetic W4A8 model;
  * host-to-device bytes per frame, compressed (stream + descriptor) against raw;
  * whether run_batch's results from paths equal run()'s on the first --check frames.
Writes jpeg_decode.json into --out-dir."""
import argparse
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from codenet_b200 import compat, jpeg  # noqa: E402
from codenet_b200.arch import NetConfig  # noqa: E402
from codenet_b200.compat.detector import JPEG_DEVICE_MIN_FRAMES, default_opt  # noqa: E402
from codenet_b200.synth import make_quant_state  # noqa: E402
from tools.bench_detect_batch import SHAPES, card, equal  # noqa: E402

CALLS = (32, 128, 256, 1024)
BATCHES = (32, 128, 256)
KERNELS = ("jpeg_restart_index_kernel", "jpeg_entropy_kernel", "jpeg_idct_kernel", "jpeg_color_kernel")


def make_files(d, n, q, seed):
    rng = np.random.default_rng(seed)
    paths = []
    for i in range(n):
        h, w = SHAPES[int(rng.integers(0, 4))]
        y, x = np.mgrid[:h, :w].astype(np.float32)
        a = rng.uniform(0.005, 0.05, 6)
        img = np.stack([128 + 90 * np.sin(a[0] * x + a[1] * y), 128 + 80 * np.cos(a[2] * x - a[3] * y),
                        128 + 100 * np.sin(a[4] * (x + y)) * np.cos(a[5] * x)], -1)
        img += rng.normal(0, 10, img.shape)
        ok, buf = cv2.imencode(".jpg", np.clip(img, 0, 255).astype(np.uint8),
                               [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420])
        p = os.path.join(d, "q%d_%04d.jpg" % (q, i))
        with open(p, "wb") as f:
            f.write(buf.tobytes())
        paths.append(p)
    return paths


class DeviceBatch:
    """All frames' streams and descriptors on the device once; call k of size b decodes frames [k*b, (k+1)*b) into their own
    workspace and output ranges."""

    def __init__(self, blobs):
        self.desc = np.zeros(len(blobs), jpeg.JPEG_FRAME)
        for i, b in enumerate(blobs):
            assert jpeg.parse(b, self.desc[i:i + 1])[0] == 0
        head = -(-self.desc.nbytes // jpeg.WS_ALIGN) * jpeg.WS_ALIGN
        offs, end, out_end, ws = jpeg.layout(self.desc, head, [len(b) for b in blobs], 0)
        host = np.zeros(end, np.uint8)
        for o, b in zip(offs, blobs):
            host[o:o + len(b)] = np.frombuffer(b, np.uint8)
        host[:self.desc.nbytes] = self.desc.view(np.uint8)
        self.pool = torch.from_numpy(host).cuda()
        self.ws = torch.empty(ws, dtype=torch.uint8, device="cuda")
        self.out = torch.empty(out_end, dtype=torch.uint8, device="cuda")
        self.status = torch.empty(len(blobs), dtype=torch.int32, device="cuda")
        self.working_set = int(end + ws + out_end)

    def call(self, k, b):
        lo = k * b
        d = self.desc[lo:lo + b]
        jpeg.decode_batch(self.pool.data_ptr(), self.pool.numel(), d, self.pool.data_ptr() + lo * jpeg.JPEG_FRAME.itemsize,
                          self.ws.data_ptr(), self.ws.numel(), self.out.data_ptr(), self.out.numel(), self.status[lo:].data_ptr(),
                          torch.cuda.current_stream().cuda_stream)


def device_decode(blobs, reps):
    dbat = DeviceBatch(blobs)
    n = len(blobs)
    rows = []
    for b in CALLS:
        if b > n:
            continue
        k_calls = n // b
        for k in range(k_calls):
            dbat.call(k, b)
        torch.cuda.synchronize()
        assert int(dbat.status.abs().sum()) == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        calls = max(reps, k_calls)
        e0.record()
        for c in range(calls):
            dbat.call(c % k_calls, b)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / calls
        rows.append({"frames_per_call": b, "ms_per_call": round(ms, 3), "frames_per_s": round(b / ms * 1e3, 1)})
    # per kernel, in a profiled pass of its own
    from torch.profiler import ProfilerActivity, profile
    per = {}
    for b in CALLS:
        if b > n:
            continue
        k_calls = n // b
        calls = max(reps, k_calls)                       # the same call sequence as the timed loop
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            for c in range(calls):
                dbat.call(c % k_calls, b)
            torch.cuda.synchronize()
        ev = {e.key: e for e in prof.key_averages()}
        row = {}
        for k in KERNELS:
            hit = [e for key, e in ev.items() if k in key]
            # a kernel the profiler did not report (the restart index runs only for frames with restart markers) is null
            row[k] = round(sum(e.device_time_total for e in hit) / 1e3 / calls, 4) if hit else None
        per[str(b)] = row
    # results equal cv2
    same = 0
    outs = dbat.out.cpu().numpy()
    for i, b in enumerate(blobs):
        h, w, o = int(dbat.desc[i]["height"]), int(dbat.desc[i]["width"]), int(dbat.desc[i]["out_offset"])
        same += np.array_equal(outs[o:o + h * w * 3].reshape(h, w, 3), cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR))
    return {"calls": rows, "ms_per_call_per_kernel": per, "working_set_bytes": dbat.working_set,
            "equal_to_cv2": "%d/%d" % (same, n)}


def host_decode(blobs):
    arr = [np.frombuffer(b, np.uint8) for b in blobs]
    cv2.setNumThreads(1)
    t0 = time.perf_counter()
    for a in arr:
        cv2.imdecode(a, cv2.IMREAD_COLOR)
    one = len(arr) / (time.perf_counter() - t0)
    cores = os.cpu_count() or 1
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(lambda a: cv2.imdecode(a, cv2.IMREAD_COLOR), arr[:cores]))
        t0 = time.perf_counter()
        list(ex.map(lambda a: cv2.imdecode(a, cv2.IMREAD_COLOR), arr))
        pool = len(arr) / (time.perf_counter() - t0)
    return {"one_thread_frames_per_s": round(one, 1), "pool_threads": cores, "pool_frames_per_s": round(pool, 1)}


def forced_device(det, paths):
    """run_batch(paths) with the device decode at every step size (both sides of JPEG_DEVICE_MIN_FRAMES)."""
    from codenet_b200.compat import detector as D
    keep, D.JPEG_DEVICE_MIN_FRAMES = D.JPEG_DEVICE_MIN_FRAMES, 1
    try:
        return det.run_batch(paths)
    finally:
        D.JPEG_DEVICE_MIN_FRAMES = keep


def detector_rows(det, paths, check):
    rows = []
    nc = det.num_classes
    for flip in (False, True):
        det.opt.flip_test = flip
        det.opt.max_batch = 1
        want = [det.run(p)["results"] for p in paths[:check]]
        line = {"config": "scale 1" + (", flip" if flip else ""), "run_batch": []}
        for mb in BATCHES:
            det.opt.max_batch = mb
            arrays = [cv2.imread(p) for p in paths]
            timed, same = {}, {}
            for tag, fn in (("paths", lambda: det.run_batch(paths)),
                            ("paths_device_decode", lambda: forced_device(det, paths)),
                            ("host_imread_then_arrays", lambda: det.run_batch([cv2.imread(p) for p in paths])),
                            ("predecoded_arrays", lambda: det.run_batch(arrays))):
                fn()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                got = fn()
                timed[tag] = round(len(paths) / (time.perf_counter() - t0), 1)
                if tag.startswith("paths"):
                    same[tag] = "%d/%d" % (sum(equal(g["results"], w, nc) for g, w in zip(got, want)), check)
            spf = 2 if flip else 1
            decoder = "device" if min(mb // spf, len(paths)) >= JPEG_DEVICE_MIN_FRAMES else "host"
            line["run_batch"].append({"max_batch": mb, "frames_per_step": mb // spf, "paths_decoded_on": decoder,
                                      "frames_per_s": timed, "equal_to_run": same})
        rows.append(line)
        print(json.dumps(line), flush=True)
    det.opt.flip_test = False
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--check", type=int, default=64)
    ap.add_argument("--out-dir", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg needs a GPU")
    name, power = card()
    report = {"card": name, "power_limit": power, "frames": a.frames, "frame_mix": ["%dx%d" % (w, h) for h, w in SHAPES],
              "content": "smooth sinusoids + N(0, 10) noise, 4:2:0", "qualities": {}}
    st = make_quant_state(NetConfig(num_classes=20), np.load(os.path.join(ROOT, "tests", "golden", "codenet1x_calib.npz")),
                          "bilinear", 512)
    det = compat.CtdetDetector(default_opt(state_dict=st, offset_mode="bilinear"))
    with tempfile.TemporaryDirectory() as d:
        for q in (75, 95):
            paths = make_files(d, a.frames, q, q)
            blobs = [open(p, "rb").read() for p in paths]
            raw = float(np.mean([int(h) * int(w) * 3 for h, w in (cv2.imread(p).shape[:2] for p in paths[:64])]))
            r = {"mean_file_bytes": round(float(np.mean([len(b) for b in blobs])), 1),
                 "h2d_bytes_per_frame": {"compressed_stream_plus_descriptor": round(float(np.mean([len(b) for b in blobs])) +
                                                                                    jpeg.JPEG_FRAME.itemsize),
                                         "raw_frame": round(raw)}}
            r["device_decode"] = device_decode(blobs, a.reps)
            print(json.dumps({"q": q, "device": r["device_decode"]}), flush=True)
            r["host_decode"] = host_decode(blobs)
            print(json.dumps({"q": q, "host": r["host_decode"]}), flush=True)
            r["run_batch_512"] = detector_rows(det, paths, a.check)
            report["qualities"]["q%d" % q] = r
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "jpeg_decode.json"), "w") as f:
            json.dump(report, f, indent=1)
    full = "%d/%d" % (a.check, a.check)
    bad = [q for q, r in report["qualities"].items()
           if r["device_decode"]["equal_to_cv2"] != "%d/%d" % (a.frames, a.frames) or
           any(v != full for c in r["run_batch_512"] for x in c["run_batch"] for v in x["equal_to_run"].values())]
    if bad:
        raise SystemExit("device decode differs from cv2 / run() at %s" % bad)


if __name__ == "__main__":
    main()
