"""GPU box only: CtdetDetector.run_batch at five test scales (0.5, 0.75, 1, 1.25, 1.5) with flip, with and without nms, with the
resize on the device (cdn_warp_affine_resize_*) against the host cv2.resize path it replaces, and the resize kernel alone.

Seeded synthetic calibrated W4A8 CoDeNet1x (VOC, 20 classes) at 512x512 with bilinear offsets, and the seeded frames of
tools/bench_detect_frames.py (500x375 / 375x500 / 500x333 / 333x500 mix cut to even sizes).  Inputs: host BGR arrays, JPEG paths
(q90 files in a temporary directory), host I420 frames, CUDA BGR tensors, CUDA NV12 surfaces.  Per configuration and max_batch
(128, 256) and input kind: frames/s of run_batch over all frames, each path timed twice after an untimed pass, the device path
(opt.device_resize on) and the host path (off, the default: frames go through cv2.resize / to_bgr / .cpu() as before) alternating; the H2D frame bytes per frame from the shapes; whether the results equal run()'s
on the first --loop-frames frames.  JPEGs are decoded on the device only from JPEG_DEVICE_MIN_FRAMES (48) frames per step, which
at 10 slots per frame needs max_batch 480: one more row for JPEG paths at that size.  Then the warp alone, CUDA-event time over
--reps launches of 240 descriptors (48 frames x 5 scales) into 240 slots of 512x512 (destinations 189 MB, above the 126 MB L2):
today's kernel from host-resized copies in a pool and the resize kernel from the 1x frames (pool BGR, CUDA NV12).  The card's
name and power limit are read in the same run.  Writes detect_multiscale.json into --out-dir."""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import cv2  # noqa: E402
from bench_detect_batch import SHAPES, card, equal  # noqa: E402
from bench_detect_frames import inputs  # noqa: E402
from codenet_b200 import _lib, compat  # noqa: E402
from codenet_b200.arch import NetConfig  # noqa: E402
from codenet_b200.compat import detector as D  # noqa: E402
from codenet_b200.compat.detector import default_opt, plan_frame_steps, _pool_src_descs, _rs_descs  # noqa: E402
from codenet_b200.frames import to_bgr  # noqa: E402
from codenet_b200.synth import make_quant_state  # noqa: E402

FIVE = [0.5, 0.75, 1.0, 1.25, 1.5]
CONFIGS = (("5 scales + flip + nms", True), ("5 scales + flip", False))
BATCHES = (128, 256)
KINDS = ("host BGR", "JPEG paths", "host I420", "CUDA BGR", "CUDA NV12")
def h2d_frame_bytes(kind, frames, on, device_jpeg, file_bytes):
    """Frame bytes staged per frame, from the shapes: on the device-resize path (on) a host BGR or decoded JPEG frame once at 1x
    (3 bytes a pixel), an I420 frame at 1.5 bytes a pixel, CUDA frames nothing, a device-decoded JPEG its file; on the host path
    every scale's cv2.resize copy (3 bytes a pixel each)."""
    if kind == "JPEG paths" and on and device_jpeg:
        return file_bytes
    if on:
        per = {"host BGR": 3.0, "JPEG paths": 3.0, "host I420": 1.5}.get(kind, 0.0)
        return sum(f.shape[0] * f.shape[1] * per for f in frames) / len(frames)
    return sum(int(f.shape[0] * s) * int(f.shape[1] * s) * 3 for f in frames for s in FIVE) / len(frames)


def timed(det, xs):
    t0 = time.perf_counter()
    got = det.run_batch(xs)
    return len(xs) / (time.perf_counter() - t0), got


def compare(det, xs, want, nc):
    """Both paths, an untimed pass each, then device / host / device / host."""
    fps = {True: [], False: []}
    same = {}
    for on in (True, False):
        det.opt.device_resize = on
        det.run_batch(xs)
    torch.cuda.synchronize()
    for _ in range(2):
        for on in (True, False):
            det.opt.device_resize = on
            f, got = timed(det, xs)
            fps[on].append(round(f, 1))
            same[on] = "%d/%d" % (sum(equal(g["results"], w, nc) for g, w in zip(got, want)), len(want))
    return fps, same


def warp_alone(frames, nv12, reps):
    """240 descriptors (48 frames x 5 scales) into 240 slots of 512x512: today's warp from host-resized copies in a pool, and
    the resize kernel from the frames at 1x (pool BGR; CUDA NV12 surfaces).  u8 outputs must be equal."""
    det = compat.CtdetDetector.__new__(compat.CtdetDetector)
    det.opt = default_opt(test_scales=FIVE)
    det.scales = FIVE
    nf, S = 48, len(FIVE)
    layouts = [det._frame_layout(f.shape[0], f.shape[1], FIVE) for f in frames[:nf]]
    (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in L] for L in layouts], S, nf * S)
    pool = np.empty(nbytes, np.uint8)
    wdesc = np.empty(nf * S, _lib.WARP_DESC)
    for k in range(nf):
        det._pack_frame(frames[k], layouts[k], FIVE, pool, offsets[k], wdesc[k * S:(k + 1) * S], k * S)
    d_pool = torch.from_numpy(pool).cuda()
    (_, offs1, nbytes1), = plan_frame_steps([[f.size] for f in frames[:nf]], S, nf * S)
    pool1 = np.empty(nbytes1, np.uint8)
    w1 = np.empty(nf * S, _lib.WARP_DESC)
    for k in range(nf):
        pool1[offs1[k][0]:offs1[k][0] + frames[k].size] = frames[k].reshape(-1)
        det._frame_descs(w1[k * S:(k + 1) * S], offs1[k][0], frames[k].shape[:2], layouts[k], k * S)
    d_pool1 = torch.from_numpy(pool1).cuda()
    rs_hw = [(sh, sw) for L in layouts for sh, sw, _, _ in L]
    rs_pool = _rs_descs(_pool_src_descs(w1, d_pool1), rs_hw)
    s_nv12 = np.zeros(nf * S, _lib.WARP_SRC_DESC)
    for k in range(nf):
        det._frame_src_descs(nv12[k], layouts[k], None, None, None, s_nv12[k * S:(k + 1) * S], k * S)
    rs_nv12 = _rs_descs(s_nv12, rs_hw)
    dst = torch.empty((nf * S, 512, 512, 3), dtype=torch.uint8, device="cuda")
    runs = {"pool BGR, host-resized copies (cdn_warp_affine_u8_batch)": (lambda: det._warp(d_pool, wdesc, dst), pool.nbytes),
            "pool BGR at 1x (cdn_warp_affine_resize_u8_batch)": (lambda: det._warp_src(rs_pool, dst), pool1.nbytes),
            "CUDA NV12 at 1x (cdn_warp_affine_resize_u8_batch)": (lambda: det._warp_src(rs_nv12, dst),
                                                                  sum(f.y.numel() * 3 // 2 for f in nv12[:nf]))}
    out, ref = [], None
    for name, (fn, src_bytes) in runs.items():
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        row = {"source": name, "descriptors": nf * S, "ms_per_launch": round(ms, 4), "source_bytes": int(src_bytes),
               "destination_bytes": int(dst.numel()), "GB_per_s": round((src_bytes + dst.numel()) / ms / 1e6, 1)}
        if "NV12" not in name:
            now = dst.cpu().numpy()
            ref = now if ref is None else ref
            row["equal_to_host_resize_kernel"] = bool(np.array_equal(now, ref))
        out.append(row)
        print(json.dumps(row), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--loop-frames", type=int, default=64)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out-dir", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detect_multiscale needs a GPU")
    name, power = card()
    calib = np.load(os.path.join(ROOT, "tests", "golden", "codenet1x_calib.npz"))
    det = compat.CtdetDetector(default_opt(state_dict=make_quant_state(NetConfig(num_classes=20), calib, "bilinear", 512),
                                           test_scales=FIVE, flip_test=True))
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, SHAPES[int(rng.integers(0, 4))] + (3,), dtype=np.uint8) for _ in range(a.frames)]
    frames = [np.ascontiguousarray(f[:f.shape[0] & ~1, :f.shape[1] & ~1]) for f in frames]
    kinds_in = inputs(frames)
    tmp = tempfile.mkdtemp()
    try:
        paths, decoded, file_bytes = [], [], 0
        for i, f in enumerate(frames):
            ok, buf = cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])
            p = os.path.join(tmp, "%d.jpg" % i)
            with open(p, "wb") as fh:
                fh.write(buf.tobytes())
            paths.append(p)
            file_bytes += buf.size
            if i < a.loop_frames:
                decoded.append(cv2.imdecode(buf, cv2.IMREAD_COLOR))
        kinds_in["JPEG paths"] = paths
        jpeg_mean = file_bytes / len(paths)
        shared = a.loop_frames
        report = {"card": name, "power_limit": power, "model": "synthetic W4A8 CoDeNet1x, 20 classes, 512x512, offsets bilinear",
                  "test_scales": FIVE, "flip_test": True, "frames": a.frames,
                  "frame_mix": sorted({"%dx%d" % (f.shape[1], f.shape[0]) for f in frames}),
                  "timing": "frames/s of one run_batch call over all frames, two timed calls per path, device and host path "
                            "alternating after an untimed call of each", "configs": []}
        for tag, nms in CONFIGS:
            det.opt.nms = nms
            det.opt.max_batch = 1
            want = {"bgr": [det.run(f)["results"] for f in frames[:shared]],
                    "yuv": [det.run(to_bgr(f))["results"] for f in kinds_in["host I420"][:shared]],
                    "jpeg": [det.run(f)["results"] for f in decoded]}
            line = {"config": tag, "run_batch": []}
            runs = [(mb, kind) for mb in BATCHES for kind in KINDS] + [(480, "JPEG paths")]
            for mb, kind in runs:
                det.opt.max_batch = mb
                w = want["yuv"] if "I420" in kind or "NV12" in kind else want["jpeg"] if "JPEG" in kind else want["bgr"]
                fps, same = compare(det, kinds_in[kind], w, det.num_classes)
                device_jpeg = max(mb, 10) // 10 >= D.JPEG_DEVICE_MIN_FRAMES
                row = {"max_batch": mb, "input": kind,
                       "frames_per_s_device_resize": fps[True], "frames_per_s_host_resize": fps[False],
                       "speedup": round(np.mean(fps[True]) / np.mean(fps[False]), 2),
                       "h2d_frame_bytes_per_frame_device_resize": round(h2d_frame_bytes(kind, frames, True, device_jpeg, jpeg_mean)),
                       "h2d_frame_bytes_per_frame_host_resize": round(h2d_frame_bytes(kind, frames, False, False, jpeg_mean)),
                       "equal_to_run_device_resize": same[True], "equal_to_run_host_resize": same[False]}
                print(json.dumps(dict(row, config=tag)), flush=True)
                line["run_batch"].append(row)
            report["configs"].append(line)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    del det
    report["warp_kernel"] = warp_alone(frames, kinds_in["CUDA NV12"], a.reps)
    report["warp_kernel_note"] = ("240 descriptors (48 frames x 5 scales) into 240 slots of 512x512x3, no mirror; bytes moved = "
                                  "sources + destinations")
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "detect_multiscale.json"), "w") as f:
            json.dump(report, f, indent=1)
    full = "%d/%d" % (shared, shared)
    bad = [r for c in report["configs"] for r in c["run_batch"]
           if r["equal_to_run_device_resize"] != full or r["equal_to_run_host_resize"] != full]
    if bad or not all(w.get("equal_to_host_resize_kernel", True) for w in report["warp_kernel"]):
        raise SystemExit("run_batch and run() differ: %s" % bad)


if __name__ == "__main__":
    main()
