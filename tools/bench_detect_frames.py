"""GPU box only: CtdetDetector.run_batch from each input kind (host BGR arrays, host I420 frames, CUDA BGR tensors, CUDA NV12
surfaces) and the warp kernels alone per source kind.

Seeded synthetic calibrated W4A8 CoDeNet1x (VOC, 20 classes) at 512x512 with bilinear offsets, and the 1024 seeded frames of
tools/bench_detect_batch.py (same seed, same 500x375 / 375x500 / 500x333 / 333x500 mix) cut to even sizes (374x500, ...)
because 4:2:0 needs an even height and width.  The YUV frames are cv2.cvtColor(frame, COLOR_BGR2YUV_I420) of the same frames
(an NV12 surface per frame for the CUDA kind).  Per configuration (scale 1; scale 1 + flip) and max_batch (128, 256): frames/s of
run_batch over all frames from each kind (timed after one untimed pass), the H2D frame bytes per frame computed from the shapes
(BGR 3 bytes a pixel, I420 1.5, CUDA frames 0), and whether the results equal run()'s on the first --loop-frames frames (run() of
the BGR frame for BGR kinds, of to_bgr(frame) for YUV kinds).  One more row: CoDeNet2x COCO float (tf32x3, synthetic weights with
the golden BatchNorm statistics) at scale 1, max_batch 256.  Then each warp kernel alone: CUDA-event time over --reps launches of
256 descriptors into 256 slots of 512x512 (sources + destinations about 350 MB, above the 126 MB L2).  The card's name and power
limit are read in the same run.  Writes detect_frames.json into --out-dir."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import cv2  # noqa: E402
from bench_detect_batch import SHAPES, card, equal  # noqa: E402
from codenet_b200 import _lib, compat  # noqa: E402
from codenet_b200.arch import NetConfig  # noqa: E402
from codenet_b200.compat.detector import default_opt, plan_frame_steps  # noqa: E402
from codenet_b200.frames import YUV420, to_bgr  # noqa: E402
from codenet_b200.synth import make_quant_state, make_raw_state  # noqa: E402

CONFIGS = (("scale 1", False), ("scale 1, flip", True))
BATCHES = (128, 256)
KINDS = ("host BGR", "host I420", "CUDA BGR", "CUDA NV12")


def i420_planes(buf):
    H, W = buf.shape[0] * 2 // 3, buf.shape[1]
    flat = buf.reshape(-1)
    return buf[:H], flat[H * W:H * W * 5 // 4].reshape(H // 2, W // 2), flat[H * W * 5 // 4:].reshape(H // 2, W // 2)


def nv12_surface(buf):
    y, u, v = i420_planes(buf)
    return np.concatenate([y.reshape(-1), np.stack([u, v], -1).reshape(-1)]).reshape(buf.shape)


def inputs(frames):
    """kind -> the run_batch inputs of every frame."""
    i420 = [cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in frames]
    surfaces = [torch.from_numpy(nv12_surface(b)).cuda() for b in i420]
    H = lambda s: s.shape[0] * 2 // 3
    return {"host BGR": frames,
            "host I420": [YUV420(*i420_planes(b)) for b in i420],
            "CUDA BGR": [torch.from_numpy(f).cuda() for f in frames],
            "CUDA NV12": [YUV420(s[:H(s)], s[H(s):, 0::2], s[H(s):, 1::2]) for s in surfaces]}


def h2d_frame_bytes(kind, frames):
    per = {"host BGR": 3.0, "host I420": 1.5}.get(kind, 0.0)
    return sum(f.shape[0] * f.shape[1] * per for f in frames) / len(frames)


def time_run_batch(det, xs, shared_want, nc):
    det.run_batch(xs)                                        # engine build, graph capture, staging growth
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = det.run_batch(xs)
    dt = time.perf_counter() - t0
    same = sum(equal(g["results"], w, nc) for g, w in zip(got, shared_want))
    return round(len(xs) / dt, 1), "%d/%d" % (same, len(shared_want))


def warp_alone(frames, kinds_in, reps):
    """Each kernel writing 256 slots of 512x512 from 256 frames: today's pool kernel, and the general-source kernel from the pool
    (BGR), from CUDA BGR tensors, from I420 planes in a pool and from CUDA NV12 surfaces."""
    det = compat.CtdetDetector.__new__(compat.CtdetDetector)
    det.opt = default_opt()
    det.scales = [1.0]
    n = 256
    layouts = [det._frame_layout(f.shape[0], f.shape[1], [1.0]) for f in frames[:n]]
    (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in L] for L in layouts], 1, n)
    pool = np.empty(nbytes, np.uint8)
    wdesc = np.empty(n, _lib.WARP_DESC)
    for k in range(n):
        det._pack_frame(frames[k], layouts[k], [1.0], pool, offsets[k], wdesc[k:k + 1], k)
    d_pool = torch.from_numpy(pool).cuda()
    from codenet_b200.compat.detector import _pool_src_descs
    # the I420 planes of the same frames, back to back in a second pool
    ys = [kinds_in["host I420"][k] for k in range(n)]
    (_, yoffs, ybytes), = plan_frame_steps([[p.size for p in (f.y, f.u, f.v)] for f in ys], 1, n)
    ypool = np.empty(ybytes, np.uint8)
    d_ypool = torch.empty(ybytes, dtype=torch.uint8, device="cuda")
    src = {"pool BGR (general kernel)": _pool_src_descs(wdesc, d_pool),
           "CUDA BGR": np.zeros(n, _lib.WARP_SRC_DESC), "pool I420": np.zeros(n, _lib.WARP_SRC_DESC),
           "CUDA NV12": np.zeros(n, _lib.WARP_SRC_DESC)}
    for k in range(n):
        det._frame_src_descs(kinds_in["CUDA BGR"][k], layouts[k], None, None, None, src["CUDA BGR"][k:k + 1], k)
        det._frame_src_descs(ys[k], layouts[k], ypool, d_ypool, yoffs[k], src["pool I420"][k:k + 1], k)
        det._frame_src_descs(kinds_in["CUDA NV12"][k], layouts[k], None, None, None, src["CUDA NV12"][k:k + 1], k)
    d_ypool.copy_(torch.from_numpy(ypool))
    dst = torch.empty((n, 512, 512, 3), dtype=torch.uint8, device="cuda")
    runs = {"pool BGR (cdn_warp_affine_u8_batch)": lambda: det._warp(d_pool, wdesc, dst)}
    for name, d in src.items():
        runs[name] = lambda d=d: det._warp_src(d, dst)
    src_bytes = {"pool BGR (cdn_warp_affine_u8_batch)": pool.nbytes, "pool BGR (general kernel)": pool.nbytes,
                 "CUDA BGR": pool.nbytes, "pool I420": ybytes, "CUDA NV12": ybytes}
    out, ref = [], None
    for name, fn in runs.items():
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        moved = src_bytes[name] + dst.numel()
        row = {"source": name, "descriptors": n, "launches_timed": reps, "ms_per_launch": round(ms, 4),
               "source_bytes": int(src_bytes[name]), "destination_bytes": int(dst.numel()), "GB_per_s": round(moved / ms / 1e6, 1)}
        # BGR kinds must write what today's kernel writes
        if "I420" not in name and "NV12" not in name:
            now = dst.cpu().numpy()
            ref = now if ref is None else ref
            row["equal_to_pool_kernel"] = bool(np.array_equal(now, ref))
        out.append(row)
        print(json.dumps(row), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--loop-frames", type=int, default=128)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--out-dir", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detect_frames needs a GPU")
    name, power = card()
    calib = np.load(os.path.join(ROOT, "tests", "golden", "codenet1x_calib.npz"))
    det = compat.CtdetDetector(default_opt(state_dict=make_quant_state(NetConfig(num_classes=20), calib, "bilinear", 512)))
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, SHAPES[int(rng.integers(0, 4))] + (3,), dtype=np.uint8) for _ in range(a.frames)]
    frames = [np.ascontiguousarray(f[:f.shape[0] & ~1, :f.shape[1] & ~1]) for f in frames]
    kinds_in = inputs(frames)
    shared = a.loop_frames
    report = {"card": name, "power_limit": power, "model": "synthetic W4A8 CoDeNet1x, 20 classes, 512x512, offsets bilinear",
              "frames": a.frames, "frame_mix": sorted({"%dx%d" % (f.shape[1], f.shape[0]) for f in frames}),
              "h2d_frame_bytes_per_500x375_frame": {"BGR": 500 * 375 * 3, "I420": 500 * 375 * 3 // 2, "CUDA": 0},
              "configs": []}
    for tag, flip in CONFIGS:
        det.opt.flip_test = flip
        det.opt.max_batch = 1
        want_bgr = [det.run(f)["results"] for f in frames[:shared]]
        want_yuv = [det.run(to_bgr(f))["results"] for f in kinds_in["host I420"][:shared]]
        line = {"config": tag, "run_batch": []}
        for mb in BATCHES:
            det.opt.max_batch = mb
            for kind in KINDS:
                want = want_yuv if "I420" in kind or "NV12" in kind else want_bgr
                fps, same = time_run_batch(det, kinds_in[kind], want, det.num_classes)
                row = {"max_batch": mb, "input": kind, "frames_per_s": fps,
                       "h2d_frame_bytes_per_frame": round(h2d_frame_bytes(kind, frames)), "equal_to_run": same}
                print(json.dumps(dict(row, config=tag)), flush=True)
                line["run_batch"].append(row)
        report["configs"].append(line)
    del det
    # the unquantised CoDeNet2x COCO at scale 1
    cfg = NetConfig(num_classes=80, w2=True)
    g = np.load(os.path.join(ROOT, "tests", "golden", "codenet_float_2x_coco_256.npz"))
    raw = make_raw_state(cfg, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    fdet = compat.CtdetDetector(default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()},
                                            f32_gemm="tf32x3", heads={"hm": 80, "wh": 2, "reg": 2}, num_classes=80, w2=True))
    want_bgr = [fdet.run(f)["results"] for f in frames[:shared]]
    want_yuv = [fdet.run(to_bgr(f))["results"] for f in kinds_in["host I420"][:shared]]
    fdet.opt.max_batch = 256
    line = {"config": "CoDeNet2x COCO float (tf32x3), scale 1", "run_batch": []}
    for kind in KINDS:
        want = want_yuv if "I420" in kind or "NV12" in kind else want_bgr
        fps, same = time_run_batch(fdet, kinds_in[kind], want, 80)
        row = {"max_batch": 256, "input": kind, "frames_per_s": fps, "h2d_frame_bytes_per_frame": round(h2d_frame_bytes(kind, frames)),
               "equal_to_run": same}
        print(json.dumps(dict(row, config=line["config"])), flush=True)
        line["run_batch"].append(row)
    report["configs"].append(line)
    del fdet
    report["warp_kernel"] = warp_alone(frames, kinds_in, a.reps)
    report["warp_kernel_note"] = "256 descriptors into 256 slots of 512x512x3, no mirror; bytes moved = sources + destinations"
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "detect_frames.json"), "w") as f:
            json.dump(report, f, indent=1)
    bad = [r for c in report["configs"] for r in c["run_batch"] if r["equal_to_run"] != "%d/%d" % (shared, shared)]
    if bad or not all(w.get("equal_to_pool_kernel", True) for w in report["warp_kernel"]):
        raise SystemExit("run_batch and run() differ: %s" % bad)


if __name__ == "__main__":
    main()
