"""GPU box only: CtdetDetector.run_batch (many raw frames per engine step, ragged warp on the device, pipelined staging) against
a run() loop, and the ragged warp kernel cdn_warp_affine_u8_batch alone.

Seeded synthetic calibrated W4A8 CoDeNet1x (VOC, 20 classes) at 512x512 with the detector's default bilinear offsets
(--offset-mode round for the integer mode), 1024 seeded uint8 frames in a VOC-like mix of 500x375, 375x500, 500x333 and
333x500.  Per configuration (scale 1; scale 1 + flip; five scales + flip + nms): frames/s of a run() loop over the first 128
frames (opt.max_batch = 1, the default), frames/s of run_batch over all frames at max_batch 32, 128 and 256 (each timed after
one untimed pass over the same frames), the H2D bytes per frame of run_batch's staging copies, and whether run_batch's results
equal run()'s on the 128 shared frames.  Then the warp kernel alone: CUDA-event time over --reps launches of a 256-slot ragged
batch (scale 1 frames of the mix into 512x512 slots, without and with the mirror), bytes = sources + destinations (+ mirrors).
The card's name and power limit are read in the same run.  Writes detect_batch.json into --out-dir."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from codenet_b200 import _lib, compat  # noqa: E402
from codenet_b200.arch import NetConfig  # noqa: E402
from codenet_b200.compat.detector import default_opt, plan_frame_steps  # noqa: E402
from codenet_b200.synth import make_quant_state  # noqa: E402

SHAPES = ((375, 500), (500, 375), (333, 500), (500, 333))
CONFIGS = (("scale 1", [1.0], False, False), ("scale 1, flip", [1.0], True, False),
           ("5 scales, flip, nms", [0.5, 0.75, 1.0, 1.25, 1.5], True, True))
BATCHES = (32, 128, 256)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # the number is reported as unknown rather than guessed
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


def equal(a, b, nc):
    return all(np.array_equal(a[j], b[j]) for j in range(1, nc + 1))


def h2d_bytes_per_frame(det, frames, max_batch):
    """What run_batch copies host -> device: every step's staging pool (frames and resized copies, 16-byte aligned)."""
    spf = len(det.scales) * (2 if det.opt.flip_test else 1)
    sizes = [[sh * sw * 3 for sh, sw, _, _ in det._frame_layout(f.shape[0], f.shape[1], det.scales)] for f in frames]
    return sum(nb for _, _, nb in plan_frame_steps(sizes, spf, max_batch)) / len(frames)


def warp_alone(frames, reps, mirror):
    """256 output slots from scale-1 frames of the mix: 256 descriptors, or 128 with a mirror each."""
    det = compat.CtdetDetector.__new__(compat.CtdetDetector)
    det.opt = default_opt(flip_test=mirror)
    det.scales = [1.0]
    n = 128 if mirror else 256
    layouts = [det._frame_layout(f.shape[0], f.shape[1], [1.0]) for f in frames[:n]]
    (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in L] for L in layouts], 2 if mirror else 1, 256)
    pool = np.empty(nbytes, np.uint8)
    desc = np.empty(n, _lib.WARP_DESC)
    for k in range(n):
        det._pack_frame(frames[k], layouts[k], [1.0], pool, offsets[k], desc[k:k + 1], k * (2 if mirror else 1))
    d_pool = torch.from_numpy(pool).cuda()
    dst = torch.empty((256, 512, 512, 3), dtype=torch.uint8, device="cuda")
    for _ in range(5):
        det._warp(d_pool, desc, dst)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        det._warp(d_pool, desc, dst)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    src = int(sum(f.nbytes for f in frames[:n]))
    moved = src + dst.numel()
    return {"slots": 256, "descriptors": n, "mirror": mirror, "launches_timed": reps, "ms_per_launch": round(ms, 4),
            "source_bytes": src, "destination_bytes": int(dst.numel()), "GB_per_s": round(moved / ms / 1e6, 1),
            "working_set_note": "sources + destinations %.0f MB, above the 126 MB L2" % (moved / 1e6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--loop-frames", type=int, default=128)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--offset-mode", default="bilinear", choices=("bilinear", "round"))
    ap.add_argument("--out-dir", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detect_batch needs a GPU")
    name, power = card()
    cfg = NetConfig(num_classes=20)
    calib = np.load(os.path.join(ROOT, "tests", "golden", "codenet1x_calib.npz"))
    st = make_quant_state(cfg, calib, a.offset_mode, 512)
    det = compat.CtdetDetector(default_opt(state_dict=st, offset_mode=a.offset_mode))
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, SHAPES[int(rng.integers(0, 4))] + (3,), dtype=np.uint8) for _ in range(a.frames)]
    shared = frames[:a.loop_frames]
    nc = det.num_classes
    report = {"card": name, "power_limit": power, "model": "synthetic W4A8 CoDeNet1x, 20 classes, 512x512, offsets %s" % a.offset_mode,
              "frames": a.frames, "frame_mix": ["%dx%d" % (w, h) for h, w in SHAPES], "configs": []}
    for tag, scales, flip, nms in CONFIGS:
        det.scales, det.opt.test_scales, det.opt.flip_test, det.opt.nms = scales, scales, flip, nms
        det.opt.max_batch = 1
        for f in shared[:4]:
            det.run(f)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        want = [det.run(f)["results"] for f in shared]
        t_loop = time.perf_counter() - t0
        line = {"config": tag, "run_loop": {"frames": len(shared), "frames_per_s": round(len(shared) / t_loop, 1)}, "run_batch": []}
        for mb in BATCHES:
            det.opt.max_batch = mb
            det.run_batch(frames)                                # engine build, graph capture, staging growth
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = det.run_batch(frames)
            dt = time.perf_counter() - t0
            same = sum(equal(g["results"], w, nc) for g, w in zip(got, want))
            line["run_batch"].append({"max_batch": mb, "frames_per_s": round(len(frames) / dt, 1),
                                      "h2d_bytes_per_frame": round(h2d_bytes_per_frame(det, frames, mb)),
                                      "equal_to_run": "%d/%d" % (same, len(shared))})
        line["network_input_u8_bytes_per_frame"] = 512 * 512 * 3 * len(scales) * (2 if flip else 1)
        print(json.dumps(line), flush=True)
        report["configs"].append(line)
    report["warp_kernel"] = [warp_alone(frames, a.reps, False), warp_alone(frames, a.reps, True)]
    for w in report["warp_kernel"]:
        w["bytes_moved_note"] = "sources + destinations (mirror slots included in the destinations)"
        print(json.dumps(w), flush=True)
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "detect_batch.json"), "w") as f:
            json.dump(report, f, indent=1)
    if any(r["equal_to_run"] != "%d/%d" % (len(shared), len(shared)) for c in report["configs"] for r in c["run_batch"]):
        raise SystemExit("run_batch and run() differ")


if __name__ == "__main__":
    main()
