"""GPU box only: CtdetDetector.run_batch for the unquantised model (many raw frames per engine step, one ragged warp-and-normalise
launch per step, EngineF32 eagerly) against a run() loop, and the kernel cdn_warp_affine_u8_f32_batch alone.

Two seeded synthetic float models at 512x512, both with gemm="tf32x3": CoDeNet1x (VOC, 20 classes) and CoDeNet2x COCO (80
classes, BASELINE config 5's geometry); weights from synth.make_raw_state(seed 0) with the BatchNorm statistics of
tests/golden/codenet_float_*_256.npz.  1024 seeded uint8 frames in the VOC-like mix of tools/bench_detect_batch.py.  Per model and
configuration (scale 1; scale 1 + flip; five scales + flip + nms): frames/s of a run() loop over the first 128 frames, frames/s
of run_batch over all frames at max_batch 32, 128 and 256 (--passes timed passes after one untimed pass over the same frames:
the median and every pass are reported, since other work on the host moves single passes by up to 2x), the H2D
bytes per frame of run_batch's staging copies, and whether run_batch's results equal run()'s on the 128 shared frames (the
script exits non-zero if any does not).  Then the kernel alone: CUDA-event time over --reps launches of a 256-slot ragged batch
(scale 1 frames of the mix into 512x512 fp32 slots, without and with the mirror), bytes = sources + destinations (+ mirrors).
The card's name and power limit are read in the same run.  Writes detect_batch_f32.json into --out-dir."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from codenet_b200 import _lib, compat  # noqa: E402
from codenet_b200.arch import NetConfig  # noqa: E402
from codenet_b200.compat.detector import default_opt, plan_frame_steps  # noqa: E402
from codenet_b200.synth import make_raw_state  # noqa: E402
from bench_detect_batch import BATCHES, CONFIGS, SHAPES, card, equal, h2d_bytes_per_frame  # noqa: E402

MODELS = (("CoDeNet1x VOC", "1x", NetConfig(num_classes=20)), ("CoDeNet2x COCO", "2x_coco", NetConfig(num_classes=80, w2=True)))


def float_detector(tag, cfg, res=512):
    g = np.load(os.path.join(ROOT, "tests", "golden", "codenet_float_%s_256.npz" % tag))
    raw = make_raw_state(cfg, 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    nc = cfg.num_classes
    opt = default_opt(resume_quantize=False, state_dict={k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()},
                      input_h=res, input_w=res, f32_gemm="tf32x3", heads={"hm": nc, "wh": 2, "reg": 2}, num_classes=nc, w2=cfg.w2)
    return compat.CtdetDetector(opt)


def warp_alone(det, frames, reps, mirror):
    """256 output slots from scale-1 frames of the mix: 256 descriptors, or 128 with a mirror each, through the device table."""
    det.opt.flip_test, det.scales = mirror, [1.0]
    n = 128 if mirror else 256
    layouts = [det._frame_layout(f.shape[0], f.shape[1], [1.0]) for f in frames[:n]]
    (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in L] for L in layouts], 2 if mirror else 1, 256)
    pool = np.empty(nbytes, np.uint8)
    desc = np.empty(n, _lib.WARP_DESC)
    for k in range(n):
        det._pack_frame(frames[k], layouts[k], [1.0], pool, offsets[k], desc[k:k + 1], k * (2 if mirror else 1))
    d_pool = torch.from_numpy(pool).cuda()
    dst = torch.empty((256, 3, 512, 512), dtype=torch.float32, device="cuda")
    tables, index = det._norm_tables(0), det._table_index([1.0], n)
    for _ in range(5):
        det._warp_f32(d_pool, desc, index, tables, dst)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        det._warp_f32(d_pool, desc, index, tables, dst)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    src = int(sum(f.nbytes for f in frames[:n]))
    out = dst.numel() * 4
    moved = src + out
    return {"slots": 256, "descriptors": n, "mirror": mirror, "launches_timed": reps, "ms_per_launch": round(ms, 4),
            "source_bytes": src, "destination_bytes": int(out), "GB_per_s": round(moved / ms / 1e6, 1),
            "working_set_note": "sources + destinations %.0f MB, above the 126 MB L2" % (moved / 1e6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--loop-frames", type=int, default=128)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--out-dir", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detect_batch_f32 needs a GPU")
    name, power = card()
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, SHAPES[int(rng.integers(0, 4))] + (3,), dtype=np.uint8) for _ in range(a.frames)]
    shared = frames[:a.loop_frames]
    report = {"card": name, "power_limit": power, "frames": a.frames, "frame_mix": ["%dx%d" % (w, h) for h, w in SHAPES],
              "models": []}
    ok = True
    for model, tag, cfg in MODELS:
        det = float_detector(tag, cfg)
        nc = det.num_classes
        entry = {"model": "synthetic float %s (%d classes), 512x512, gemm tf32x3, EngineF32 eager" % (model, nc), "configs": []}
        for ctag, scales, flip, nms in CONFIGS:
            det.scales, det.opt.test_scales, det.opt.flip_test, det.opt.nms = scales, scales, flip, nms
            det.opt.max_batch = 1
            for f in shared[:4]:
                det.run(f)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            want = [det.run(f)["results"] for f in shared]
            t_loop = time.perf_counter() - t0
            line = {"model": model, "config": ctag, "run_loop": {"frames": len(shared), "frames_per_s": round(len(shared) / t_loop, 1)},
                    "run_batch": []}
            for mb in BATCHES:
                det.opt.max_batch = mb
                det.run_batch(frames)                            # EngineF32 workspaces, staging growth
                rates, same = [], len(shared)
                for _ in range(a.passes):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    got = det.run_batch(frames)
                    rates.append(round(len(frames) / (time.perf_counter() - t0), 1))
                    same = min(same, sum(equal(g["results"], w, nc) for g, w in zip(got, want)))
                ok &= same == len(shared)
                line["run_batch"].append({"max_batch": mb, "frames_per_s": float(np.median(rates)), "frames_per_s_passes": rates,
                                          "h2d_bytes_per_frame": round(h2d_bytes_per_frame(det, frames, mb)),
                                          "equal_to_run": "%d/%d" % (same, len(shared))})
            line["network_input_f32_bytes_per_frame"] = 512 * 512 * 3 * 4 * len(scales) * (2 if flip else 1)
            print(json.dumps(line), flush=True)
            entry["configs"].append(line)
        report["models"].append(entry)
        if tag == "1x":
            report["warp_f32_kernel"] = [warp_alone(det, frames, a.reps, False), warp_alone(det, frames, a.reps, True)]
            for w in report["warp_f32_kernel"]:
                w["bytes_moved_note"] = "uint8 sources + fp32 destinations (mirror slots included in the destinations)"
                print(json.dumps(w), flush=True)
        del det
        torch.cuda.empty_cache()
    if a.out_dir:
        os.makedirs(a.out_dir, exist_ok=True)
        with open(os.path.join(a.out_dir, "detect_batch_f32.json"), "w") as f:
            json.dump(report, f, indent=1)
    if not ok:
        raise SystemExit("run_batch and run() differ")


if __name__ == "__main__":
    main()
