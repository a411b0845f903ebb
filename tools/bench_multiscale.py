"""GPU box only: CtdetDetector.run() with multi-scale testing / --nms on one GPU, the device path (all scales in one engine batch,
post-affine + grouping + cdn_ctdet_merge on the device) against the host composition it replaces (per scale pre_process ->
process -> post_process, then merge_outputs with the host soft_nms mirror), alternating frame by frame in one process.

Per configuration: per-image wall time of both paths (median over the frames), the device time of cdn_ctdet_merge from CUDA
events, and whether every frame's results are equal between the two paths.  Synthetic calibrated W4A8 CoDeNet1x (VOC, 20
classes) at 512x512, seeded 480x640 uint8 frames.  Prints one JSON line per configuration (and writes them to --out)."""
import argparse
import ctypes as C
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
from codenet_b200.compat.detector import default_opt, get_affine_transform  # noqa: E402
from codenet_b200.synth import make_quant_state  # noqa: E402

CONFIGS = (("1 scale, nms", [1.0], False, True), ("5 scales", [0.5, 0.75, 1.0, 1.25, 1.5], False, False),
           ("5 scales, flip", [0.5, 0.75, 1.0, 1.25, 1.5], True, False))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # the number is reported as unknown rather than guessed
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


def host_composition(det, img):
    per_scale = []
    for scale in det.scales:
        images, meta = det.pre_process(img, scale)
        _, dets = det.process(images.to(det.opt.device))
        per_scale.append(det.post_process(dets, meta, scale))
    return det.merge_outputs(per_scale)


def merge_kernel_ms(det, img, reps):
    """CUDA-event time of one cdn_ctdet_merge call on this frame's grouped detections (mean over `reps` launches)."""
    L = _lib.load()
    (ih, iw) = det.input_geometry(img.shape[0], img.shape[1], det.scales[0])[1]
    images, metas = det._slots_u8(img, det.scales, ih, iw)
    _, dets = det.process(images)
    S, K, nc = dets.shape[0], dets.shape[1], det.num_classes
    d = dets.contiguous().clone()
    t = np.ascontiguousarray(np.stack([get_affine_transform(m['c'], m['s'], 0, (m['out_width'], m['out_height']), inv=1).reshape(6)
                                       for m in metas]), dtype=np.float64)
    g = torch.empty_like(d); counts = torch.empty((S, nc), dtype=torch.int32, device=d.device)
    rows = torch.empty((S * K, 5), dtype=torch.float32, device=d.device); cc = torch.empty(nc, dtype=torch.int32, device=d.device)
    sc = np.asarray(det.scales, np.float32)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.cdn_ctdet_post_affine(C.c_void_p(d.data_ptr()), S, K, C.c_void_p(t.ctypes.data), st))
    _lib.check(L.cdn_ctdet_group_by_class(C.c_void_p(d.data_ptr()), S, K, nc, C.c_void_p(g.data_ptr()), C.c_void_p(counts.data_ptr()), st))
    launch = lambda: _lib.check(L.cdn_ctdet_merge(C.c_void_p(g.data_ptr()), C.c_void_p(counts.data_ptr()), 1, S, K, nc,
                                                  C.c_void_p(sc.ctypes.data), int(bool(det.opt.nms)), 100, C.c_void_p(rows.data_ptr()),
                                                  C.c_void_p(cc.data_ptr()), st))
    for _ in range(5):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, int(cc.sum().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multiscale needs a GPU")
    name, power = card()
    cfg = NetConfig(num_classes=20)
    calib = np.load(os.path.join(ROOT, "tests", "golden", "codenet1x_calib.npz"))
    st = make_quant_state(cfg, calib, "round", 512)
    det = compat.CtdetDetector(default_opt(state_dict=st, offset_mode="round", max_batch=10))
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for _ in range(a.frames)]
    lines = []
    for tag, scales, flip, nms in CONFIGS:
        det.scales, det.opt.test_scales, det.opt.flip_test, det.opt.nms = scales, scales, flip, nms
        for img in frames[:2]:                                   # warm-up of both paths (engine, cv2, modules)
            det.run(img); host_composition(det, img)
        torch.cuda.synchronize()
        t_dev, t_host, equal = [], [], 0
        for img in frames:
            t0 = time.perf_counter()
            got = det.run(img)["results"]
            t1 = time.perf_counter()
            want = host_composition(det, img)
            t2 = time.perf_counter()
            t_dev.append(t1 - t0); t_host.append(t2 - t1)
            equal += all(np.array_equal(got[j], want[j]) for j in range(1, det.num_classes + 1))
        k_ms, kept = merge_kernel_ms(det, frames[0], a.reps)
        line = {"config": tag, "card": name, "power_limit": power, "frames": a.frames, "input": "480x640 uint8 -> 512x512",
                "device_path_ms_per_image": round(1e3 * float(np.median(t_dev)), 3),
                "host_path_ms_per_image": round(1e3 * float(np.median(t_host)), 3),
                "merge_kernel_ms": round(k_ms, 4), "rows_kept_frame0": kept, "frames_equal": "%d/%d" % (equal, a.frames)}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")
    if any(x["frames_equal"] != "%d/%d" % (a.frames, a.frames) for x in lines):
        raise SystemExit("device and host paths differ")


if __name__ == "__main__":
    main()
