#!/usr/bin/env python
"""Benchmark of the hot path: CoDeNet W4A8 forward + ctdet decode, images/s (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference's PyTorch CPU forward on the host
    python bench.py --config {c,e,2x_fp32}                   # c (default) = the metric's config; e / 2x_fp32 = configs 4 / 5
    python bench.py --dump-outputs DIR                       # also write the last timed step's detections / indices (.npy) to
                                                             # DIR: same arguments, same inputs, so two builds can be compared

One JSON line on stdout (rank 0).
  value         whole-job images/s, inputs resident in HBM, CUDA events, max over ranks
  parity_checked  the timed step's detections / indices of the distinct images compared with the oracle AFTER the timed
                loop (outside the timed region); the run fails (exit 3) on a mismatch
  e2e           the same metric through the public host API (Engine.submit_host / wait: pinned uint8 images in, detections
                out, H2D and D2H inside the timed region, two steps in flight), plus the measured H2D fabric ceiling
  roofline      algorithmic bytes / device time of the dominant kernel family against the measured HBM peak
  deform        the three fused deformable layers (SURVEY 8(d) algorithmic bytes) against the HBM peak
  cpu_baseline  the reference's own CPU forward (oracle/ref_cpu_bench.py, kind "reference") on this box's host cores on a
                bounded sample, with the numpy port as a second, labelled number
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "images/s"
FALLBACK_HBM_GBS = 6650.0


def configs():
    from codenet_b200.arch import NetConfig
    return {
        "c": dict(cfg=NetConfig(num_classes=20), calib="codenet1x_calib.npz", res=512, batch=256,
                  metric="CoDeNet1x 512x512 W4A8 forward + ctdet decode throughput",
                  workload="BASELINE config c: CoDeNet1x 512x512 stride-4 W4A8, 20 classes, K=100, batch %d per GPU"),
        "e": dict(cfg=NetConfig(num_classes=20, w2=True, maxpool=True), calib="codenet_w2mp_calib.npz", res=512, batch=256,
                  metric="CoDeNet w2 (S2+MaxPool) 512x512 W4A8 forward + ctdet decode throughput",
                  workload="BASELINE config e: CoDeNet w2 width, stride-2 stem + MaxPool, 512x512 W4A8, 20 classes, K=100, "
                           "batch %d per GPU"),
        "2x_fp32": dict(cfg=NetConfig(num_classes=80, w2=True), calib=None, res=512, batch=128,
                        metric="CoDeNet2x fp32 COCO 512x512 forward + ctdet decode throughput",
                        workload="BASELINE config 5: CoDeNet2x (w2, stride-4) fp32, 80 classes, bilinear offsets, 512x512, "
                                 "K=100, batch %d per GPU"),
    }


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---- algorithmic bytes per op (DESIGN.md / SURVEY.md 8(d)) ----------------------------------------------------------
def op_bytes(plan, op, batch, stored=False):
    """Bytes one launch must move: logical input elements read once + logical output elements written once.
    Deformable layers follow SURVEY 8(d): B*(C*H*W*e_in + C*Ho*Wo*e_out) + 9*C with H, W the layer's LOGICAL input size (the
    nearest x2 upsample in front of two of them is virtual here, so the bytes actually stored are fewer: `stored=True`)."""
    a = op.a
    T = plan.tensors
    if op.kind == "stem":
        to = T[a["out_t"]]
        return batch * (3 * a["H"] * a["W"] * 4 + to.C * to.H * to.W)
    if op.kind == "dw" and a.get("fused_into_next"):
        # heads tail as one kernel: stored int8 input read once, fp32 planes written once; nothing in between touches HBM
        ti = T[a["in_t"]]
        return batch * (ti.C * ti.H * ti.W + 4 * a["fused_n_f32"] * 4 * ti.H * ti.W) + 9 * ti.C
    if a.get("fused_with_prev"):
        return 0
    if a.get("unit_head"):
        # a whole stride-1 unit as one kernel: the stage tensor (both halves) read once, the unit's output written once, the
        # weights of its three convs; the two int8 tensors between the convs never touch HBM
        ti = T[a["in_t"]]
        if a["unit_head"] == 2:                  # stride-2 branch: input read once, branch 1's output read once, unit output written once
            co = 2 * a["N_real"]
            return batch * (ti.H * ti.W * ti.C + (ti.H // 2) * (ti.W // 2) * (co // 2 + co)) + a["unit_weights"]
        return batch * ti.H * ti.W * 2 * ti.C + a["unit_weights"]
    if op.kind == "deform" and not stored:
        to = T[a["out_t"]]
        return batch * 2 * to.C * to.H * to.W + 9 * to.C
    if op.kind in ("dw", "deform"):
        ti, to = T[a["in_t"]], T[a["out_t"]]
        return batch * (ti.C * ti.H * ti.W + to.C * to.H * to.W) + 9 * ti.C
    ti = T[a["in_t"]]
    k_real = int((np.abs(a["wq"]).sum(0) > 0).sum())
    px = batch * ti.H * ti.W
    if a["n_f32"]:
        return px * (k_real + 4 * a["n_f32"])
    n_pass = sum(int(c[1]) for c in a["chunks"] if c[2] >= 0)
    n_new = sum(int(c[1]) for c in a["chunks"])
    return px * (k_real + n_pass + n_new + n_pass) + a["wq"].size


def family(op):
    if op.a.get("unit_head") or op.a.get("unit_member"):
        return "unit_fused_kernel"
    if op.a.get("fused_into_next") or op.a.get("fused_with_prev"):
        return "heads_fused_kernel"
    if op.kind == "deform":
        return "deform_int_kernel" if op.a.get("mode", 0) == 0 else "deform_bilinear_kernel"
    return {"pw": "pw_gemm_tc_kernel", "dw": "dw3x3_kernels", "stem": "stem_kernel"}[op.kind]


def ncu_traffic():
    """DRAM bytes per step and kernel family from the latest committed ncu launch list (profiles/*_families.json)."""
    d = os.path.join(ROOT, "profiles")
    try:
        f = sorted(x for x in os.listdir(d) if x.endswith("_families.json"))[-1]
        j = json.load(open(os.path.join(d, f)))
        return {k: (v["dram_bytes"], v["launches"]) for k, v in j["families"].items()}, f
    except Exception:
        return {}, None


def check_parity(cfg, st, mode, base, dets, inds, n_check):
    """Engine detections / indices of a step against the oracle for the first `n_check` distinct images, and every replica
    of the tiled batch against its original.  Returns (ok, message).  Outside any timed region."""
    from oracle import int_oracle as io
    n_base = base.shape[0]
    B = dets.shape[0]
    cat = cfg.num_classes
    o = io.IntOracle(cfg, st, mode)
    for i in range(min(n_check, n_base, B)):
        ref = o.forward(base[i:i + 1])
        want = np.concatenate([ref["hm"], ref["wh"], ref["reg"]], 1).astype(np.float32).astype(np.float64)
        odets, oinds = io.ctdet_decode(want[:, :cat], want[:, cat:cat + 2], want[:, cat + 2:cat + 4], dets.shape[1])
        if not np.array_equal(inds[i], oinds[0]):
            return False, "image %d: top-K indices differ from the oracle (%d of %d)" % (i, int((inds[i] != oinds[0]).sum()), inds.shape[1])
        if not np.allclose(dets[i], odets[0], rtol=1e-5, atol=1e-4):
            return False, "image %d: detections differ from the oracle (max abs %.3g)" % (i, float(np.abs(dets[i] - odets[0]).max()))
    for b in range(n_base, B):
        if not (np.array_equal(inds[b], inds[b % n_base]) and np.array_equal(dets[b], dets[b % n_base])):
            return False, "replica %d differs from image %d" % (b, b % n_base)
    return True, "dets + inds of %d distinct images equal the oracle; %d replicas equal their originals" % (
        min(n_check, n_base, B), max(B - n_base, 0))


DUMP_BYTES = 64_000_000


def dump_outputs(path, arrays):
    """Writes what one timed step returned as <path>/<name>.npy, so that two builds can be compared output for output: float32
    arrays as they are, integer ones as float64 (exact).  The arrays share the batch axis; if together they exceed 64 MB, the
    same fixed, seeded sample of images is kept from each and its batch indices are written as sample.npy."""
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    B = next(iter(arrays.values())).shape[0]
    per_image = sum(v.nbytes for v in arrays.values()) // B
    if per_image * B > DUMP_BYTES:
        n = (DUMP_BYTES - 4096 * (len(arrays) + 1)) // (per_image + 8)          # room for the .npy headers and sample.npy
        keep = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["sample"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(v))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from codenet_b200.engine import Engine
    from codenet_b200.synth import make_quant_state, make_images

    C = configs()[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = C["cfg"]
    calib = np.load(os.path.join(ROOT, "tests", "golden", C["calib"]))
    B, R = args.batch or C["batch"], C["res"]
    st = make_quant_state(cfg, calib, args.offset_mode, R)
    eng = Engine.from_state_dict(cfg, st, R, R, B, offset_mode=args.offset_mode, device=local)
    if args.no_fuse_heads:
        eng.set_option("fuse_heads", 0)
    if eng.heads_fused:                          # heads.dw2 + heads.out run as one kernel: account them as one launch
        ops = eng.plan.ops
        i = next(k for k, o in enumerate(ops) if o.name == "heads.dw2")
        ops[i].a["fused_into_next"], ops[i].a["fused_n_f32"], ops[i + 1].a["fused_with_prev"] = True, ops[i + 1].a["n_f32"], True
    if args.no_fuse_units:
        eng.set_option("fuse_units", 0)
    ops = eng.plan.ops
    for i in range(len(ops)):                    # stride-1 units that run as one kernel: account the three ops as one launch
        if eng.op_fusion(i) in (2, 3):
            ops[i].a["unit_head"] = 2 if eng.op_fusion(i) == 3 else 1
            ops[i].a["unit_weights"] = int(ops[i].a["wq"].size + ops[i + 1].a["wq"].size + ops[i + 2].a["wq"].size)
            ops[i].a["N_real"] = int(eng.plan.tensors[ops[i].a["out_t"]].C)
            for o in ops[i + 1:i + 3]:
                o.a["fused_with_prev"], o.a["unit_member"] = True, True
    eng.set_option("host_chunk", args.host_chunk)
    # synthetic images: 16 distinct ones per rank, tiled to the batch (805 MB fp32 at B=256: larger than L2)
    base = make_images(min(16, B), R, seed=100 + rank)
    reps = (B + base.shape[0] - 1) // base.shape[0]
    host = torch.from_numpy(np.concatenate([base] * reps)[:B].copy()).pin_memory()
    dev = host.cuda(non_blocking=True)
    torch.cuda.synchronize()
    out = {}

    def step():
        eng.run(dev, maps=False, dets=True, out=out)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(flag):
        t = torch.tensor([0 if flag else 1], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item()) == 0

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    value = world * B * args.steps / (ms / 1e3)

    # ---- parity of what was just timed (outside the timed region): every rank checks its own images --------------------
    dev_dets, dev_inds = out["dets"].cpu().numpy(), out["inds"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"dets": dev_dets, "inds": dev_inds})
    n_check = args.parity_images if world == 1 else min(args.parity_images, 4)
    p_ok, p_msg = check_parity(cfg, st, args.offset_mode, base, dev_dets, dev_inds, n_check)
    parity_ok = all_ok(p_ok)

    # ---- end to end through host buffers ------------------------------------------------------------------------------
    # Detector-level input: uint8 HWC images at the input size, as cv2 hands them to the reference's run() (pre_process is
    # then normalisation only, applied inside the stem kernel).  Engine.submit_host / wait with two steps in flight: the
    # H2D copy of step n+1 overlaps the compute of step n; every step's detections are copied back to pinned host memory.
    mean, std = np.array([0.485, 0.456, 0.406], np.float32), np.array([0.229, 0.224, 0.225], np.float32)
    eng.set_normalization(mean, std)
    hnp = host.numpy()
    u8 = np.clip(np.rint((hnp.transpose(0, 2, 3, 1) * std + mean) * 255.0), 0, 255).astype(np.uint8)
    u8_t = torch.from_numpy(np.ascontiguousarray(u8)).pin_memory()
    u8 = u8_t.numpy()
    bufs = [(torch.empty((B, eng.K, 6), dtype=torch.float32).pin_memory(), torch.empty((B, eng.K), dtype=torch.int32).pin_memory())
            for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 20))

    def run_pipelined(n):
        for i in range(n):
            sl = i & 1
            if i >= 2:
                eng.wait(sl)
            eng.submit_host(u8, bufs[sl][0].numpy(), bufs[sl][1].numpy(), sl)
        eng.wait(0)
        eng.wait(1)

    def timed(fn, n):
        fn(2)
        barrier()
        t0 = time.perf_counter()
        fn(n)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        return world * B * n / dt

    e2e_val = timed(run_pipelined, e2e_steps)
    # the uint8 path's detections (quantised pixels) against the same engine on the same uint8 images resident on the device
    u8_dev = u8_t.cuda()
    o8 = eng.run(u8_dev, maps=False, dets=True)
    torch.cuda.synchronize()
    e2e_same = all(np.array_equal(bufs[s][1].numpy(), o8["inds"].cpu().numpy()) and
                   np.array_equal(bufs[s][0].numpy(), o8["dets"].cpu().numpy()) for s in (0, 1))
    e2e_ok = all_ok(e2e_same)

    dets_h, inds_h = bufs[0][0].numpy(), bufs[0][1].numpy()

    def run_serial(n):
        for _ in range(n):
            eng.run_host(u8, dets_h, inds_h)

    e2e_serial = timed(run_serial, max(2, e2e_steps // 2))

    # fabric ceiling: every rank copies the same pinned uint8 batch to its GPU, all ranks at once, nothing else running
    copy_stream = torch.cuda.Stream()
    fab_n = 10

    def run_copies(n):
        with torch.cuda.stream(copy_stream):
            for _ in range(n):
                u8_dev.copy_(u8_t, non_blocking=True)
        copy_stream.synchronize()

    fabric_ips = timed(run_copies, fab_n)
    fabric_gbs = fabric_ips * 3 * R * R / 1e9
    clocks = sampler.stop() if rank == 0 else None

    # ---- the reference's default semantics (fractional offsets -> bilinear gather) on the same workload --------------------
    bil = None
    if args.offset_mode == "round" and not args.no_bilinear and ("ranges_bilinear_%d/stem" % R) in calib.files:
        st_b = make_quant_state(cfg, calib, "bilinear", R)
        eng_b = Engine.from_state_dict(cfg, st_b, R, R, B, offset_mode="bilinear", device=local)
        ob = {}
        for _ in range(3):
            eng_b.run(dev, maps=False, dets=True, out=ob)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nb = max(3, args.steps // 2)
        b0.record()
        for _ in range(nb):
            eng_b.run(dev, maps=False, dets=True, out=ob)
        b1.record()
        barrier()
        msb = max_over_ranks(b0.elapsed_time(b1))
        okb, msgb = check_parity(cfg, st_b, "bilinear", base, ob["dets"].cpu().numpy(), ob["inds"].cpu().numpy(), min(n_check, 4))
        okb = all_ok(okb)
        parity_ok = parity_ok and okb
        prb = eng_b.profile(dev) if rank == 0 else []
        bil = {"offset_mode": "bilinear", "value": round(world * B * nb / (msb / 1e3), 1), "unit": UNIT,
               "ms_per_step": round(msb / nb, 4), "parity_checked": bool(okb), "parity": msgb,
               "deform_ms": round(sum(t for n, k, t in prb if k == "deform"), 4),
               "note": "the reference's default arithmetic (quant_modules.py:668-671: fractional s, bilinear gather)"}
        eng_b.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if not (p_ok and e2e_same):
            sys.exit(3)
        return
    # ---- per-kernel times (eager, CUDA events between launches on the launching stream) -----------------------------
    prof_runs = 3
    acc = None
    for _ in range(prof_runs):
        pr = eng.profile(dev)
        acc = [x[2] for x in pr] if acc is None else [a + x[2] for a, x in zip(acc, pr)]
    per_op = [a / prof_runs for a in acc]
    if args.dump_ops:
        rows = [{"op": o.name, "kind": o.kind, "ms": round(m, 4), "MB": round(op_bytes(eng.plan, o, B) / 1e6, 1),
                 "GBps": round(op_bytes(eng.plan, o, B) / m / 1e6, 1) if m > 0 else None} for o, m in zip(eng.plan.ops, per_op)]
        rows.append({"op": "ctdet_decode", "kind": "decode", "ms": round(per_op[-1], 4)})
        with open(args.dump_ops, "w") as f:
            json.dump(rows, f, indent=1)
    fam_ms, fam_bytes, deform_layers = {}, {}, []
    for op, msop in zip(eng.plan.ops, per_op):
        f = family(op)
        by = op_bytes(eng.plan, op, B)
        fam_ms[f] = fam_ms.get(f, 0.0) + msop
        fam_bytes[f] = fam_bytes.get(f, 0) + by
        if op.kind == "deform":
            deform_layers.append({"layer": op.name, "C": int(op.a["C"]), "H": int(eng.plan.tensors[op.a["out_t"]].H),
                                  "ms": round(msop, 4), "GBps": round(by / msop / 1e6, 1),
                                  "GBps_stored": round(op_bytes(eng.plan, op, B, stored=True) / msop / 1e6, 1)})
    fam_ms["ctdet_decode"] = per_op[-1]
    fam_bytes["ctdet_decode"] = B * (eng.plan.cat + 4) * eng.plan.out_H * eng.plan.out_W * 4
    fam_launches = {"ctdet_decode": 2}
    for op in eng.plan.ops:
        if not op.a.get("fused_with_prev"):
            fam_launches[family(op)] = fam_launches.get(family(op), 0) + 1
    total_ms = sum(fam_ms.values())
    dom = max(fam_ms, key=fam_ms.get)
    peak, peak_src = peaks()
    ach = fam_bytes[dom] / fam_ms[dom] / 1e6
    traffic, traffic_src = ncu_traffic()
    tr = traffic.get(dom)
    roofline = {"kernel": dom, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4),
                "traffic": (round(tr[0] / tr[1]) if tr and B == 256 and args.config == "c" else None),
                "traffic_note": "mean DRAM bytes per launch of this family (ncu dram__bytes_read+write, %s); algorithmic bytes "
                                "per launch: %d" % (traffic_src, fam_bytes[dom] // max(fam_launches.get(dom, 1), 1)),
                "launches_per_step": fam_launches.get(dom), "peak_source": peak_src,
                "share_of_step": round(fam_ms[dom] / total_ms, 3),
                "whole_step": {"algorithmic_GB": round(sum(fam_bytes.values()) / 1e9, 3), "ms": round(total_ms, 4),
                               "GBps": round(sum(fam_bytes.values()) / total_ms / 1e6, 1),
                               "frac": round(sum(fam_bytes.values()) / total_ms / 1e6 / peak, 4)},
                "families": {k: {"ms": round(v, 4), "GBps": round(fam_bytes[k] / v / 1e6, 1), "share": round(v / total_ms, 3),
                                 "frac": round(fam_bytes[k] / v / 1e6 / peak, 4)}
                             for k, v in sorted(fam_ms.items(), key=lambda kv: -kv[1])}}
    dby = sum(op_bytes(eng.plan, op, B) for op in eng.plan.ops if op.kind == "deform")
    dbs = sum(op_bytes(eng.plan, op, B, stored=True) for op in eng.plan.ops if op.kind == "deform")
    dms = sum(v for k, v in fam_ms.items() if k.startswith("deform_"))
    deform = {"GBps": round(dby / dms / 1e6, 1), "frac_of_hbm_peak": round(dby / dms / 1e6 / peak, 4), "ms": round(dms, 4),
              "bytes": "SURVEY 8(d): B*(C*H*W + C*Ho*Wo) int8 per layer (2.10 MB/image in config c)",
              "GBps_stored": round(dbs / dms / 1e6, 1), "frac_stored": round(dbs / dms / 1e6 / peak, 4),
              "bytes_stored": "input bytes actually stored (the x2 upsample in front of two layers is virtual)",
              "layers": deform_layers}
    cpu = None if (args.no_cpu or world > 1) else cpu_baseline(args)     # rank 0 at N = 1 only
    bpi = 3 * R * R
    line = {
        "metric": C["metric"], "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int8",
        "data": "synthetic", "impl": "codenet_b200",
        "config": workload_config(args, B),
        "parity_checked": bool(parity_ok), "parity": p_msg,
        "e2e": {"value": round(e2e_val, 1), "unit": UNIT, "h2d_bytes_per_step": int(B * bpi),
                "d2h_bytes_per_step": int(B * eng.K * (6 * 4 + 4)), "steps": e2e_steps, "in_flight": 2,
                "input": "uint8 HWC images at the input size in pinned host memory (the detector's run() input; "
                         "normalisation inside the stem kernel), detections [B,100,6] + indices back to pinned host memory "
                         "every step",
                "api": "Engine.submit_host / Engine.wait -> cdn_engine_submit_host_u8 / cdn_engine_wait",
                "results_equal_device_path": bool(e2e_ok),
                "serial_value": round(e2e_serial, 1),
                "serial_api": "Engine.run_host -> cdn_engine_run_host_u8 (one step at a time, chunked copy/compute overlap inside the step)",
                "fabric": {"h2d_GBps_all_ranks": round(fabric_gbs, 2), "ceiling_images_per_s": round(fabric_ips, 1),
                           "e2e_frac_of_ceiling": round(e2e_val / fabric_ips, 4),
                           "how": "%d plain pinned cudaMemcpyAsync H2D copies of the step's uint8 batch per rank, all %d "
                                  "ranks at once, no compute" % (fab_n, world)}},
        "gpu_launches": int(eng.num_launches * args.steps),
        "requant": dict(zip(("int_layers", "guarded_fp32_layers"), eng.requant_stats)),
        "heads_fused": bool(eng.heads_fused), "units_fused": int(eng.units_fused),
        "clocks": clocks, "roofline": roofline, "deform": deform, "reference_semantics": bil, "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not (parity_ok and e2e_ok):
        sys.stderr.write("bench.py: PARITY FAILURE: %s (e2e equal: %s)\n" % (p_msg, e2e_ok))
        sys.exit(3)


def workload_config(args, B):
    C = configs()[args.config]
    R = C["res"]
    return {"workload": C["workload"] % B, "name": args.config, "batch_per_gpu": B, "offset_mode": args.offset_mode,
            "arithmetic": "s8 x s8 -> s32 (4-bit weights, 8-bit activations), exact integer requantisation",
            "parallelism": "batch-sharded, no collective",
            "l2": "inputs larger than L2 (%.0f MB fp32 images per step)" % (B * 3 * R * R * 4 / 1e6),
            "outputs": "detections [B,100,6] (+ heat-map/wh/reg maps on request)"}


# ---- CPU arm ----------------------------------------------------------------------------------------------------------
def cpu_reference(args, steps, warmup, budget_s):
    """The UNMODIFIED reference's PyTorch CPU forward + ctdet_decode (oracle/ref_cpu_bench.py) on all host cores, batch 8."""
    from oracle import ref_cpu_bench
    C = configs()[args.config]
    r = ref_cpu_bench.measure(C["cfg"], args.offset_mode, res=C["res"], batch=8, steps=steps, warmup=warmup, budget_s=budget_s,
                              calib_name=C["calib"])
    r["sample"] = ("%d timed steps (median) of the UNMODIFIED reference: PoseShuffleNetV2 + quantize_shufflenetv2_dcn forward, "
                   "sigmoid, ctdet_decode on a batch of %d %dx%d images, fp32, torch.set_num_threads(%d), QuantAct ranges "
                   "frozen, weights re-quantised every call, torchvision CPU deform_conv2d in place of the CUDA-only op "
                   "(oracle/ref_cpu_bench.py)" % (r["steps"], r["batch"], C["res"], C["res"], r["cores"]))
    return r


def cpu_port(args, seconds=10.0):
    from oracle import cpu_bench
    value, workers, n = cpu_bench.measure(args.offset_mode, seconds=seconds)
    return {"value": round(value, 3), "unit": UNIT, "cores": workers, "kind": "port",
            "sample": "%d x (forward + decode) of 1 image at 512x512 in %.0f s on %d worker processes, integer-exact numpy oracle "
                      "(oracle/int_oracle.py via oracle/cpu_bench.py)" % (n, seconds, workers)}


def cpu_baseline(args):
    from oracle import ref_cpu_bench
    if ref_cpu_bench.available():
        r = cpu_reference(args, steps=5, warmup=1, budget_s=25.0)
        cpu = {"value": round(r["value"], 3), "unit": UNIT, "cores": r["cores"], "kind": "reference", "sample": r["sample"]}
        if args.config == "c" and not args.no_port:
            cpu["port"] = cpu_port(args, seconds=6.0)
        return cpu
    return cpu_port(args)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_cpu_bench
    C = configs()[args.config]
    B = args.batch or C["batch"]
    if ref_cpu_bench.available():
        r = cpu_reference(args, steps=max(args.steps, 2), warmup=max(1, min(args.warmup, 3)), budget_s=150.0)
        cpu = {"value": round(r["value"], 3), "unit": UNIT, "cores": r["cores"], "kind": "reference", "sample": r["sample"]}
        ms_step, steps, dtype = r["ms_per_step"], r["steps"], "fp32 (fake-quantised W4A8, PyTorch CPU)"
    else:
        cpu = cpu_port(args)
        ms_step, steps, dtype = 1e3 / max(cpu["value"], 1e-9), args.steps, "fp64/int64 (numpy)"
    line = {"metric": C["metric"], "value": cpu["value"], "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
            "steps": steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype,
            "data": "synthetic", "impl": "reference",
            "config": workload_config(args, B),
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c", choices=["c", "e", "2x_fp32"])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's, 256 for c / e)")
    ap.add_argument("--offset-mode", default="round", choices=["round", "bilinear"])
    ap.add_argument("--host-chunk", type=int, default=64)
    ap.add_argument("--parity-images", type=int, default=16, help="distinct images compared with the oracle after the timed loop")
    ap.add_argument("--no-fuse-heads", action="store_true", help="run heads.dw2 and heads.out as separate kernels (A/B)")
    ap.add_argument("--no-fuse-units", action="store_true", help="run every ShuffleNetV2 unit as three launches (A/B)")
    ap.add_argument("--no-bilinear", action="store_true", help="skip the reference-semantics (bilinear offsets) leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs only)")
    ap.add_argument("--no-port", action="store_true", help="cpu_baseline: skip the numpy-port number beside the reference's")
    ap.add_argument("--dump-ops", default="", help="write the per-op device times (JSON) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write rank 0's detections and indices of the last timed step to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config == "2x_fp32":
        from tools import bench_f32_config5
        return bench_f32_config5.main(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
