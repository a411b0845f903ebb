"""bench.py --config 2x_fp32: BASELINE config 5 -- CoDeNet2x (w2, stride-4 stem) fp32, COCO heads (80 classes), bilinear offsets,
512x512, batch 1024 sharded over 8 GPUs = 128 images per GPU (weak scaling; N = 1 runs one shard).

Our arm: codenet_b200.engine_f32.EngineF32 (fp32 NCHW kernels of csrc/f32_net.cu + the fused deformable module of
csrc/deform_f32.cu, forward + ctdet decode), the step replayed as a CUDA graph when capture succeeds.  Parity inside the run
(outside the timed region): the 256x256 image of tests/golden/codenet_float_2x_coco_256.npz through the same engine against the
reference's fp64 evaluation -- relative L2 error per head tensor <= max(1e-4, the reference's own fp32-vs-fp64 error recorded
in the fixture), the run fails otherwise.
Reference arm (--impl reference): the UNMODIFIED reference's float PoseShuffleNetV2 forward + ctdet_decode on the host cores
(oracle/ref_harness.py), batch 8.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
UNIT = "images/s"


def _cfg():
    from codenet_b200.arch import NetConfig
    return NetConfig(num_classes=80, w2=True)


def _state():
    from codenet_b200.synth import make_raw_state
    g = np.load(os.path.join(ROOT, "tests", "golden", "codenet_float_2x_coco_256.npz"))
    raw = make_raw_state(_cfg(), 0)
    for k in g.files:
        if k.startswith("bn/"):
            raw[k[3:]] = g[k]
    return raw, g


def check_parity(eng, g):
    import torch
    from codenet_b200.synth import make_images
    x = torch.from_numpy(make_images(2, 256, seed=2)[:1].copy()).cuda()
    dets, inds, v = eng.detect(x)
    torch.cuda.synchronize()
    worst = {}
    ok = True
    for name, key in (("hm", "hm_logit"), ("wh", "wh"), ("reg", "reg")):
        got, ref = v[name].cpu().numpy().astype(np.float64), g[key].astype(np.float64)
        l2 = float(np.sqrt(((got - ref) ** 2).sum() / (ref ** 2).sum()))
        tol = max(1e-4, float(g["ref_fp32_l2rel/" + name]))
        worst[name] = {"l2_rel": l2, "tol": tol}
        ok = ok and l2 <= tol
    return ok, worst


def run_ours(args, C):
    import torch
    import torch.distributed as dist
    from codenet_b200.engine_f32 import EngineF32
    from codenet_b200.synth import make_images
    import bench
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    raw, g = _state()
    gemm = os.environ.get("CODENET_F32_GEMM", "tf32x3")           # "fp32" = the SIMT kernel with fp64 block sums (strict accuracy mode)
    eng = EngineF32(_cfg(), raw, device=local, gemm=gemm)
    B, R = args.batch or C["batch"], C["res"]
    base = make_images(8, R, seed=100 + rank)
    host = torch.from_numpy(np.concatenate([base] * ((B + 7) // 8))[:B].copy()).pin_memory()
    x = host.cuda()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def maxr(v):
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    static = {"dets": torch.empty((B, 100, 6), dtype=torch.float32, device=x.device),
              "inds": torch.empty((B, 100), dtype=torch.int32, device=x.device)}
    out = (static["dets"], static["inds"])
    for _ in range(2):
        eng.detect(x, out)
    torch.cuda.synchronize()
    graph = None
    try:                                         # one graph per step: the ~115 launches of forward + decode replayed without host work
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            eng.detect(x, out)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            eng.detect(x, out)
        graph.replay()
        torch.cuda.synchronize()
    except Exception as e:                       # noqa: BLE001 -- fall back to eager launches, say so in the line
        graph = None
        static["graph_error"] = str(e)[:200]
        torch.cuda.synchronize()

    def step():
        if graph is not None:
            graph.replay()
        else:
            eng.detect(x, out)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = bench.ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = maxr(e0.elapsed_time(e1))
    value = world * B * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        bench.dump_outputs(args.dump_outputs, {"dets": static["dets"].cpu().numpy(), "inds": static["inds"].cpu().numpy()})
    # end to end: fp32 NCHW images from pinned host memory each step, detections back to the host
    dets_h = torch.empty((B, 100, 6), dtype=torch.float32).pin_memory()
    n_e2e = max(4, min(args.steps, 10))

    # pipelined submit: the H2D copy of step n + 1 (copy stream, its own staging buffer) runs under the compute of step n; every
    # step's detections are copied back to pinned memory.  Two staging buffers, events in both directions.
    copy_stream = torch.cuda.Stream()
    xs = [torch.empty_like(x) for _ in range(2)]
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream()

    def submit_copy(j):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[j])
            xs[j].copy_(host, non_blocking=True)
            h2d_done[j].record(copy_stream)

    def e2e_run(n):
        for j in range(2):
            consumed[j].record(main)
        submit_copy(0)
        for i in range(n):
            j = i & 1
            if i + 1 < n:
                submit_copy(j ^ 1)
            main.wait_event(h2d_done[j])
            x.copy_(xs[j], non_blocking=True)                     # the graph reads the fixed tensor x
            consumed[j].record(main)
            step()
            dets_h.copy_(static["dets"], non_blocking=True)
        torch.cuda.synchronize()

    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e_run(n_e2e)
    e2e = world * B * n_e2e / maxr(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    # launches per step and the 1x1-conv family's rate: one eager, event-traced forward outside the timed region
    torch.cuda.synchronize()
    eng.launches = 0
    eng.trace = []
    eng.detect(x, out)
    torch.cuda.synchronize()
    trace, eng.trace = eng.trace, None
    launches = eng.launches
    pw_ms = sum(e0.elapsed_time(e1) for _, _, e0, e1 in trace)
    pw_flops = sum(f for _, f, _, _ in trace)
    roofline = None
    if gemm == "tf32x3" and pw_ms > 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:                            # noqa: BLE001
            pass
        bf16 = float(peaks.get("bf16_tflops_sustained", 0) or 0)
        peak, src = (bf16 / 2.0, "MEASURED_PEAKS.json bf16_tflops_sustained / 2 (kind::tf32 runs at half the bf16 rate)") if bf16 else \
                    (1125.0, "fallback: nominal dense tf32 (B200_PROFILING.md: 2250 bf16 / 2)")
        ach = pw_flops / (pw_ms * 1e-3) / 1e12
        roofline = {"kernel": "pw_tf32x3_kernel (%d launches)" % len(trace), "bound": "tensor", "achieved": round(ach, 1), "peak": round(peak, 1),
                    "unit": "TFLOP/s", "frac": round(ach / peak, 4), "traffic": None, "peak_source": src, "ms_per_step": round(pw_ms, 3),
                    "share_of_step": round(pw_ms / (ms / args.steps), 3),
                    "note": "achieved = algorithmic fp32 flops (2*C*Co*pixels, unpadded); every fp32 product costs three tf32 MMAs, so the "
                            "ceiling of frac is 1/3; timed per launch with CUDA events in an eager pass"}
    cpu_baseline = None
    if rank == 0 and world == 1 and not getattr(args, "no_cpu", False):
        try:                                         # bounded sample (2 timed steps of batch 8) of the unmodified reference on the host cores
            cpu_baseline, _, _ = time_reference(C, raw, _cfg(), 2, 1, budget_s=60.0)
        except Exception as e:                       # noqa: BLE001 -- the reference tree is not on this box
            cpu_baseline = {"value": None, "unit": UNIT, "kind": "reference", "unavailable": str(e)[:160]}
    ok, worst = check_parity(eng, g)
    t = torch.tensor([0 if ok else 1], device="cuda")
    if world > 1:
        dist.all_reduce(t)
        dist.destroy_process_group()
    ok_all = int(t.item()) == 0
    if rank == 0:
        line = {"metric": C["metric"], "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "codenet_b200",
                "config": {"workload": C["workload"] % B, "name": "2x_fp32", "batch_per_gpu": B, "offset_mode": "bilinear",
                           "arithmetic": ("fp32; 1x1 convs on tcgen05 kind::tf32 with a 3-way split (hi*hi + hi*lo + lo*hi), 16-channel chunk sums added in fp32 registers"
                                          if gemm == "tf32x3" else "fp32 (1x1 convs: SIMT fp32 with two-level fp32 -> fp64 accumulation)"), "gemm": gemm,
                           "parallelism": "batch-sharded, no collective",
                           "l2": "inputs larger than L2 (%.0f MB fp32 images per step)" % (B * 3 * R * R * 4 / 1e6),
                           "launch": "CUDA graph" if graph is not None else "eager (%s)" % static.get("graph_error", "")},
                "parity_checked": bool(ok_all), "parity": worst,
                "e2e": {"value": round(e2e, 1), "unit": UNIT, "h2d_bytes_per_step": int(B * 3 * R * R * 4),
                        "d2h_bytes_per_step": int(B * 100 * 6 * 4), "steps": n_e2e,
                        "api": "EngineF32.detect on images copied from pinned host memory every step (copy of step n+1 under the compute of step n)"},
                "gpu_launches": launches * args.steps, "launches_per_step": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline}
        print(json.dumps(line))
    if not ok_all:
        sys.stderr.write("bench.py --config 2x_fp32: PARITY FAILURE %s\n" % worst)
        sys.exit(3)


def time_reference(C, raw, cfg, steps, warmup, budget_s=150.0):
    """The UNMODIFIED reference's float forward + sigmoid + ctdet_decode on the host cores (oracle/ref_harness.py), batch 8:
    (cpu_baseline dict, median seconds per step, timed steps)."""
    import torch
    from oracle import ref_harness as H
    from codenet_b200.synth import make_images
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    R_ = H.load_reference()
    m = H.build_reference_model({k: torch.from_numpy(np.asarray(v)) for k, v in raw.items()}, dict(cfg.head_list()), cfg.w2, cfg.maxpool,
                                dtype=torch.float32)
    m.eval()
    x = torch.from_numpy(make_images(8, C["res"], seed=100))

    def step():
        with torch.no_grad():
            o = m(x)[-1]
            return R_.decode.ctdet_decode(o["hm"].sigmoid_(), o["wh"], reg=o["reg"], K=100)

    for _ in range(max(1, min(warmup, 2))):
        step()
    times = []
    t_all = time.perf_counter()
    for i in range(max(steps, 2)):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if i >= 1 and time.perf_counter() - t_all > budget_s:
            break
    med = float(np.median(times))
    cpu = {"value": round(8 / med, 3), "unit": UNIT, "cores": threads, "kind": "reference",
           "sample": "%d timed steps (median) of the UNMODIFIED reference's float PoseShuffleNetV2(w2) forward + sigmoid + ctdet_decode on "
                     "a batch of 8 512x512 images, fp32, torch.set_num_threads(%d), torchvision CPU deform_conv2d in place of the "
                     "CUDA-only op" % (len(times), threads)}
    return cpu, med, len(times)


def run_reference(args, C):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    raw, g = _state()
    cpu, med, n = time_reference(C, raw, _cfg(), args.steps, args.warmup)
    B = args.batch or C["batch"]
    print(json.dumps({"metric": C["metric"], "value": cpu["value"], "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
                      "steps": n, "warmup": args.warmup, "ms_per_step": round(med * 1e3, 3), "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
                      "config": {"workload": C["workload"] % B, "name": "2x_fp32", "batch_per_gpu": B, "offset_mode": "bilinear"},
                      "cpu_baseline": cpu,
                      "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main(args):
    import bench
    C = bench.configs()["2x_fp32"]
    if args.impl == "reference":
        run_reference(args, C)
    else:
        run_ours(args, C)
