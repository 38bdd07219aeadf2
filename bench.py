#!/usr/bin/env python
"""bench.py -- ICAFusion hot path on B200: 640x512 RGB+IR pairs/s end to end (+ roofline of the dominant kernel).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`):
    yolov5l_b16  (default)  configs[2]: yolov5l_ICAFusion, 640x512 synthetic RGB+IR, batch 16 per GPU, inference -- the largest
                            single-GPU configuration; the headline line at every N
    yolov5s_b1              configs[1]: yolov5s_ICAFusion, batch 1 per GPU (latency-bound regime; reported under `secondary` at N=1)
A "step" = one forward of the whole two-stream detector (stage images -> two CSPDarknet streams -> 3 DMFF blocks ->
PANet head -> Detect decode) over one batch.  N>1: one process per GPU (torchrun), the batch dimension is sharded --
every rank runs its own pairs, there is no collective on the inference path ("weak" scaling).

`value`  : pairs/s with inputs resident in HBM, CUDA-graph replay, timed with CUDA events per step, L2 flushed
           between steps, max over ranks.
`e2e`    : pairs/s through the reference-facing call with HOST (pinned, uint8) frames: H2D + forward + D2H of the
           decoded predictions inside the timed region.
`roofline`: the tcgen05 implicit-GEMM conv kernels (every Conv / Linear / Detect GEMM of a step): algorithmic FLOPs of those
           launches / the time they take INSIDE the timed step = ms_per_step x their share of the step's kernel time (the
           share from a CUDA-event pass over one step on the launching stream; profiles/ holds the ncu launch list of the
           same step for comparison), against the SUSTAINED tensor peak of MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the oracle (fp32 PyTorch-CPU restatement of the reference forward; the reference
           itself is Python and cannot travel to the GPU box) timed on this host's cores at a FIXED intra-op thread count
           (32, or fewer if the host has fewer usable cores) so the two arms share one denominator.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# NCCL's version / debug banner goes to stdout by default; stdout of this script carries exactly one JSON line.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
os.environ.setdefault("NCCL_DEBUG", "WARN")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    "yolov5s_b1": dict(size="s", batch=1, H=512, W=640, desc="yolov5s_ICAFusion 640x512 synthetic RGB+IR, batch 1, inference"),
    "yolov5l_b16": dict(size="l", batch=16, H=512, W=640, desc="yolov5l_ICAFusion 640x512 synthetic RGB+IR, batch 16, inference"),
}
METRIC = "640x512 RGB+IR pairs/sec end-to-end"
DUMP_LIMIT = 64 << 20       # bytes written by --dump-outputs


def _to_host(arrays):
    """name -> tensor  =>  name -> float32 numpy copy (taken now: graph outputs are overwritten by the next replay)."""
    return {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}


def _dump(outdir, host):
    """--dump-outputs: DIR/<name>.npy per array."""
    import numpy as np
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(outdir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(outdir, k + ".npy"), a)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"tensor": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "tensor_burst": p["bf16_tflops"], "hbm": p["hbm_gbs"],
                "src": "measured (MEASURED_PEAKS.json: bf16_tflops_sustained -- the kernels run inside a multi-ms step; hbm_gbs)"}
    except Exception:  # noqa: BLE001
        return {"tensor": 1590.0, "tensor_burst": 1590.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def _build_oracle_inputs(wl, seed=0):
    import torch
    from icafusion_b200.cfg import load_cfg
    from oracle import icaf_oracle as O
    from oracle import synth
    cfg = load_cfg(f"yolov5{wl['size']}_Transfusion_kaist")
    sd = O.fold_bn(synth.synth_state_dict(synth.model_param_shapes(cfg), seed))
    return cfg, sd


def _usable_cpus() -> int:
    """Cores this process may really use: affinity mask, capped by the cgroup CPU quota if there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:  # noqa: BLE001
        pass
    return n


CPU_THREADS = 32        # fixed intra-op thread count of the CPU arm: the fastest setting round 1's sweeps found on the GPU box (PyTorch's
                        # pool stops scaling on these convolutions beyond it: 47 s/pair at 128 threads); both arms use it -> one denominator


def cpu_reference_throughput(wl, budget_s=20.0, max_pairs=64, warm=1):
    """The reference's CPU path (oracle port: same torch CPU ops, fp32, fused BN) on the host cores; bounded sample:
    batch-1 forwards of the workload's model until `max_pairs` pairs or `budget_s` seconds, median forward time."""
    import torch
    from oracle import icaf_oracle as O
    from oracle import synth
    cfg, sd = _build_oracle_inputs(wl)
    B = 1                                   # the CPU sample runs batch 1 (latency-optimal on CPU)
    rgb, ir = synth.synth_images(B, wl["H"], wl["W"], 0)
    usable = _usable_cpus()
    nt = max(1, min(CPU_THREADS, usable))
    torch.set_num_threads(nt)
    with torch.no_grad():
        for _ in range(max(1, warm)):
            O.model_forward(sd, cfg, rgb, ir)
        t0, n, times = time.perf_counter(), 0, []
        while n < max_pairs and (time.perf_counter() - t0) < budget_s:
            t = time.perf_counter()
            O.model_forward(sd, cfg, rgb, ir)
            times.append(time.perf_counter() - t)
            n += B
    per = sorted(times)[len(times) // 2]
    return {"value": round(B / per, 3), "unit": "pairs/s", "cores": nt, "kind": "port",
            "sample": f"{n} pairs of {wl['desc'].split(',')[0]} at batch 1, fp32, median of {len(times)} forwards "
                      f"({sum(times):.1f} s of CPU work) on {nt} intra-op threads (fixed; {usable} usable cores); "
                      "oracle/icaf_oracle.py (PyTorch-CPU restatement of the reference forward)",
            "cpu_model": _cpu_model(), "host_cpus": os.cpu_count()}


def _cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:  # noqa: BLE001
        pass
    return "unknown"


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    # one "step" of this arm = one pair of the workload (a bounded sample of its batch); W warm-up pairs, K timed pairs
    cb = cpu_reference_throughput(wl, budget_s=float("inf"), max_pairs=steps, warm=max(1, min(args.warmup, 3)))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": round(1000.0 / cb["value"], 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "note": "reference forward restated with the same PyTorch CPU ops (oracle port); "
                                                       "the Python reference cannot travel to the GPU box"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def _measure(args, wl, K, Wm, dev, world, rank, local, primary=True):
    """Build the detector for workload `wl` on `dev`, time K graph-replayed steps (device-resident inputs) and, for the
    primary workload, K end-to-end steps from pinned host frames; profile the kernels of one step.  Returns a dict on rank 0."""
    import torch
    import torch.distributed as dist
    from icafusion_b200 import Model, ops, synth
    from icafusion_b200.engine import GraphedDetector
    from icafusion_b200.synth import load_synth

    B, H, W = wl["batch"], wl["H"], wl["W"]
    model = Model(f"yolov5{wl['size']}_Transfusion_kaist").eval()
    load_synth(model, 0)
    model = model.fuse().half().to(dev)
    eng = GraphedDetector(model, B, H, W, in_dtype=torch.uint8, device=dev)
    rgb_u8, ir_u8 = [(t * 255).to(torch.uint8) for t in synth.synth_images(B, H, W, rank)]
    rgb_pin, ir_pin = rgb_u8.pin_memory(), ir_u8.pin_memory()
    eng.rgb.copy_(rgb_u8)
    eng.ir.copy_(ir_u8)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing: per-step CUDA events, L2 flushed between steps -----------------
    for _ in range(Wm):
        eng.replay()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    t_wall = time.perf_counter()
    for s, e in ev:
        flush.zero_()
        s.record()
        eng.replay()
        e.record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)
    if primary and args.dump_outputs and rank == 0:       # what the last timed replay returned: (z, logits, [x0, x1, x2])
        _dump(args.dump_outputs, _to_host({"z": eng.z, "logits": eng.logits, **{f"x{i}": x for i, x in enumerate(eng.xs)}}))
    # ---------------- end-to-end timing through the public streaming call with host frames ----------------------
    # PipelinedDetector.infer_stream: per frame H2D (pinned uint8) -> forward -> D2H of the decoded predictions; the copy
    # of frame i+1 overlaps the forward of frame i (depth-2), the host blocks on the oldest frame in flight.
    e2e_ms = e2e_sync_ms = 0.0
    if primary:
        from icafusion_b200.engine import PipelinedDetector
        pipe = PipelinedDetector(model, B, H, W, torch.uint8, dev, depth=2)
        for _ in pipe.infer_stream([(rgb_pin, ir_pin)] * Wm):
            pass
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.compute)
        for zh in pipe.infer_stream((rgb_pin, ir_pin) for _ in range(K)):
            pass
        e1.record(pipe.compute)
        barrier()
        e2e_ms = e0.elapsed_time(e1)
        # for reference: the strictly sequential call (copy, forward, copy back, sync; nothing overlapped)
        for _ in range(Wm):
            eng.infer_to_host(rgb_pin, ir_pin)
        barrier()
        e0.record()
        for _ in range(K):
            eng.infer_to_host(rgb_pin, ir_pin)
        e1.record()
        barrier()
        e2e_sync_ms = e0.elapsed_time(e1)
        del pipe
    # ---------------- the detect_twostream.py loop body: raw BGR frames -> letterbox -> forward -> NMS -> detections -------------
    # (reported separately: the headline metric stops at the Detect output, like test.py:127-129's timer)
    det_ms, det_info = 0.0, None
    if primary:
        try:
            eng_d = GraphedDetector(model, B, H, W, in_dtype=torch.uint8, device=dev, nms=dict(conf_thres=0.25, iou_thres=0.45),
                                    frame_hw=(H, W))
            fr_rgb = rgb_u8.permute(0, 2, 3, 1).flip(3).contiguous().pin_memory()        # (B, H, W, 3) BGR, as cv2.imread decodes
            fr_ir = ir_u8.permute(0, 2, 3, 1).flip(3).contiguous().pin_memory()
            for _ in range(Wm):
                eng_d.infer_frames(fr_rgb, fr_ir)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                eng_d.infer_frames(fr_rgb, fr_ir)
            e1.record()
            barrier()
            det_ms = e0.elapsed_time(e1)
            det_info = {"h2d_bytes_per_step": int(fr_rgb.numel() + fr_ir.numel()),
                        "d2h_bytes_per_step": int(eng_d.det.numel() * 4 + eng_d.count.numel() * 4),
                        "launches_per_step": eng_d.launches_per_step,
                        "api": "GraphedDetector(frame_hw=..., nms=...).infer_frames(raw uint8 BGR frames) -> (B, 300, 6) detections + counts "
                               "on the host: H2D, device letterbox, forward, device NMS (conf 0.25, iou 0.45), D2H; sequential per step"}
            del eng_d
        except Exception as e:  # noqa: BLE001  (an extra leg must never cost the headline line)
            det_info = {"error": f"{type(e).__name__}: {e}"}
    clocks = sampler.stop()
    t = torch.tensor([dev_ms, e2e_ms, e2e_sync_ms, det_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, e2e_sync_ms, det_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    if rank != 0:
        return None

    # ---------------- roofline of the dominant kernel: event-bracketed eager pass --------------------------------
    # The launches of the profiled step are queued behind a ~30 ms spin kernel so that they execute back to back (an
    # event pair then sees kernel time + inter-kernel gap, not the Python launch latency: queueing a yolov5l step takes
    # the host ~10 ms, longer than the step itself).  Three passes; every launch keeps its fastest time, so a host hiccup
    # in one pass cannot leak into the figure.
    with torch.no_grad():
        model(eng.rgb, eng.ir)
        torch.cuda.synchronize()
        reps = 3
        model.__dict__["_icaf_concurrent"] = False          # one stream: every launch is timed against its predecessor
        with ops.profile() as prof:
            for _ in range(reps):
                flush.zero_()
                torch.cuda._sleep(int(6e7))
                prof.mark()
                model(eng.rgb, eng.ir)
                torch.cuda.synchronize()
        model.__dict__["_icaf_concurrent"] = True
    allp = prof.per_launch()
    per = len(allp) // reps
    pl = [min((allp[r * per + i] for r in range(reps)), key=lambda t: t[2]) for i in range(per)]    # fastest of the passes
    summ = {}
    for name, tag, ms, fl, by in pl:
        d = summ.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        d["launches"] += reps; d["ms"] += ms * reps; d["flops"] += fl * reps; d["bytes"] += by * reps
    if primary and args.layer_profile:           # per-launch table of the profiled step (geometry, us, TFLOP/s, GB/s)
        with open(args.layer_profile, "w") as f:
            f.write("kernel,geometry,us,tflops,gbs\n")
            for name, tag, ms, fl, by in pl:
                f.write(f"{name},{tag},{ms * 1e3:.2f},{fl / (ms * 1e-3) / 1e12 if ms > 0 else 0:.2f},{by / (ms * 1e-3) / 1e9 if ms > 0 else 0:.1f}\n")
    conv = summ.get("icaf_conv2d_fwd", {"ms": 1.0, "flops": 0.0, "launches": 1, "bytes": 0.0})
    traffic, traffic_src = None, None      # DRAM bytes per conv launch from the committed ncu capture of the same step
    try:
        import glob
        cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
        wl_key = [k for k, v in WORKLOADS.items() if v is wl][0]
        tj = json.load(open(cands[-1]))[wl_key]
        traffic = round(tj["conv_dram_bytes_per_launch"] * (B / wl["batch"]))
        traffic_src = os.path.relpath(cands[-1], ROOT) + " (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean over the conv launches of one step)"
    except Exception:  # noqa: BLE001
        pass
    pk = _peaks()
    # The conv kernels' time INSIDE the timed step: the graph-replayed step time x their share of the step's kernel time
    # (event pass: every launch bracketed on its stream; the share cancels the constant per-launch event overhead, which
    # the absolute event times carry).  By construction launches x avg_launch_us <= ms_per_step.
    total_ms = sum(v["ms"] for v in summ.values())
    share = conv["ms"] / total_ms if total_ms > 0 else 0.0
    step_ms = dev_ms / K
    conv_launches = conv["launches"] // reps
    conv_ms_in_step = step_ms * share
    conv_flops_step = conv["flops"] / reps
    ach = conv_flops_step / (conv_ms_in_step * 1e-3) / 1e12 if conv_ms_in_step > 0 else 0.0
    roofline = {"kernel": "icaf_conv2d_fwd = conv_gemm_{tc,persist,pair}_kernel (every Conv/Linear/Detect GEMM of a step)", "bound": "tensor",
                "achieved": round(ach, 3), "peak": pk["tensor"], "unit": "TFLOP/s", "frac": round(ach / pk["tensor"], 5),
                "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_flops_per_launch": round(conv_flops_step / max(1, conv_launches)),
                "algorithmic_bytes_per_launch": round(conv.get("bytes", 0.0) / max(1, conv["launches"])),
                "peak_source": pk["src"], "frac_of_burst_peak": round(ach / pk["tensor_burst"], 5),
                "launches_per_step": conv_launches,
                "avg_launch_us": round(1e3 * conv_ms_in_step / max(1, conv_launches), 2),
                "share_of_step_kernel_time": round(share, 4),
                "time_basis": "ms_per_step (CUDA-graph replay, timed region) x share_of_step_kernel_time (CUDA-event pass over the same step, "
                              "one stream); launches_per_step x avg_launch_us <= ms_per_step",
                "event_pass_us_per_launch": round(1e3 * conv["ms"] / max(1, conv["launches"]), 2),
                "per_kernel_ms_per_step_event_pass": {k: round(v["ms"] / reps, 4) for k, v in sorted(summ.items())}}
    flops_pair = sum(v["flops"] for v in summ.values()) / reps / B     # algorithmic 2*M*N*K (+ 8*N^2*C attention) of one step
    pairs = world * B * K
    out = {"value": round(pairs / (dev_ms * 1e-3), 2), "ms_per_step": round(dev_ms / K, 4), "steps": K, "warmup": Wm,
           "config": {"workload": wl["desc"], "pairs_per_gpu_per_step": B, "gflop_per_pair": round(flops_pair / 1e9, 2),
                      "weights": "seeded synthetic (icafusion_b200/synth.py), BN folded (Model.fuse())",
                      "l2": "flushed between timed steps (256 MiB memset outside the event pair)",
                      "execution": "CUDA graph replay of libicaf_b200 kernels (programmatic dependent launch)",
                      "parallelism": f"dp{world} (batch-sharded replicas, no collective)"},
           "gpu_launches": eng.launches_per_step * K,
           "model_tflops": round(flops_pair * pairs / (dev_ms * 1e-3) / 1e12, 3),
           "wall_s_timed_region": round(t_wall, 4), "clocks": clocks, "roofline": roofline}
    # whole-step bound (SURVEY 8d): sum over launches of max(F_i / tensor peak, bytes_i / HBM peak) vs the timed step
    bound_ms = sum(max(fl / (pk["tensor"] * 1e12), by / (pk["hbm"] * 1e9)) for _, _, _, fl, by in pl) * 1e3
    out["step_roofline"] = {"bound_ms": round(bound_ms, 4), "achieved_ms": round(step_ms, 4), "frac": round(bound_ms / step_ms, 4),
                            "note": "sum over the step's launches of max(flops/tensor_peak, algorithmic_bytes/hbm_peak), no cross-layer fusion assumed"}
    if primary:
        out["e2e"] = {"value": round(pairs / (e2e_ms * 1e-3), 2), "unit": "pairs/s",
                      "h2d_bytes_per_step": int(rgb_pin.numel() + ir_pin.numel()), "d2h_bytes_per_step": int(eng.z.numel() * 2),
                      "ms_per_step": round(e2e_ms / K, 4),
                      "api": "PipelinedDetector.infer_stream(frames of pinned uint8 (rgb, ir)) -> decoded predictions on the host",
                      "sequential_call_value": round(pairs / (e2e_sync_ms * 1e-3), 2),
                      "sequential_call_api": "GraphedDetector.infer_to_host (no copy/compute overlap)"}
        if det_info is not None:
            if det_ms > 0:
                det_info = {"value": round(pairs / (det_ms * 1e-3), 2), "unit": "pairs/s", "ms_per_step": round(det_ms / K, 4), **det_info}
            out["e2e_detect"] = det_info
    del eng, model, flush
    torch.cuda.empty_cache()
    return out


def _measure_train(args, wl, K, Wm, dev, world, rank, local):
    """One training step of train.py:334-349 per "step" (BASELINE configs[3]: yolov5l, 16 pairs per GPU, DDP over the GPUs of the
    box): train-mode forward (BatchNorm batch statistics, dropout 0.1, nearest DMFF tail), ComputeLoss, scaled backward with DDP's
    bucketed NCCL all-reduce of the gradients, SGD step.  Times K steps with device-resident batches, K steps end to end from
    pinned host batches, and (N > 1) K steps under no_sync() to name the all-reduce's exposed share.  Returns a dict on rank 0."""
    import torch
    import torch.distributed as dist
    from icafusion_b200 import Model, autograd, ops, synth
    from icafusion_b200.synth import load_synth
    from icafusion_b200.trainer import GraphedTrainStep, TrainStep

    B, H, W = wl["batch"], wl["H"], wl["W"]
    autograd.manual_seed(1000 + rank)
    model = Model(f"yolov5{wl['size']}_Transfusion_kaist")
    load_synth(model, 0)
    model = model.to(dev).train()
    side = torch.cuda.Stream(dev)                     # DDP is constructed on a side stream (torch's CUDA-graph + DDP recipe)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        ts = TrainStep(model, None, total_batch_size=B * world, world_size=world, local_rank=local, imgsz=max(H, W))
    torch.cuda.current_stream(dev).wait_stream(side)
    n_param = sum(p.numel() for p in model.parameters() if p.requires_grad)
    rgb_u8, ir_u8 = [(t * 255).to(torch.uint8) for t in synth.synth_images(B, H, W, rank)]
    rgb_pin, ir_pin = rgb_u8.pin_memory(), ir_u8.pin_memory()
    g = torch.Generator().manual_seed(rank)
    nt = 4 * B                                                    # KAIST-like: a few pedestrians per pair
    tg = torch.zeros(nt, 6)
    tg[:, 0] = torch.arange(nt) % B
    tg[:, 2:4] = 0.1 + 0.8 * torch.rand(nt, 2, generator=g)
    tg[:, 4:6] = 0.03 + 0.2 * torch.rand(nt, 2, generator=g)
    tg_pin = tg.pin_memory()
    rgb_d, ir_d, tg_d = rgb_u8.to(dev), ir_u8.to(dev), tg.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        """(ms of n calls, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    dump = args.mode == "train" and args.dump_outputs and rank == 0
    if dump:
        n_all = sum(p.numel() for p in model.parameters())
        pick = torch.randint(n_all, (1 << 20,), generator=torch.Generator().manual_seed(0)).to(dev)

    def outputs(step_out):
        """The step's (loss, loss_items) and a fixed sample of the parameters it updated, on the host."""
        loss, items = step_out
        params = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
        return _to_host({"loss": loss.reshape(1), "loss_items": items, "params_sample": params[pick]})

    def resident():
        return ts(rgb_d, ir_d, tg_d)

    def e2e():
        loss, _ = ts(rgb_pin.to(dev, non_blocking=True), ir_pin.to(dev, non_blocking=True), tg_pin.to(dev, non_blocking=True))
        return float(loss)                                        # D2H of the step's loss

    for _ in range(Wm):
        resident()
    n0 = ops.launch_count()
    eager_ms, last = timed(resident, K)
    launches = ops.launch_count() - n0
    dumped = outputs(last) if dump else None
    # per-kernel split of one step (event pass on one stream)
    summ = {}
    if rank == 0:
        torch.cuda.synchronize()
    prev_streams = os.environ.get("ICAF_TRAIN_STREAMS")
    os.environ["ICAF_TRAIN_STREAMS"] = "0"   # the event chain attributes a launch to the gap since the previous one: one stream only
    try:
        with ops.profile() as prof:
            torch.cuda._sleep(int(4e8))   # ~0.2 s spin: the step's launches queue up behind it and then run back to back
            prof.mark()
            ts(rgb_d, ir_d, tg_d)
            torch.cuda.synchronize()
    finally:
        if prev_streams is None:
            os.environ.pop("ICAF_TRAIN_STREAMS", None)
        else:
            os.environ["ICAF_TRAIN_STREAMS"] = prev_streams
    for name, v in prof.summary().items():
        summ[name] = {"launches": v["launches"], "ms": round(v["ms"], 3), "tflops": round(v["flops"] / max(v["ms"], 1e-6) / 1e9, 1)}
    # the same step with forward + loss + backward (+ DDP all-reduce) replayed from one CUDA graph
    gts, graph_note = None, None
    if os.environ.get("ICAF_TRAIN_GRAPH", "1") != "0":
        try:
            gts = GraphedTrainStep(ts, B, H, W, nt, dev)
        except Exception as e:  # noqa: BLE001
            graph_note = f"CUDA-graph capture of the training step failed, eager timings reported: {type(e).__name__}: {e}"
            gts = None
    if gts is not None:
        def resident():                               # noqa: F811
            return gts(rgb_d, ir_d, tg_d)

        def e2e():                                    # noqa: F811
            loss, _ = gts(rgb_pin, ir_pin, tg_pin)    # H2D copies into the graph's static batch, replay, optimiser step
            return float(loss)
        for _ in range(2):
            resident()
        res_ms, last = timed(resident, K)
        dumped = outputs(last) if dump else None
    else:
        res_ms = eager_ms
    if dump:
        _dump(args.dump_outputs, dumped)
    e2e()
    e2e_ms, _ = timed(e2e, K)
    if gts is not None:
        gts.close()
    in_sync = None
    if world > 1:      # every rank must hold the same parameters after the synchronised steps (the all-reduce really ran, also inside the graph)
        chk = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum().reshape(1)
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        in_sync = bool(all(float(c) == float(allc[0]) for c in allc))
    nosync_ms = 0.0
    if world > 1:                                                 # last: ranks drift apart without the all-reduce
        def local_only():
            with ts.model.no_sync():
                return ts(rgb_d, ir_d, tg_d)
        local_only()
        nosync_ms, _ = timed(local_only, K)
    t = torch.tensor([res_ms, e2e_ms, nosync_ms, eager_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res_ms, e2e_ms, nosync_ms, eager_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    scale = float(ts.scaler.get_scale())
    del ts, model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    pairs = world * B * K
    out = {"metric": "training pairs/sec (train.py step: forward + loss + backward + gradient all-reduce + SGD)", "value": round(pairs / (res_ms * 1e-3), 2),
           "unit": "pairs/s", "ms_per_step": round(res_ms / K, 3), "steps": K, "warmup": Wm, "global_batch": B * world,
           "config": {"workload": f"yolov5{wl['size']}_Transfusion_kaist train(), {B} pairs of {W}x{H} per GPU, dropout 0.1, SGD nesterov + GradScaler",
                      "parallelism": f"ddp{world}" if world > 1 else "single GPU",
                      "trainable_parameters": n_param, "allreduce_bytes_fp32": 4 * n_param if world > 1 else 0},
           "e2e": {"value": round(pairs / (e2e_ms * 1e-3), 2), "unit": "pairs/s", "ms_per_step": round(e2e_ms / K, 3),
                   "h2d_bytes_per_step": int(rgb_pin.numel() + ir_pin.numel() + tg_pin.numel() * 4), "d2h_bytes_per_step": 4,
                   "api": "TrainStep(model)(rgb, ir, targets) from pinned host batches; the loss is read back every step"},
           "gpu_launches": launches, "grad_scale_after": scale, "peak_mem_gib": round(mem, 2),
           "execution": ("CUDA graph replay of forward + loss + backward" + (" + DDP all-reduce" if world > 1 else "") + "; optimiser step eager")
           if gts is not None else "eager launches",
           "eager_ms_per_step": round(eager_ms / K, 3),
           "per_kernel_event_pass": summ}
    if graph_note:
        out["note"] = graph_note
    if world > 1:
        out["parameters_identical_across_ranks"] = in_sync
        out["allreduce"] = {"eager_ms_per_step_with": round(eager_ms / K, 3), "eager_ms_per_step_without": round(nosync_ms / K, 3),
                            "exposed_share_of_eager_step": round(max(0.0, 1.0 - nosync_ms / eager_ms), 4),
                            "note": "eager step under DDP.no_sync() (no gradient all-reduce) vs the synchronised eager step; DDP overlaps its 25 MB "
                                    "buckets with the remaining backward kernels, the difference is what stays exposed"}
    return out


def dmff_block_metrics(dev):
    """Second half of the BASELINE metric: DMFF-block GFLOP/s vs roofline on BASELINE configs[0]'s block
    (C=256, 32x40 map, batch 1, fp16), as shipped (pooled to 16x16 tokens) and un-pooled (1280 tokens)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from dmff_sweep import dmff_flops, peaks, time_block
    tf_peak, hbm = peaks()
    out = {}
    for name, (va, ha) in (("pooled_16x16", (16, 16)), ("unpooled_32x40", (32, 40))):
        C, H, W, B = 256, 32, 40, 1
        ms = time_block(C, H, W, va, ha, 1, B, dev)
        F = dmff_flops(B, C, H, W, va * ha, 1)
        by = 2.0 * (3 * B * C * H * W + 2 * va * ha * C + 26 * C * C)
        t_bound = max(F / (tf_peak * 1e12), by / (hbm * 1e9))
        out[name] = {"ms": round(ms, 4), "gflops": round(F / ms / 1e6, 1), "algorithmic_gflop": round(F / 1e9, 3),
                     "frac_of_roofline": round(t_bound / (ms * 1e-3), 4),
                     "bound": "tensor" if F / (tf_peak * 1e12) > by / (hbm * 1e9) else "hbm"}
    out["note"] = ("TransformerFusionBlock(256) on 1x256x32x40 RGB+IR maps, CUDA-graph replay, L2 flushed; roofline time = "
                   "max(F/peak_tensor, ideal_bytes/peak_hbm); latency-bound at batch 1 (8 launches per block: pooling, 5 per loop, tail, 1x1 conv)")
    return out


def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import datetime
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")      # required to capture DDP's all-reduce in a CUDA graph
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"), timeout=datetime.timedelta(seconds=300))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    K, Wm = args.steps, max(3, args.warmup)
    if args.mode == "train":
        tr = _measure_train(args, wl, K, max(4, Wm // 2), dev, world, rank, local)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if rank != 0:
            return
        per = tr.pop("per_kernel_event_pass")
        line = {"metric": "640x512 RGB+IR training pairs/sec (train.py step)", "value": tr["value"], "unit": "pairs/s", "n_gpus": world, "steps": tr["steps"],
                "warmup": tr["warmup"], "ms_per_step": tr["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
                "data": "synthetic", "config": tr["config"], "e2e": tr["e2e"], "gpu_launches": tr["gpu_launches"],
                **{k: v for k, v in tr.items() if k in ("execution", "eager_ms_per_step", "allreduce", "parameters_identical_across_ranks", "grad_scale_after",
                                                        "peak_mem_gib", "note")},
                "per_kernel_event_pass": per}
        print(json.dumps(line))
        return
    m = _measure(args, wl, K, Wm, dev, world, rank, local, primary=True)      # the same workload at every N
    tr, tr_err = None, None
    if args.train != "off":
        try:      # BASELINE configs[3]: the training step, the one place the data-parallel path has an exchange (DDP all-reduce)
            tr = _measure_train(args, wl, max(3, min(K, args.train_steps)), 4, dev, world, rank, local)
        except Exception as e:  # noqa: BLE001  (an extra leg must never cost the headline line)
            tr_err = f"train leg failed: {type(e).__name__}: {e}"
    if world > 1:
        # every rank is done with the GPU work once this barrier returns; rank 0 alone goes on to the CPU baseline and the
        # single-GPU extras, so no rank spins in NCCL while it does
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    notes = [tr_err] if tr_err else []
    sec_name = args.secondary
    if sec_name == "auto":
        sec_name = "yolov5s_b1" if (args.workload == "yolov5l_b16" and world == 1) else "none"
    sec = dm = cb = None
    if sec_name != "none" and world == 1:
        try:
            sec = _measure(args, WORKLOADS[sec_name], 200 if WORKLOADS[sec_name]["batch"] == 1 else max(5, min(K, 20)), 5, dev, 1, 0, local,
                           primary=False)
        except Exception as e:  # noqa: BLE001  (an extra leg must never cost the headline line)
            notes.append(f"secondary workload {sec_name} failed: {type(e).__name__}: {e}")
    if world == 1:
        try:
            dm = dmff_block_metrics(dev)
        except Exception as e:  # noqa: BLE001
            notes.append(f"dmff_block leg failed: {type(e).__name__}: {e}")
    try:
        cb = cpu_reference_throughput(wl, budget_s=20.0)
    except Exception as e:  # noqa: BLE001
        notes.append(f"cpu_baseline leg failed: {type(e).__name__}: {e}")
    line = {"metric": METRIC, "value": m["value"], "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic", "config": m["config"], "e2e": m["e2e"], "gpu_launches": m["gpu_launches"],
            "model_tflops": m["model_tflops"], "wall_s_timed_region": m["wall_s_timed_region"], "clocks": m["clocks"],
            "roofline": m["roofline"], "step_roofline": m["step_roofline"], "cpu_baseline": cb}
    if "e2e_detect" in m:
        line["e2e_detect"] = m["e2e_detect"]
    if tr is not None:
        line["train"] = tr
    if dm is not None:
        line["dmff_block"] = dm
    if sec is not None:
        line["secondary"] = {"note": "same detector path at BASELINE configs[1] (batch 1: the launch/latency-bound regime of the same kernels)",
                             "metric": METRIC, "unit": "pairs/s", **{k: sec[k] for k in
                             ("value", "ms_per_step", "steps", "warmup", "config", "model_tflops", "roofline", "step_roofline", "gpu_launches")}}
    if notes:
        line["notes"] = notes
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="yolov5l_b16", choices=sorted(WORKLOADS))
    ap.add_argument("--layer-profile", default=None, help="write a per-launch CSV (event-timed eager pass) to this path")
    ap.add_argument("--secondary", default="auto", help="also measure this workload (device-resident value + roofline) and report it "
                    "under 'secondary'; 'auto' = yolov5s_b1 when the primary is yolov5l_b16 on 1 GPU; 'none' disables")
    ap.add_argument("--train", default="on", choices=["on", "off"], help="also time the training step of the workload's model (reported "
                    "under 'train'; with N > 1 it runs under DDP and names the gradient all-reduce's share)")
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--mode", default="infer", choices=["infer", "train"], help="train: the JSON line's top-level metric is the training "
                    "step (BASELINE configs[3]; under torchrun it is the DDP step with its gradient all-reduce) instead of inference")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="after the timed steps, write what the timed path computed in "
                    "its last step as DIR/<name>.npy (float32; rank 0): infer -> z, logits, x0..x2 of the detector; train -> loss, "
                    "loss_items and a fixed sample of 2^20 parameter values after the step")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        from icafusion_b200 import _lib
        _lib.lib()        # fail loudly if the CUDA library is missing
        run_ours(args, wl)


if __name__ == "__main__":
    main()
