#!/usr/bin/env python
"""bench.py -- FasterSeg student (arch_1, F12.L16) inference FPS @ 1x3x1024x2048 on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one 1024x2048 frame through the student network (BASELINE.json configs[1]).
  value : frames/s with the frame already resident in HBM (CUDA-graph replay of the whole forward; full-resolution
          fp16 NCHW logits are materialised, i.e. the work the reference's `model(input)` does in
          tools/utils/darts_utils.py:182-223)
  e2e   : frames/s through the public host API (fasterseg_b200.runtime.InferencePipeline) on the evaluator path
          (tools/engine/evaluator.py:206-225): pinned-host uint8 HWC image -> H2D -> normalisation folded into the stem kernel
          -> network -> fused upsample+argmax -> uint8 label map D2H, 3 frames in flight.  `e2e_fp32_input` is the same with
          the normalised fp32 NCHW frame of round 1 (25 MB per frame over PCIe).
  roofline    : the dominant kernel (tcgen05 implicit-GEMM conv) timed live on BOTH 9.66-GFLOP layers of the frame
                (heads8 3x3 128->128 @128x256 and stem.1.conv2 64->64 @256x512); the line reports the WORSE of the two
  supernet_steps: the other half of BASELINE's metric -- pretrain (configs[2]) and search (configs[4]) step of the 16-layer
                supernet with the reference's OHEM criterion, as captured passes; under torchrun data parallel (SyncBN over
                NVLink peer memory + one flat gradient all-reduce), images/s summed over ranks
  cpu_baseline: the CPU oracle port of the reference path (same weights) on the host cores (N=1, rank 0 only)
Multi-GPU: inference has no exchange step -> N independent replicas ("replicas only"), weak scaling.
`--impl reference` times the reference's CPU path (oracle port; the Python reference tree does not exist on the GPU box).
`--dump-outputs DIR`: after the timed steps, DIR/logits.npy holds what the last one computed (see dump_outputs); weights and input
frames are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fasterseg_student_fps_1024x2048"
UNIT = "frames/s"
H, W = 1024, 2048
WORKLOAD = "FasterSeg student arch_1 (F12.L16, lasts=[2,1]) inference, 1x3x1024x2048, batch 1 per GPU"  # BASELINE configs[1]
STUDENT_GFLOP = 55.54  # 2*MAC over the 45 convs of arch_1 @1024x2048 (SURVEY section 8a)


def synth_weights_(model, seed=12345):
    """Synthetic parameters per SURVEY 8(d): kaiming_normal(fan_in, relu) convs, BN gamma/beta/running stats randomised
    so eval-mode BN is not a no-op.  Deterministic (CPU generator) so every rank / impl sees the same network."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in sorted(model.state_dict().items()):
            if name.endswith("num_batches_tracked"):
                continue
            shp = tuple(p.shape)
            if p.dim() == 4:
                fan_in = shp[1] * shp[2] * shp[3]
                v = torch.randn(shp, generator=g) * (2.0 / fan_in) ** 0.5
            elif name.endswith("running_var"):
                v = torch.rand(shp, generator=g) + 0.5
            elif name.endswith("running_mean"):
                v = torch.randn(shp, generator=g) * 0.1
            elif name.endswith("conv_1x1.bias"):
                v = torch.randn(shp, generator=g) * 0.05
            elif name.endswith(".weight"):
                v = 1.0 + 0.1 * torch.randn(shp, generator=g)
            else:
                v = 0.1 * torch.randn(shp, generator=g)
            p.copy_(v)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps, m.momentum = 1e-5, 0.1


class ClockSampler:
    """SM clock / throttle reasons sampled every 100 ms during the timed regions (B200_PROFILING.md).  Uses NVML in-process
    (nvidia_ml_py): spawning `nvidia-smi -lms` next to a host-driven copy/launch pipeline halves its throughput because each
    poll takes driver locks; the nvidia-smi CLI is only the fallback."""

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.mode = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.nv = pynvml
            self.mode = "nvml"
        except Exception:
            self.mode = "smi"
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip() != ""]
            try:
                return int(ids[self.gpu_index])
            except (ValueError, IndexError):
                pass
        return self.gpu_index

    def _loop(self):
        while not self.stop_flag:
            try:
                if self.mode == "nvml":
                    nv = self.nv
                    sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    smax = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append((float(sm), float(smax), int(reasons)))
                else:
                    out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                                          "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                                          "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-i",
                                          str(self.gpu_index)], capture_output=True, text=True, timeout=5).stdout
                    f = [x.strip() for x in out.strip().split(",")]
                    bits = 0
                    for bit, val in zip((0x8, 0x40, 0x20, 0x4), f[2:6]):
                        if val.lower().startswith("active"):
                            bits |= bit
                    self.samples.append((float(f[0]), float(f[1]), bits))
            except Exception:
                pass
            time.sleep(0.1 if self.mode == "nvml" else 1.0)

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=3)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = sorted({n for _, _, r in self.samples for bit, n in names.items() if r & bit})
        return {"sm_mhz": statistics.median(s for s, _, _ in self.samples), "sm_max_mhz": max(m for _, m, _ in self.samples),
                "reasons": reasons, "samples": len(self.samples), "via": self.mode}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


KERNEL_NAMES = {0: "conv_direct_kernel", 1: "conv_tc_kernel (per-tap, 128 px x Cout tile)", 2: "conv_tc2_kernel (row strip)",
                3: "conv_tc3_kernel (channel-major 128 x 256 MMA)", 4: "conv_tc4_kernel (CTA pair, cta_group::2)",
                5: "conv_tc5_kernel (tap-concatenated N = 3*Cout, flattened-pixel tiles)"}


def _time_conv_layer(device, Cin, Cout, h, w, reps=5):
    """one 3x3 stride-1 conv+BN+ReLU launch, CUDA events over rotating > L2 buffers -> (us per launch, kernel id)"""
    import ctypes as C
    from fasterseg_b200 import _lib
    from fasterseg_b200 import functional as F_
    per_pair = 2.0 * (Cin + Cout) * h * w
    nbuf = max(6, int(160e6 / per_pair) + 1)   # > 126 MB L2: every launch reads its input from HBM
    xs = [F_.empty_nhwc(1, Cin, h, w, device).normal_() for _ in range(nbuf)]
    ys = [F_.empty_nhwc(1, Cout, h, w, device) for _ in range(nbuf)]
    wt = torch.randn(Cout, Cin, 3, 3, device=device) * 0.03
    wp = F_.pack_conv_weight(wt, Cin, Cout, 3)
    scale = torch.rand(Cout, device=device) + 0.5
    shift = torch.randn(Cout, device=device) * 0.1
    d = _lib.ConvDesc(1, h, w, Cin, Cout, 3, 1, 1, 1, 0, 0, h, w, Cin, Cout, _lib.FSB_CONV_RELU | _lib.FSB_CONV_AFFINE)
    kid = _lib.lib().fsb_conv_kernel_id(C.byref(d), C.c_void_p(ys[0].data_ptr()), 0)
    for i in range(nbuf):
        F_.conv_fwd(xs[i], wp, Cout, 3, 1, 1, scale, shift, relu=True, out=ys[i])
    torch.cuda.synchronize()
    st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st.record()
    for _ in range(reps):
        for i in range(nbuf):
            F_.conv_fwd(xs[i], wp, Cout, 3, 1, 1, scale, shift, relu=True, out=ys[i])
    en.record()
    en.synchronize()
    return st.elapsed_time(en) * 1000.0 / (reps * nbuf), kid


def dominant_kernel_roofline(device):
    """The tcgen05 implicit-GEMM conv on the two most expensive launches of the student frame (9.66 GFLOP each, 17 % of the
    frame's FLOPs each): heads8.conv_3x3 (128 -> 128 channels on the 128x256 map, intensity 566 FLOP/B: tensor-bound) and
    stem.1.conv2 (64 -> 64 on the 256x512 map, intensity 288 FLOP/B: at the ridge, 5.7 us by FLOPs vs 5.1 us by bytes).
    Algorithmic work per launch: 2*9*Cin*Cout*h*w FLOP; bytes = input + output + weights, each once, fp16.
    The line's `roofline` is the WORSE of the two; both are listed under `layers`."""
    pk = measured_peaks()
    traffic = {}  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures, per layer
    tj = os.path.join(ROOT, "profiles", "r2_roofline_traffic.json")
    if os.path.isfile(tj):
        with open(tj) as f:
            traffic = {k: v.get("traffic_bytes") for k, v in json.load(f).get("layers", {}).items()}
    layers = []
    for label, Cin, Cout, h, w in (("heads8.conv_3x3: 3x3 128->128 @128x256", 128, 128, 128, 256),
                                   ("stem.1.conv2: 3x3 64->64 @256x512", 64, 64, 256, 512)):
        us, kid = _time_conv_layer(device, Cin, Cout, h, w)
        flops = 2.0 * 9 * Cin * Cout * h * w
        abytes = 2.0 * (Cin * h * w + Cout * h * w + 9 * Cin * Cout)
        t_tensor, t_hbm = flops / (pk["tflops"] * 1e12), abytes / (pk["hbm_gbs"] * 1e9)
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        achieved = flops / (us * 1e-6) / 1e12 if bound == "tensor" else abytes / (us * 1e-6) / 1e9
        peak = pk["tflops"] if bound == "tensor" else pk["hbm_gbs"]
        layers.append({"kernel": "%s on %s" % (KERNEL_NAMES.get(kid, "?"), label), "bound": bound, "achieved": round(achieved, 2),
                       "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": round(achieved / peak, 4),
                       "us_per_launch": round(us, 2), "roofline_us": round(max(t_tensor, t_hbm) * 1e6, 2),
                       "algorithmic_flops": flops, "algorithmic_bytes": abytes})
    worst = dict(min(layers, key=lambda r: r["frac"]))
    worst.update({"traffic": next((v for k, v in traffic.items() if k in worst["kernel"]), None), "peak_source": pk["source"], "layers": layers,
                  "note": "worse of the two 9.66-GFLOP launches of the frame.  A tcgen05.mma costs ~130-180 cycles whatever N is "
                          "(tools/umma_rate.cu), so heads8 runs channel-major (weights as M = 128, 256 pixels as N) and "
                          "stem.1.conv2 (64 output channels) concatenates the three horizontal taps along N (N = 192, 12 MMAs per "
                          "120 pixels instead of 36 per 128) and applies the horizontal shift in the epilogue; with K = 576 the "
                          "accumulator drain (TMEM -> registers, 98 KB per tile) is as long as the MMAs themselves"})
    return worst


def cpu_port_fps(model_state_cpu, frames, threads):
    """Time the oracle port (CPU fp32 restatement of train/model_seg.py:337-366, executing the same ATen conv / batch-norm /
    interpolate calls the reference makes) on `frames` 1024x2048 frames."""
    from oracle import fasterseg_oracle as orc
    from tests import helpers as Hh
    torch.set_num_threads(threads)
    st, _ = Hh.student_structure(1)
    x = orc.random_input((1, 3, H, W), seed=12345)
    orc.RESIZE_IMPL["aten"] = True
    try:
        with torch.no_grad():
            orc.student_forward(x, model_state_cpu, st, training=False)  # warm-up
            t0 = time.perf_counter()
            for _ in range(frames):
                orc.student_forward(x, model_state_cpu, st, training=False)
            dt = time.perf_counter() - t0
    finally:
        orc.RESIZE_IMPL["aten"] = False
    return frames / dt, dt


def reference_student_cpu():
    """The UNMODIFIED reference's own student network (train/model_seg.py Network_Multi_Path_Infer built as train/train.py:95-118 builds
    it) on CPU, from the mounted tree or the verbatim copy build() keeps under oracle/_ref -- or None where neither exists."""
    try:
        import contextlib
        from oracle import ref_harness
        if not ref_harness.reference_available():
            return None
        with contextlib.redirect_stdout(sys.stderr):      # the reference prints at import time; stdout carries the JSON line only
            ns = ref_harness.load_reference("train", "model_seg")
            model, _, _ = ref_harness.build_reference_student(ns, 1)
        synth_weights_(model)
        return model.eval()
    except Exception:  # noqa: BLE001 -- the port is the fallback
        return None


def reference_fps(model, frames, threads):
    torch.set_num_threads(threads)
    x = torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(12345))
    with torch.no_grad():
        model(x)
        t0 = time.perf_counter()
        for _ in range(frames):
            model(x)
        dt = time.perf_counter() - t0
    return frames / dt, dt


def bind_to_one_numa_node():
    """Reference arm only: a batch-1 CPU forward is memory-bound and loses ~3x when its threads and buffers straddle two sockets
    (14.5 vs 4.9 frames/s measured on the same box), so give the reference its best case -- every thread of this process on the
    CPUs of ONE NUMA node.  Best effort; returns the number of CPUs kept (0 = nothing changed)."""
    try:
        have = os.sched_getaffinity(0)
        best = set()
        base = "/sys/devices/system/node"
        for d in sorted(os.listdir(base)):
            if not (d.startswith("node") and d[4:].isdigit()):
                continue
            cpus = set()
            for part in open(os.path.join(base, d, "cpulist")).read().strip().split(","):
                if part:
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
            cpus &= have
            if len(cpus) > len(best):
                best = cpus
        if not best or best == have:
            return 0
        for tid in os.listdir("/proc/self/task"):
            try:
                os.sched_setaffinity(int(tid), best)
            except OSError:
                pass
        return len(best)
    except Exception:  # noqa: BLE001 -- best effort
        return 0


def best_reference_threads(model):
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best = (0.0, ncpu)
    for t in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True):
        fps, _ = reference_fps(model, 2, t)
        if fps > best[0]:
            best = (fps, t)
    return best[1], best[0]


def best_cpu_threads(model_state_cpu):
    """Batch-1 convolutions do not scale to every core of a large host: try a few thread counts on one frame each and keep
    the fastest (the reference arm may use all the host threads it can USE)."""
    ncpu = os.cpu_count() or 1
    best = (0.0, ncpu)
    for t in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        fps, _ = cpu_port_fps(model_state_cpu, 1, t)
        if fps > best[0]:
            best = (fps, t)
    return best[1]


def student_cpu_baseline(sd_cpu, seconds=12.0):
    """`cpu_baseline` of the default run: the student frame on the host cores, ~`seconds` of CPU work -- through the UNMODIFIED reference
    network where its tree is available (kind "reference"), else through the oracle port (kind "port"); same weights as the GPU model."""
    ref = reference_student_cpu()
    if ref is not None:
        ref.load_state_dict(sd_cpu)
        threads, probe_fps = best_reference_threads(ref)
        frames = int(min(200, max(10, seconds * probe_fps)))
        fps, dt = reference_fps(ref, frames, threads)
        return {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "reference",
                "sample": "%d frames of 1x3x%dx%d through the UNMODIFIED reference network (train/model_seg.py, same weights) on CPU, "
                          "torch fp32, %.1f s" % (frames, H, W, dt)}
    frames = 10
    threads = best_cpu_threads(sd_cpu)
    fps, dt = cpu_port_fps(sd_cpu, frames, threads)
    return {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d frames of 1x3x%dx%d through the CPU oracle port (torch CPU fp32), %.1f s" % (frames, H, W, dt)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # nothing of the product (fasterseg_b200) is on this arm
    bound = bind_to_one_numa_node()
    ref = reference_student_cpu()
    if ref is not None:      # the reference itself (kind "reference")
        threads, _ = best_reference_threads(ref)
        for _ in range(max(0, min(args.warmup, 3) - 1)):
            reference_fps(ref, 1, threads)
        fps, dt = reference_fps(ref, args.steps, threads)
        line = {"impl": "reference", "metric": METRIC, "value": round(fps, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(1000.0 / fps, 2), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "arithmetic": "UNMODIFIED reference (train/model_seg.py) on CPU: fp32 NCHW, torch CPU (ATen/oneDNN)"},
                "cpu_baseline": {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "reference",
                                 "sample": "%d frames of 1x3x1024x2048 through the reference's own Network_Multi_Path_Infer (arch_1), torch CPU fp32, best of {all, 1/2, 32, 16, 8} threads = %d (host has %d CPUs; process bound to %s)" % (args.steps, threads, os.cpu_count() or 1, ("the %d CPUs of one NUMA node" % bound) if bound else "its inherited affinity")},
                "e2e": {"value": round(fps, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    # fallback: the oracle port (structure, weights and arithmetic all from oracle/)
    from oracle import fasterseg_oracle as orc
    from tests import helpers as Hh
    st, _ = Hh.student_structure(1)
    sd = orc.random_state_dict(orc.student_param_shapes(st, training=False), seed=12345)
    threads = best_cpu_threads(sd)
    for _ in range(max(0, min(args.warmup, 3) - 1)):
        cpu_port_fps(sd, 1, threads)
    fps, dt = cpu_port_fps(sd, args.steps, threads)
    line = {"impl": "reference", "metric": METRIC, "value": round(fps, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(1000.0 / fps, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "arithmetic": "reference CPU path (oracle port): fp32 NCHW, torch CPU (ATen/oneDNN)"},
            "cpu_baseline": {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "%d frames of 1x3x1024x2048, torch CPU fp32 (ATen/oneDNN), best of {all, 1/2, 32, 16} threads = %d (host has %d)" % (args.steps, threads, os.cpu_count() or 1)},
            "e2e": {"value": round(fps, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


DUMP_PIXELS = 1 << 19
DUMP_SEED = 2024


def dump_outputs(directory, logits):
    """The frame's NCHW logits as float32 DIR/logits.npy of shape (N, C, DUMP_PIXELS): every class at DUMP_PIXELS pixel positions
    drawn without replacement from a fixed seed and kept in row-major order (40 MB instead of the 159 MB of the full frame)."""
    import numpy as np
    n, c, h, w = logits.shape
    pix = np.sort(np.random.RandomState(DUMP_SEED).choice(h * w, min(DUMP_PIXELS, h * w), replace=False))
    sample = logits.reshape(n, c, h * w).index_select(2, torch.from_numpy(pix).to(logits.device))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "logits.npy"), sample.float().cpu().numpy())


def frame_sigma_roofline(model, x, frame_us):
    """Whole-frame efficiency: sum over the frame's launches of max(FLOPs / tensor peak, algorithmic bytes / HBM peak) at the
    measured peaks, divided by the measured frame time (SURVEY section 8d).  The launch list comes from one eager forward
    with the wrappers instrumented (fasterseg_b200/roofline.py); extra key only."""
    try:
        from fasterseg_b200 import roofline as RL
        with torch.no_grad():
            recs = RL.trace_launches(lambda: model(x))
        torch.cuda.synchronize()
        pk = measured_peaks()
        s = RL.sigma_roofline(recs, pk["tflops"], pk["hbm_gbs"])
        return {"sum_us": round(s["sum_us"], 1), "frame_us": round(frame_us, 1), "frac": round(s["sum_us"] / frame_us, 4),
                "launches": s["launches"], "tensor_bound_launches": s["tensor_bound_launches"], "gflop": round(s["gflop"], 2),
                "algorithmic_mbytes": round(s["mbytes"], 1), "peak_source": pk["source"]}
    except Exception as e:  # noqa: BLE001 -- analysis key, reported not raised
        return {"error": "%s: %s" % (type(e).__name__, e)}


def _load_tool(name):
    import importlib.util
    path = os.path.join(ROOT, "tools", name + ".py")
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def supernet_cpu_step_ms(mode, threads):
    """The reference's CPU path for one supernet step (oracle port of search/model_search.py:478-505 + backward, fp32, torch CPU):
    ONE step (bounded sample: ~10-40 s), same synthetic shapes as the GPU measurement."""
    import numpy as np
    import torch.nn as nn
    from oracle import fasterseg_oracle as orc
    from oracle import supernet_oracle as sno
    torch.set_num_threads(threads)
    B, Hh, Ww = (3, 256, 512) if mode == "pretrain" else (2, 224, 448)
    from fasterseg_b200.model_search import Network_Multi_Path
    m = Network_Multi_Path(19, 16, nn.CrossEntropyLoss(ignore_index=255), Fch=12, width_mult_list=orc.WIDTH_MULT_LIST,
                           prun_modes=['max', 'arch_ratio'], stem_head_width=[(1, 1), (8. / 12, 8. / 12)])
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    del m
    sd = orc.random_state_dict(shapes, seed=1)
    for k, v in sd.items():
        if "running" not in k and v.dtype.is_floating_point:
            v.requires_grad_(True)
    x = orc.random_input((B, 3, Hh, Ww), seed=2)
    t = torch.randint(0, 19, (B, Hh // 8, Ww // 8), generator=torch.Generator().manual_seed(3))
    from fasterseg_b200.losses import ProbOhemCrossEntropy2d
    crit = ProbOhemCrossEntropy2d(ignore_label=255, thresh=0.7, min_kept=int(B * (Hh // 8) * (Ww // 8) // 16))
    np.random.seed(4)
    torch.manual_seed(5)
    t0 = time.perf_counter()
    n_losses = 2 if mode == "search" else 1          # the search step evaluates `_loss` twice (architect step + weight step)
    for _ in range(n_losses):
        loss = sno.supernet_loss(x, t, sd, sno.SupernetConfig(layers=16), crit, True if mode == "pretrain" else "dir")
        loss.backward()
    return (time.perf_counter() - t0) * 1e3


def distill_cpu_step_ms(threads, batch=1, hw=(512, 1024)):
    """The reference's CPU path for the teacher -> student distillation step (train/train.py:219-271) through the oracle port: teacher
    forward (eval), student forward (train) -> 3 upsampled logits, OHEM x3 + KLDivLoss, backward.  Bounded sample: `batch` images
    (the GPU number is for 12); returns ms for that batch."""
    from oracle import fasterseg_oracle as orc
    from tests import helpers as Hh
    torch.set_num_threads(threads)
    Hh_, Ww = hw
    st_t, _ = Hh.student_structure(0)
    st_s, _ = Hh.student_structure(1)
    sd_t = orc.random_state_dict(orc.student_param_shapes(st_t, training=False), seed=1)
    sd_s = orc.random_state_dict(orc.student_param_shapes(st_s, training=True), seed=2)
    for k, v in sd_s.items():
        if "running" not in k and v.dtype.is_floating_point:
            v.requires_grad_(True)
    x = orc.random_input((batch, 3, Hh_, Ww), seed=3)
    t = torch.randint(0, 19, (batch, Hh_, Ww), generator=torch.Generator().manual_seed(4))
    t0 = time.perf_counter()
    with torch.no_grad():
        tl = orc.student_forward(x, sd_t, st_t, training=False)
    l8, l16, l32 = orc.student_forward(x, sd_s, st_s, training=True)
    mk = int(batch * Hh_ * Ww // 16)
    loss = (orc.ohem_cross_entropy(l8, t, 255, 0.7, mk) + 0.2 * orc.ohem_cross_entropy(l16, t, 255, 0.7, mk)
            + 0.2 * orc.ohem_cross_entropy(l32, t, 255, 0.7, mk) + orc.distill_kl(l8, tl))
    loss.backward()
    return (time.perf_counter() - t0) * 1e3


def distill_step_metric(with_cpu):
    """BASELINE configs[3]: teacher -> student KL-distillation train step, 12 x 3 x 512 x 1024 per GPU, with the reference's criteria
    (3 x ProbOhemCrossEntropy2d + KLDivLoss) -- fused on the low-resolution logits (N1, csrc/loss.cu) and, for comparison, on
    materialised label-resolution logits.  Extra key, N = 1 only."""
    out = {}
    try:
        mod = _load_tool("distill_step_bench")
        for key, lazy in (("fused", True), ("materialised", False)):
            try:
                out[key] = mod.measure(12, (512, 1024), steps=5, warmup=2, lazy=lazy, criterion="ohem")
            except Exception as e:  # noqa: BLE001
                out[key] = {"error": "%s: %s" % (type(e).__name__, e)}
            finally:
                torch.cuda.empty_cache()
        if with_cpu:
            try:
                threads = min(os.cpu_count() or 1, 32)
                ms = distill_cpu_step_ms(threads, batch=1, hw=(256, 512))
                out["cpu_baseline"] = {"value": round(ms, 1), "unit": "ms per sample step", "cores": threads, "kind": "port",
                                       "sample": "ONE step at batch 1 x 3 x 256 x 512 through the CPU oracle port = 1/48 of the pixels of "
                                                 "the GPU step (12 x 3 x 512 x 1024); bounded to keep the bench within minutes"}
            except Exception as e:  # noqa: BLE001
                out["cpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, e)}
    except Exception as e:  # noqa: BLE001
        out["error"] = "%s: %s" % (type(e).__name__, e)
    return out


def supernet_steps_metric(rank, world, with_cpu):
    """Second half of BASELINE.json's metric: supernet pretrain step (configs[2], 3x3x256x512 per GPU) and search step
    (configs[4], 2x3x224x448 per GPU) of the 16-layer / 252 M parameter supernet through the reference-facing classes:
    `_loss` (4 forwards, 5 OHEM terms each) + backward + clip + SGD (+ the architect's first-order step for search).
    Captured passes (fasterseg_b200/graphed.py); under torchrun: data parallel, SyncBN over NVLink peer memory, one flat
    gradient all-reduce per `_loss`.  Extra key only -- it never fails the headline line."""
    out = {}
    try:
        mod = _load_tool("search_step_bench")
        for mode, steps, warm in (("pretrain", 8, 3), ("search", 5, 2)):
            try:
                res = mod.measure(mode, 16, steps=steps, warmup=warm, rank=rank, world=world, graph=True, criterion="ohem")
                res["timing"] = "host wall clock around step + synchronize, median of %d, max over ranks" % steps
                if with_cpu and rank == 0:
                    try:
                        threads = min(os.cpu_count() or 1, 32)
                        ms = supernet_cpu_step_ms(mode, threads)
                        res["cpu_baseline"] = {"value": round(ms, 1), "unit": "ms/step", "cores": threads, "kind": "port",
                                               "sample": "1 step of the same shapes through the CPU oracle port (torch CPU fp32)"}
                    except Exception as e:  # noqa: BLE001
                        res["cpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, e)}
                out[mode] = res
            except Exception as e:  # noqa: BLE001 -- secondary metric, reported not raised
                out[mode] = {"error": "%s: %s" % (type(e).__name__, e)}
            finally:
                try:
                    torch.cuda.empty_cache()
                except Exception:  # noqa: BLE001
                    pass
    except Exception as e:  # noqa: BLE001
        out["error"] = "%s: %s" % (type(e).__name__, e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-supernet-step", action="store_true",
                    help="skip the secondary metrics (supernet pretrain / search step, BASELINE configs[2] / [4]; distillation "
                         "step, configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the logits the last one computed to DIR/logits.npy (a fixed sample of pixels)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what our timed path computed; it has no meaning with --impl reference")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        from fasterseg_b200 import parallel
        parallel.init_from_env()          # NCCL group + the library's peer-memory exchange for the data-parallel supernet steps

    from fasterseg_b200 import zoo
    from fasterseg_b200.runtime import GraphedInference, InferencePipeline, bind_host_thread_to_gpu
    # before any pinned allocation: keep the host side of the H2D/D2H pipeline on the GPU's own socket
    local_cpus = None if os.environ.get("FSB_NO_CPU_BIND") == "1" else bind_host_thread_to_gpu(local_rank)

    model = zoo.build_network(1)
    synth_weights_(model)
    model = model.to(device).eval()

    # ---- device-resident FPS (value) ----
    g = torch.Generator(device="cpu").manual_seed(12345 + rank)
    npool = 6  # 6 x 25.2 MB = 151 MB of distinct frames > 126 MB L2
    pool = [torch.randn(1, 3, H, W, generator=g).to(device) for _ in range(npool)]
    runner = GraphedInference(model, pool[0], mode="logits", logits_dtype=torch.float16)
    launches_value = runner.launches_per_replay
    for i in range(args.warmup):
        runner(pool[i % npool])
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st.record()
    for i in range(args.steps):
        logits = runner(pool[i % npool])
    en.record()
    torch.cuda.synchronize()
    ms_total = st.elapsed_time(en)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logits)
    if world > 1:
        t = torch.tensor([ms_total], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * args.steps / (ms_total / 1000.0)

    # ---- end-to-end FPS through the host API ----
    checksum = [0]

    def consume(lbl):
        checksum[0] += int(lbl[0, 0, 0])  # touch the result on the host

    e2e_steps = args.steps

    def run_e2e(example, host_frames):
        pipe = InferencePipeline(model, example, mode="labels", depth=3)
        pipe.run(host_frames[i % 4] for i in range(max(3, args.warmup // 2)))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        pipe.run((host_frames[i % 4] for i in range(e2e_steps)), consume)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device=device)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        return pipe, world * e2e_steps / dt

    # evaluator path: the uint8 HWC image itself crosses PCIe (6.3 MB), normalisation happens inside the stem kernel
    model.set_input_normalization([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
    u8_frames = [torch.randint(0, 256, (1, H, W, 3), generator=g, dtype=torch.uint8).pin_memory().permute(0, 3, 1, 2) for _ in range(4)]
    pipe, e2e_fps = run_e2e(u8_frames[0].to(device), u8_frames)
    # round-1 input format (normalised fp32 NCHW frame, 25 MB): kept for comparison / fp32-input parity
    f32_frames = [torch.randn(1, 3, H, W, generator=g).pin_memory() for _ in range(4)]
    pipe32, e2e32_fps = run_e2e(pool[0], f32_frames)
    clocks = sampler.stop() if rank == 0 else None

    # Everything the headline needs from the device is measured BEFORE the secondary metrics: a failure inside the data-parallel
    # supernet steps (a peer that never arrives traps the exchange kernel and poisons the CUDA context) must not cost the line.
    roof = frame_roof = sd_cpu = None
    if rank == 0:
        roof = dominant_kernel_roofline(device)
        frame_roof = frame_sigma_roofline(model, pool[0], ms_total / args.steps * 1000.0)
        if world == 1 and not args.no_cpu_baseline:
            sd_cpu = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    steps_metric = None
    distill_metric = None
    if not args.no_supernet_step:
        del runner, pipe32
        torch.cuda.empty_cache()
        steps_metric = supernet_steps_metric(rank, world, with_cpu=(world == 1 and not args.no_cpu_baseline))
        if world == 1:
            distill_metric = distill_step_metric(with_cpu=not args.no_cpu_baseline)
    if rank != 0:
        if world > 1:
            try:
                dist.barrier()
                dist.destroy_process_group()
            except Exception:  # noqa: BLE001 -- a failed secondary metric must not turn into a non-zero exit of this rank
                pass
        return

    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "arithmetic": "fp16 NHWC storage / fp32 accumulate, full-res fp16 logits materialised",
                   "parallelism": "replicas x%d (no exchange step in inference)" % world,
                   "l2_policy": "inputs rotate through a 6-frame device pool (151 MB > 126 MB L2); activations per frame "
                                "(~430 MB) exceed L2",
                   "timing": "CUDA events around %d CUDA-graph replays, max over ranks" % args.steps,
                   "frame_gflop": STUDENT_GFLOP},
        "clocks": clocks,
        "e2e": {"value": round(e2e_fps, 1), "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
                "what": "pinned uint8 HWC image -> H2D -> normalisation folded into the stem kernel -> student -> fused "
                        "upsample+argmax -> uint8 labels D2H; 3 frames in flight (evaluator path, tools/engine/evaluator.py:206-225)",
                "steps": e2e_steps, "host_cpus_bound_to_gpu_socket": local_cpus},
        "e2e_fp32_input": {"value": round(e2e32_fps, 1), "unit": UNIT, "h2d_bytes_per_step": H * W * 3 * 4,
                           "what": "same pipeline fed with the normalised fp32 NCHW frame (round-1 format)"},
        "gpu_launches": launches_value * args.steps + pipe.launches_per_frame * e2e_steps * 2,
        "launches_per_frame": launches_value,
        "roofline": roof,
        "frame_tflops": round(STUDENT_GFLOP * value / world / 1000.0, 2),
    }
    line["frame_roofline"] = frame_roof
    if steps_metric is not None:
        line["supernet_steps"] = steps_metric
        if isinstance(steps_metric.get("pretrain"), dict) and "value" in steps_metric["pretrain"]:
            line["supernet_step"] = steps_metric["pretrain"]      # round-1 key: the pretrain step
    if distill_metric is not None:
        line["distill_step"] = distill_metric
    if sd_cpu is not None:
        try:
            line["cpu_baseline"] = student_cpu_baseline(sd_cpu)
        except Exception as e:  # noqa: BLE001 -- the baseline leg must never cost the measured line
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %s: %s" % (type(e).__name__, e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass


if __name__ == "__main__":
    main()
