#!/usr/bin/env python
"""bench.py — detection frames/sec of the LocoMouse_TM per-frame detection path on N B200s.

Contract (see the task prompt / BASELINE.json):
  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR   also writes the results of the last timed step as DIR/<name>.npy

A "step" is one pass of the hot path (lm_detect_batch through the C ABI) over one batch of synthetic
frames: SURVEY config 2 = 10 000 raw 400x1700 u8 frames per GPU, resident in HBM, six random-init
30x30 templates, LocoMouse_TM geometry.  Frames are sharded across ranks as whole videos (one 10k-frame
video per rank -> weak scaling, no data-path collective); candidate lists are gathered to rank 0.

  value  : whole-job frames/s with the frames already resident in HBM (results still return to host).
  e2e    : the same through the public API with HOST (pinned) frame buffers: H2D of every frame and D2H
           of every result inside the timed region; for N>1 the gather of the candidate lists to rank 0 too.
  roofline : the dominant kernel, k_screen2 (int8 tcgen05 screen that decides the six correlations, SURVEY §8d):
           algorithmic FLOPs per launch / its CUDA-event duration against the measured bf16 tensor peak, plus the int8
           work it actually executes against the int8 pipe; the exact dense FP32 kernel (k_corr) beside it.
  cpu_baseline : the CPU oracle (a port of the reference path), 1 thread like the reference, on the first 1000 frames
           (BASELINE configs[0]: one 1000-frame video, CPU vs 1 GPU).
  other_configs : configs[0] (1000-frame video, host frames), configs[4] (2x frames, 60x60 templates) and a
           throughput-vs-detection-density sweep; bounded samples, never part of `value`.
"""
from __future__ import annotations

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

METRIC = "detection_frames_per_sec"
UNIT = "frames/s"
FRAMES_PER_STEP = 10_000
WORKLOAD = ("configs[1]: LocoMouse_TM batched detection, 10k synthetic 400x1700 u8 frames per GPU resident in HBM, "
            "six random-init 30x30 templates")
# --dump-outputs writes the results of this many frames, drawn with a fixed seed: about 11 kB per frame in the dumped
# dtypes, 45 MB in all (the full 10k-frame result set would be 110 MB)
DUMP_FRAMES = 4096
DUMP_SEED = 0


def dump_outputs(res, out_dir: str) -> None:
    """Writes every array of `res` (the Results of one detect_batch call) for a seeded sample of its frames as
    out_dir/<name>.npy: integer fields as float32 (coordinates, counts and flags are far below 2**24, so exactly),
    scores as float64; the candidate records are split into <name>_x, <name>_y, <name>_s.  frame_index.npy holds the
    sampled frame numbers."""
    from locomouse_cpp_b200.types import CAND_DTYPE

    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(res.n, min(res.n, DUMP_FRAMES), replace=False))
    out = {"frame_index": idx.astype(np.float64)}
    for name in res.ARRAYS:
        a = getattr(res, name)[idx]
        if a.dtype == CAND_DTYPE:
            out.update({f"{name}_x": a["x"].astype(np.float32), f"{name}_y": a["y"].astype(np.float32), f"{name}_s": a["s"].copy()})
        elif a.dtype == np.float64:
            out[name] = a
        else:
            out[name] = a.astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def algorithmic_fma_per_frame(cfg, model) -> float:
    """SURVEY §8d: sum over views/templates of out_h * out_w * kh * kw (unpadded outputs x taps)."""
    tot = 0.0
    for v, h in ((0, cfg.bb_h_bottom), (1, cfg.bb_h_side)):
        for k in range(3):
            kh, kw = model.w[v][k].shape
            w = cfg.tail_w if k == 2 else cfg.bb_w
            tot += float(h) * w * kh * kw
    return tot


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.power = [], set(), []
        self.stop_flag = threading.Event()
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        while not self.stop_flag.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    self.nv, "nvmlDeviceGetCurrentClocksEventReasons") else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "nvml unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "power_w_max": max(self.power) if self.power else None, "samples": len(self.samples)}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (here: the oracle port, the reference
# itself needs the OpenCV C++ SDK which this image lacks — DESIGN.md §7), all host threads.
# ---------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from locomouse_cpp_b200 import synth
    from oracle import oracle

    spec = synth.SynthSpec()
    threads = host_threads()
    per_step = max(threads * 32, 256)  # ~0.5 s of work per step on all host threads
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, per_step, seed=1000)
    frames = frames.numpy()
    for _ in range(args.warmup):
        oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    v = per_step * args.steps / dt
    sample = f"{per_step} frames/step of the same synthetic workload (first frames of video 0), {threads} threads"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": per_step,
                       "note": "reference CPU path = oracle port (reference needs the OpenCV C++ SDK, absent here); "
                               "frames farmed over all host threads"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
def main():
    sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree and leaves nothing in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_STEP, help="frames per step per GPU (default: the 10k config)")
    ap.add_argument("--cpu-sample", type=int, default=1000, help="frames of the workload timed on the CPU oracle (1 thread); 1000 = configs[0]'s video")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[0] / configs[4] / density side measurements")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--shard-weights", default="", help="N > 1: comma-separated per-rank weights for the end-to-end job's shards instead of the measured host rates")
    ap.add_argument("--nccl-gather", action="store_true", help="N > 1: move the result records to rank 0 with an NCCL gather instead of shared host memory")
    ap.add_argument("--even-shards", action="store_true", help="N > 1: keep the end-to-end job evenly split even when the ranks' measured host rates differ")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE", help="library option for the measured arm (lm_set_option), e.g. streams=3")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help=f"write the results of the last timed step (all ranks' frames; a seeded sample of {DUMP_FRAMES} of them) "
                         "as DIR/<name>.npy in float32 / float64.  With --impl reference the dump holds the oracle's results "
                         "for that arm's own frames (their number depends on the host's thread count), so it compares only "
                         "with reference-arm dumps from hosts with as many threads")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from locomouse_cpp_b200 import sharding, synth
    from locomouse_cpp_b200.api import Detector

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    numa_bound = sharding.bind_to_gpu_numa_node(local) if world > 1 else False  # before any pinned allocation
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.frames
    spec = synth.SynthSpec()
    # identical static inputs (model incl. rho, background, calibration) on every rank; one video per rank
    cfg, model, bkg, calib, _, _, _, _ = synth.make_problem(spec, 8, seed=1000)
    frames, bx, bs, bb = synth.make_video(spec, n, 1000 + rank, dev, bkg)
    torch.cuda.synchronize()
    det = Detector(cfg, model, bkg, calib, device=local)
    for kv in args.opt:
        det.set_option(kv.split('=')[0], int(kv.split('=')[1]))
    n_streams = int(det.info("streams"))
    fma_frame = algorithmic_fma_per_frame(cfg, model)

    # ---- value: frames resident in HBM ------------------------------------------------------------------
    from locomouse_cpp_b200.types import Results

    # caller-allocated result buffers in page-locked memory, reused every step: the library copies device -> here directly
    res = Results(n, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, pinned=True)
    for _ in range(args.warmup):
        det.detect_batch(frames, bx, bs, bb, results=res)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    launches = 0
    dev_total = 0.0
    ms_screen_overlapped = 0.0
    screen_mode = int(det.info("screen_active"))
    screen_on = screen_mode >= 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        det.detect_batch(frames, bx, bs, bb, results=res)
        tm, nl = det.last_timing()
        dev_total += tm["total"]
        launches += nl
        if screen_on:
            ms_screen_overlapped += det.info("ms_screen")
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    sampler.stop_flag.set()
    barrier()
    wall = max_over_ranks(wall)
    dev_ms = max_over_ranks(dev_total)
    value = world * n * args.steps / wall
    overflow = int((res.flags != 0).sum())
    if args.dump_outputs:   # before the passes below reuse `res`
        parts = sharding.gather_to_rank0(res, device=dev) if world > 1 else [res]
        if rank == 0:
            dump_outputs(sharding.concat(parts) if world > 1 else res, args.dump_outputs)
        barrier()

    # ---- instrumented pass: per-kernel device times --------------------------------------------------------------
    # In the timed loop above consecutive sub-batches overlap on two streams, so a kernel's event-to-event time there
    # includes waiting for SMs held by the other stream.  The same steps are therefore repeated with "streams" = 1
    # (identical kernels and results, strictly serial) to time each stage alone with CUDA events on the library's stream.
    det.set_option("streams", 1)
    det.detect_batch(frames, bx, bs, bb, results=res)
    stage = {k: 0.0 for k in Detector.STAGES}
    ms_screen = 0.0
    isteps = max(1, min(args.steps, 2))
    for _ in range(isteps):
        det.detect_batch(frames, bx, bs, bb, results=res)
        tm, _nl = det.last_timing()
        for k in stage:
            stage[k] += tm[k]
        if screen_on:
            ms_screen += det.info("ms_screen")
    for k in stage:
        stage[k] *= args.steps / isteps   # normalised to the number of timed steps, as the fields below assume
    ms_screen *= args.steps / isteps
    subb = int(det.info("subbatch"))   # sub-batch size of the resident passes above
    # int8 MACs of the LAST launch of those passes (n - (nsub - 1) * subb frames), scaled to the average launch the roofline uses
    try:
        _last = n - ((n + subb - 1) // subb - 1) * subb
        macs_per_avg_launch = float(det.info("screen_macs")) / _last * (n / ((n + subb - 1) // subb))
    except Exception:
        macs_per_avg_launch = 0.0
    det.set_option("streams", n_streams)
    det.detect_batch(frames[: min(n, 512)], bx[: min(n, 512)], bs[: min(n, 512)], bb[: min(n, 512)])

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------
    # Screen on (default): k_screen, the int8 tcgen05 implicit GEMM, is the dominant kernel -> "tensor" bound; its
    # algorithmic work is the correlation it decides (SURVEY §8d: 720.7 MFLOP per frame), not the MMA work it executes.
    # Screen off: k_corr, the dense exact FP32 kernel -> FP32 FMA pipe.
    nsub = (n + subb - 1) // subb
    launches_per_step = nsub
    flop_per_launch = 2.0 * fma_frame * (n / nsub)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_nominal = 148 * 128 * 2 * sm_max * 1e6 / 1e12
    ffma_measured = None
    try:
        if rank == 0:
            out = subprocess.run([os.path.join(ROOT, "tools", "ffma_peak")], capture_output=True, text=True, timeout=60,
                                 env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(local))).stdout
            ffma_measured = json.loads(out.strip().splitlines()[-1])
    except Exception:
        ffma_measured = None

    def traffic_of(kernel):
        """DRAM bytes of one launch from the round's ncu capture, scaled from the capture's frames per launch to this run's."""
        try:
            j = json.load(open(os.path.join(ROOT, "profiles", f"{kernel}_traffic.json")))
            per = j.get("dram_bytes_per_launch")
            fpl = j.get("frames_per_launch")
            if per is None:
                return None
            return int(per * (n / nsub) / fpl) if fpl else per
        except Exception:
            return None

    def executed_int8(det, ms_per_launch, flop_alg, sm_mhz, rank, local):
        """The int8 multiply-accumulates k_screen2 issues per launch (counted by the launcher from its job table) against
        the int8 tensor pipe: nominal 8192 MAC/clk/SM and the rate tools/umma_pair_probe measures on this GPU for the kernel's own
        instruction (tcgen05.mma.cta_group::2.kind::i8, M = 256, N = 192, same descriptors, no producer / epilogue)."""
        macs = macs_per_avg_launch
        if macs <= 0:
            return None
        tops = 2.0 * macs / (ms_per_launch * 1e-3) / 1e12
        nominal = 148 * 8192 * 2 * sm_mhz * 1e6 / 1e12
        out = {"int8_mac_per_launch": macs, "int8_tops": tops, "int8_nominal_peak_tops": nominal, "frac_of_int8_nominal": tops / nominal,
               "executed_over_algorithmic": 2.0 * macs / flop_alg,
               "note": "executed/algorithmic = two int8 weight digits x 64/30 Toeplitz K padding x tile padding"}
        try:
            if rank == 0:
                o = subprocess.run([os.path.join(ROOT, "tools", "umma_pair_probe")], capture_output=True, text=True, timeout=120,
                                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(local))).stdout
                best = 0.0
                for ln in o.splitlines():
                    try:
                        j = json.loads(ln)
                    except Exception:
                        continue
                    if j.get("cg") == 2 and j.get("N") == 192 and j.get("cuda") == "no error" and j.get("grid", 0) >= 148 and not j.get("mix"):
                        best = max(best, float(j.get("mac_per_cycle_per_sm", 0.0)))
                if best > 0:
                    probe = 148 * best * 2 * sm_mhz * 1e6 / 1e12
                    out["int8_probe_peak_tops"] = probe
                    out["frac_of_int8_probe_peak"] = tops / probe
                    out["probe"] = "tools/umma_pair_probe: the kernel's own pair instruction (M 256, N 192, K 32, kind::i8) on all SMs (mac/clk/SM) x 148 x SM clock"
        except Exception as ex:  # pragma: no cover
            out["probe_error"] = repr(ex)
        return out

    corr_ms_per_launch = stage["corr"] / (launches_per_step * args.steps)
    corr_tflops = flop_per_launch / (corr_ms_per_launch * 1e-3) / 1e12
    if screen_on:
        scr_ms_per_launch = ms_screen / (launches_per_step * args.steps)
        achieved = flop_per_launch / (scr_ms_per_launch * 1e-3) / 1e12
        # the kernel is timed alone (serial instrumented pass, a few tens of ms, SM clock at its maximum): the burst figure applies
        tensor_peak = float(peaks.get("bf16_tflops", 1590.0))
        tensor_sustained = peaks.get("bf16_tflops_sustained")
        roofline = {"kernel": "k_screen2" if screen_mode == 2 else "k_screen", "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": achieved / tensor_peak,
                    "frac_of_sustained_peak": (achieved / float(tensor_sustained)) if tensor_sustained else None,
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops (burst: the kernel is timed alone in a short serial pass at the maximum SM clock); "
                                    "bf16_tflops_sustained beside it" if "bf16_tflops" in peaks else "fallback 1590 TFLOP/s"),
                    "traffic": traffic_of("k_screen2" if screen_mode == 2 else "k_screen"), "launch_ms": scr_ms_per_launch, "flop_per_launch": flop_per_launch,
                    "share_of_step": ms_screen / max(stage["total"], 1e-9),
                    "launch_ms_in_timed_region_overlapped": ms_screen_overlapped / (launches_per_step * args.steps),
                    "note": "algorithmic FLOPs = the exact correlation the screen decides (SURVEY 8d), not the int8 MMA work executed "
                            "(see `executed`)",
                    "executed": executed_int8(det, scr_ms_per_launch, flop_per_launch, sm_max, rank, local),
                    "correlation_stage": {"kernels": ("k_screen2" if screen_mode == 2 else "k_screen") + " + k_corr_sparse", "launch_ms": corr_ms_per_launch,
                                          "achieved_tflops": corr_tflops, "vs_fp32_fma_nominal_peak": corr_tflops / fp32_nominal,
                                          "fp32_fma_nominal_peak": fp32_nominal,
                                          "share_of_step": stage["corr"] / max(stage["total"], 1e-9)}}
    else:
        roofline = {"kernel": "k_corr", "bound": "fp32_fma", "achieved": corr_tflops, "peak": fp32_nominal, "unit": "TFLOP/s",
                    "frac": corr_tflops / fp32_nominal,
                    "peak_source": f"nominal 148 SM x 128 FMA/clk x 2 x {sm_max:.0f} MHz (MEASURED_PEAKS.json has no FP32 entry)",
                    "traffic": traffic_of("k_corr"), "launch_ms": corr_ms_per_launch, "flop_per_launch": flop_per_launch,
                    "share_of_step": stage["corr"] / max(stage["total"], 1e-9)}
    # whole-path view of the north_star roofline ("the slower of HBM bytes at peak bandwidth and FMAs at peak"):
    flop_frame = 2.0 * fma_frame
    hbm_fps = float(peaks.get("hbm_gbs", 6650.0)) * 1e9 / (cfg.vid_rows * cfg.vid_cols)
    fma_fps = fp32_nominal * 1e12 / flop_frame
    tensor_fps = float(peaks.get("bf16_tflops", 1590.0)) * 1e12 / flop_frame
    per_gpu = value / world
    roofline["whole_path"] = {
        "frames_per_s_per_gpu": per_gpu,
        "bounds_frames_per_s": {"hbm": hbm_fps, "fp32_fma": fma_fps, "bf16_tensor": tensor_fps},
        "frac_of_north_star_roofline": per_gpu / min(hbm_fps, fma_fps),
        "frac_of_tensor_roofline": per_gpu / min(hbm_fps, tensor_fps),
        "note": "north_star roofline = min(HBM bytes at measured bandwidth, correlation FMAs at the FP32 FMA peak); the path exceeds "
                "it because the FMAs run as an exact int8 screen on the tensor cores"}
    roofline["peak_measured_ffma_microbench"] = (ffma_measured or {}).get("ffma_reg_tflops")
    roofline["hbm"] = {"kernel": "k_minmax", "achieved": (n * args.steps * 680000.0 / 1e9) / max(stage["minmax"] * 1e-3, 1e-12),
                       "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                       "note": "k_minmax + k_lut time; the only pass over whole raw frames"}
    # the dense exact kernel on a bounded sample of the same frames, for reference (never part of `value`)
    if screen_on and rank == 0:
        try:
            m = min(n, 4 * subb)
            det.set_option("screen", 0)
            det.set_option("streams", 1)   # stage events of a strictly serial run: no cross-stream waiting inside "corr"
            det.detect_batch(frames[:m], bx[:m], bs[:m], bb[:m])
            det.detect_batch(frames[:m], bx[:m], bs[:m], bb[:m])
            tm0, _ = det.last_timing()
            dense_tflops = 2.0 * fma_frame * m / (tm0["corr"] * 1e-3) / 1e12
            roofline["dense_exact_kernel"] = {"kernel": "k_corr", "bound": "fp32_fma", "achieved": dense_tflops, "peak": fp32_nominal,
                                              "frac": dense_tflops / fp32_nominal, "frames": m, "corr_ms": tm0["corr"],
                                              "frac_of_measured_ffma": (dense_tflops / ffma_measured["ffma_reg_tflops"]) if ffma_measured else None}
            det.set_option("screen", screen_mode)
            det.set_option("streams", n_streams)
            det.detect_batch(frames[:m], bx[:m], bs[:m], bb[:m])  # re-prepare scratch before the e2e leg
        except Exception as ex:  # pragma: no cover
            roofline["dense_exact_kernel"] = {"error": repr(ex)}

    # ---- SURVEY 8f-1: pass 1 of LocoMouse_TM_DE on the same resident frames (HBM-bound; not part of `value`) --------
    pass1 = None
    if rank == 0:
        try:
            from locomouse_cpp_b200.types import bb_de_params

            pp = bb_de_params(cfg, side_h=spec.side_h)
            det.bounding_box_tm_de(frames, pp)
            t1 = time.perf_counter()
            reps = 2
            for _ in range(reps):
                det.bounding_box_tm_de(frames, pp)
            dt1 = (time.perf_counter() - t1) / reps
            pass1 = {"frames_per_s": n / dt1, "ms_per_10k_frames": dt1 * 1e3 * 10000 / n,
                     "hbm_gbs_algorithmic": n * cfg.vid_rows * cfg.vid_cols / dt1 / 1e9,
                     "note": "lm_bounding_box_tm_de (k_minmax + k_lut + k_bb_hist + k_bb_pred + k_bb_cols) + host moving average; "
                             "algorithmic bytes = one read of every raw frame"}
        except Exception as ex:  # pragma: no cover
            pass1 = {"error": repr(ex)}
        try:   # the two other pass-1 variants (SURVEY 8f-1) on a bounded sample of the same resident frames
            from locomouse_cpp_b200.types import bb_base_params, bb_tm_params

            m1 = min(n, 2048)
            yy, xx = np.mgrid[-5:6, -5:6]
            dk = ((xx * xx + yy * yy) <= 5.5 ** 2).astype(np.float64)
            dk = (dk / dk.sum()).astype(np.float32)
            ptm = bb_tm_params(cfg, dk, side_h=spec.side_h, side_threshold=40, min_pixel_count=25, sums_as_float=0)
            pbs = bb_base_params(cfg, side_h=spec.side_h, sums_as_float=0)
            for name, fn in (("tm", lambda: det.bounding_box_tm(frames[:m1], ptm)), ("base", lambda: det.bounding_box_base(frames[:m1], pbs))):
                fn()
                t1 = time.perf_counter()
                fn()
                dt1 = time.perf_counter() - t1
                pass1["pass1_" + name] = {"frames": m1, "frames_per_s": m1 / dt1, "ms_per_10k_frames": dt1 * 1e7 / m1}
            pass1["pass1_note"] = ("pass1_tm: lm_bounding_box_tm (LocoMouse_TM::computeMouseBox_DD: bwAreaOpen, 11x11 disk filter, imfill); pass1_base: "
                                   "lm_bounding_box_base (11x11 median, largest component of both views); integer sums")
        except Exception as ex:  # pragma: no cover
            if isinstance(pass1, dict):
                pass1["pass1_other_error"] = repr(ex)[:200]

    # ---- SURVEY 8f-2: the tracker's cost builders for the whole result set on the device (not part of `value`) -------
    costs = None
    if rank == 0:
        try:
            from locomouse_cpp_b200.types import location_priors, pairwise_params
            from oracle import oracle as _orc  # checker + CPU timing beside it, on a bounded sample

            rows = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
                    (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0)]
            pri = location_priors(rows)
            pw = pairwise_params(cfg.bb_w, cfg.bb_h_bottom)
            det.unary_costs(res, 0, cfg.bb_w, cfg.bb_h_bottom, pri)
            offs, jc, ir, pr = det.pairwise_costs(res, 0, pw)
            def run_costs():
                for feat in range(2):
                    det.unary_costs(res, feat, cfg.bb_w, cfg.bb_h_bottom, pri)
                    det.pairwise_costs(res, feat, pw, cap=len(ir) + len(ir) // 8 + 1024)

            run_costs()   # warm-up: the page-locked output blocks return to torch's host allocator cache and are reused below
            t1 = time.perf_counter()
            run_costs()
            dt1 = time.perf_counter() - t1
            m = min(n, 512)
            t2 = time.perf_counter()
            ok = True
            for f in range(1, m):
                a = res.candidates_bottom(f - 1, 0)
                b_ = res.candidates_bottom(f, 0)
                _, nc_, wjc, wir, wpr = _orc.pairwise_potential(a, b_, pw)
                ok = ok and np.array_equal(ir[offs[f]:offs[f + 1]], wir) and np.array_equal(pr[offs[f]:offs[f + 1]].view(np.uint64), wpr.view(np.uint64))
            dt2 = time.perf_counter() - t2
            costs = {"frames_per_s": n / dt1, "ms_per_10k_frames": dt1 * 1e3 * 10000 / n, "stored_entries_paw": int(len(ir)),
                     "bit_exact_on_sample": bool(ok), "cpu_port_frames_per_s_one_feature_pairwise_only": (m - 1) / dt2,
                     "note": "lm_unary_costs + lm_pairwise_costs for both features, candidates uploaded from host memory, matrices returned to "
                             "page-locked buffers (cached by torch's host allocator) inside the timed region (transfer bound, not kernel bound); CPU figure = oracle pairwisePotential "
                             f"through ctypes on the first {m} frames, one feature"}
        except Exception as ex:  # pragma: no cover
            costs = {"error": repr(ex)}

    # ---- e2e: host (pinned) buffers, H2D + D2H inside the timed region -------------------------------------
    e2e = None
    host = None
    if not args.no_e2e:
        try:
            host = torch.empty((n,) + tuple(frames.shape[1:]), dtype=torch.uint8, pin_memory=True)
            host.copy_(frames)
            torch.cuda.synchronize()
            frames = None
            torch.cuda.empty_cache()

            # what the host can deliver at this N: every rank copies its own page-locked frames to its GPU at the same time
            # (bare cudaMemcpyAsync, no kernels); the slowest rank bounds a weak-scaling step, as it does for the real path
            ceiling = None
            try:
                devbuf = torch.empty((min(n, 2048),) + tuple(host.shape[1:]), dtype=torch.uint8, device=dev)
                nb = devbuf.shape[0]
                devbuf.copy_(host[:nb], non_blocking=True)
                torch.cuda.synchronize()
                barrier()
                t0 = time.perf_counter()
                reps = max(1, n // nb)
                for q in range(reps):
                    devbuf.copy_(host[q * nb:(q + 1) * nb], non_blocking=True)
                torch.cuda.synchronize()
                mine = reps * nb * cfg.vid_rows * cfg.vid_cols / (time.perf_counter() - t0) / 1e9
                slowest = -max_over_ranks(-mine)
                barrier()
                ceiling = {"per_gpu_gbs_slowest": slowest, "aggregate_gbs_by_slowest": slowest * world, "this_rank_gbs": mine}
                del devbuf
                torch.cuda.empty_cache()
            except Exception as ex:  # pragma: no cover
                ceiling = {"error": repr(ex)}
            # Shards by measured host rate: on a box whose GPUs sit behind unequal host paths an even split is bound by the
            # slowest rank.  8-GPU pool box (profiles/r02_bench_n8.json, profiles/r02_bench_n8_even.json): four GPUs copy at
            # 23 GB/s and four at 35 GB/s when all copy at once; even shards 331 ms per step (242 k frames/s, 164 GB/s in
            # total), shards in proportion to those rates 295 ms (271 k frames/s, 185 GB/s).  The job's world x n frames are dealt
            # by sharding.weighted_counts; rates within 5 % of each other keep the even split (--even-shards forces it,
            # --shard-weights overrides the measured rates).
            counts = [n] * world
            if world > 1 and ceiling and "this_rank_gbs" in ceiling and not args.even_shards:
                rt = torch.tensor([ceiling["this_rank_gbs"]], dtype=torch.float64, device=dev)
                rates = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
                dist.all_gather(rates, rt)
                rates = [float(x.item()) for x in rates]
                ceiling["per_rank_gbs"] = list(rates)
                if args.shard_weights:
                    rates = [float(x) for x in args.shard_weights.split(",")]
                    if len(rates) != world:
                        raise ValueError("--shard-weights needs one weight per rank")
                if max(rates) > 1.05 * min(rates):
                    counts = sharding.weighted_counts(world * n, rates)
                    if not args.shard_weights:
                        ceiling["aggregate_gbs_sum_of_rates"] = float(sum(rates))
            n_e = counts[rank]
            e_bx, e_bs, e_bb, e_res = bx, bs, bb, res
            if n_e != n:
                if n_e > n:   # this rank takes more than one video's worth: the synthetic video repeats
                    bigger = torch.empty((n_e,) + tuple(host.shape[1:]), dtype=torch.uint8, pin_memory=True)
                    bigger[:n].copy_(host)
                    bigger[n:].copy_(host[:n_e - n])
                    host = bigger
                e_bx, e_bs, e_bb = (np.resize(a, n_e) for a in (bx, bs, bb))
                e_res = Results(n_e, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, pinned=True)
            e_host = host[:n_e]
            gather_mode = "none"
            if world > 1:
                gather_mode = "nccl"
                if not args.nccl_gather:
                    # one box: every rank's result buffers live in named, page-locked shared memory and rank 0 reads them in
                    # place; the 11 kB per frame of fixed-capacity records do not cross PCIe again on their way to rank 0's host
                    try:
                        e_res = sharding.shared_results(n_e, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, rank,
                                                        tag=os.environ.get("MASTER_PORT", "0"))
                        gather_mode = "shared-memory" if getattr(e_res, "_shm_pinned", False) else "shared-memory (not page-locked)"
                    except Exception as ex:  # pragma: no cover
                        sys.stderr.write(f"shared result buffers unavailable ({ex!r}); gathering over NCCL\n")

            def e2e_step():
                r = det.detect_batch(e_host, e_bx, e_bs, e_bb, results=e_res)
                if world > 1:
                    sharding.gather_to_rank0(r, device=dev)
                return r

            for _ in range(max(1, min(args.warmup, 2))):
                e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                r = e2e_step()
            torch.cuda.synchronize()
            ew = max_over_ranks(time.perf_counter() - t0)
            barrier()
            d2h = sum(getattr(r, a).nbytes for a in r.ARRAYS)
            e2e = {"value": world * n * args.steps / ew, "unit": UNIT,
                   "h2d_bytes_per_step": int(n * cfg.vid_rows * cfg.vid_cols + 3 * 4 * n), "d2h_bytes_per_step": int(d2h),
                   "ms_per_step": ew / args.steps * 1e3, "numa_bound": bool(numa_bound),
                   "h2d_gbs_achieved": world * n * cfg.vid_rows * cfg.vid_cols * args.steps / ew / 1e9,
                   "h2d_ceiling_gbs": (ceiling or {}).get("aggregate_gbs_by_slowest"),
                   "frac_of_ceiling": (world * n * cfg.vid_rows * cfg.vid_cols * args.steps / ew / 1e9 /
                                       ceiling["aggregate_gbs_by_slowest"])
                   if ceiling and ceiling.get("aggregate_gbs_by_slowest") else None,
                   "h2d_ceiling": ceiling, "frames_per_rank": counts, "gather": gather_mode,
                   "note": f"frames in pinned host memory, copied H2D inside the call (overlapped with compute per {subb}-frame "
                           "sub-batch); results copied D2H" + ("; rank 0 reads every rank's records (see `gather`)" if world > 1 else "") +
                           "; h2d_ceiling = bare concurrent cudaMemcpyAsync of the same page-locked frames on every rank, N x the slowest rank's rate"}
        except Exception as ex:  # pragma: no cover
            e2e = {"value": None, "unit": UNIT, "error": repr(ex)}

    # ---- cpu baseline (rank 0, N=1 only) ----------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        from oracle import oracle

        m = min(args.cpu_sample, n)
        fr = host[:m].numpy() if frames is None else frames[:m].cpu().numpy()
        st = np.zeros(6)
        t0 = time.perf_counter()
        ref = oracle.detect(cfg, model, bkg, calib, fr, bx[:m], bs[:m], bb[:m], n_threads=1, stage_seconds=st)
        dt = time.perf_counter() - t0
        same = all(np.array_equal(getattr(ref, a)[:m], getattr(res, a)[:m]) for a in ref.ARRAYS)
        cpu = {"value": m / dt, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"first {m} frames of the benchmarked workload, oracle (C++ port of the reference path), 1 thread "
                         f"as the reference is single threaded",
               "stage_seconds": dict(zip(("preprocess", "correlation", "tail", "nms", "pairing", "total"), map(float, st))),
               "gpu_results_bit_exact_on_sample": bool(same)}

    # ---- other BASELINE configs and the density sweep (rank 0, N=1 only; bounded samples, never part of `value`) -------------
    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        extra = {}
        src = host if host is not None else frames   # pinned host frames after the e2e leg, else the device tensor

        def timed(fn, reps):
            fn()
            torch.cuda.synchronize()
            t = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t) / reps

        # configs[0]: one 1000-frame video, reference CPU path vs 1 GPU.  GPU side: (a) the ctypes call with host frames,
        # (b) the C++ class mirror's main() sequence on files (the drop-in path a reference user runs): its own LM_TIMING line.
        try:
            m0 = min(1000, n)
            h0 = src[:m0] if host is not None else src[:m0].cpu().pin_memory()
            r0 = Results(m0, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, pinned=True)
            dt0 = timed(lambda: det.detect_batch(h0, bx[:m0], bs[:m0], bb[:m0], results=r0), 5)
            c0 = {"frames": m0, "gpu_host_frames_per_s": m0 / dt0, "gpu_ms_per_video": dt0 * 1e3,
                  "cpu_frames_per_s_1_thread": cpu["value"] if cpu else None, "cpu_s_per_video": (m0 / cpu["value"]) if cpu else None,
                  "note": "lm_detect_batch on one 1000-frame video in pinned host memory (H2D + D2H inside); cpu_baseline is the same 1000 frames on 1 thread"}
            try:
                import pathlib
                import tempfile

                from locomouse_cpp_b200.lmfiles import write_problem_files

                exe = os.path.join(ROOT, "locomouse_cpp_b200", "host", "locomouse_b200")
                with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
                    d = pathlib.Path(td)
                    write_problem_files(d, cfg, model, bkg, calib, h0.numpy(), bx[:m0], bs[:m0], bb[:m0], spec.side_h)
                    best = None
                    for _ in range(2):
                        t = time.perf_counter()
                        pr = subprocess.run([exe, "1", str(d / "config.yml"), str(d / "video.lmv"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                                             str(d / "calib.lmc"), "R", str(d)], capture_output=True, text=True, timeout=300,
                                            env=dict(os.environ, LM_DRIVER_REPEAT="2"))
                        wall0 = time.perf_counter() - t
                        tl = [ln for ln in pr.stdout.splitlines() if ln.startswith("LM_TIMING")]
                        if pr.returncode != 0 or not tl:
                            raise RuntimeError((pr.stdout + pr.stderr)[-300:])
                        kv = dict(x.split("=") for x in tl[-1].split()[1:])
                        cur = {k: float(v) for k, v in kv.items()}
                        cur["process_wall_s"] = wall0
                        if best is None or cur["loop_s"] < best["loop_s"]:
                            best = cur
                    c0["cpp_driver"] = dict(best, loop_frames_per_s=m0 / best["loop_s"],
                                            warm_loop_frames_per_s=(m0 / best["warm_loop_s"]) if best.get("warm_loop_s", -1) > 0 else None,
                                            whole_program_frames_per_s=m0 / best["process_wall_s"],
                                            note="host/locomouse_b200 (main.cpp's call sequence through the C++ class mirror) on files in /dev/shm: "
                                                 "load_s = reading the 680 MB video into page-locked memory + CUDA context, loop_s = the per-frame "
                                                 "loop (batched lm_detect_batch behind readFrame ... matchBottomSideCandidates) of the cold process, warm_loop_s = the same "
                                                 "loop run again on the same object (LM_DRIVER_REPEAT), export_s = output file")
            except Exception as ex:  # pragma: no cover
                c0["cpp_driver"] = {"error": repr(ex)[:300]}
            extra["config0"] = c0
        except Exception as ex:  # pragma: no cover
            extra["config0"] = {"error": repr(ex)[:300]}

        # throughput vs detection density: rho re-calibrated so that x0.25 / x1 / x4 of the default fraction of pixels score > 0
        try:
            md = n   # the whole resident video: a short run would measure pipeline fill / drain, not the steady state
            dens = []
            for mult in (0.25, 1.0, 4.0):
                tf = (0.012 * mult, 0.012 * mult, 0.02 * mult)
                _c, model_d, _b, _k, _f, _x, _s, _y = synth.make_problem(spec, 8, seed=1000, target_frac=tf)
                det.set_model(model_d)
                if src.is_cuda:
                    fd = src[:md]
                else:
                    fd = src[:md].to(dev)
                rd = det.detect_batch(fd, bx[:md], bs[:md], bb[:md], allow_overflow=True)
                dtd = timed(lambda: det.detect_batch(fd, bx[:md], bs[:md], bb[:md], allow_overflow=True), 3)
                dens.append({"target_fraction_x": mult, "frames_per_s": md / dtd, "positives_per_frame": float(det.info("positives")) / subb,
                             "sparse_patches_per_frame": float(det.info("sparse_tasks")) / subb,
                             "candidates_per_frame": float(rd.n_bottom.sum() + rd.n_side.sum()) / md,
                             "overflow_frames": int((rd.flags != 0).sum())})
                del fd
            det.set_model(model)
            extra["density_sweep"] = {"frames": md, "points": dens,
                                      "note": "resident frames; the screen's exact pass and the NMS lists grow with the fraction of positive pixels "
                                              "(x1 = the benchmarked calibration: 1.2 % paw / snout, 2 % tail)"}
        except Exception as ex:  # pragma: no cover
            extra["density_sweep"] = {"error": repr(ex)[:300]}

        # configs[4]: 2x-upsampled frames (800 x 3400), six 60 x 60 templates
        try:
            det.close()
            det = None
            frames = None
            host5 = None
            torch.cuda.empty_cache()
            spec5 = synth.SynthSpec(scale=2, cand_cap=128, match_cap=512)
            cfg5, model5, bkg5, calib5, _, _, _, _ = synth.make_problem(spec5, 8, seed=1000)
            m5 = 1024
            fr5, bx5, bs5, bb5 = synth.make_video(spec5, m5, 1000, dev, bkg5)
            det5 = Detector(cfg5, model5, bkg5, calib5, device=local)
            det5.detect_batch(fr5, bx5, bs5, bb5, allow_overflow=True)
            dt5 = timed(lambda: det5.detect_batch(fr5, bx5, bs5, bb5, allow_overflow=True), 3)
            fma5 = algorithmic_fma_per_frame(cfg5, model5)
            det5.set_option("streams", 1)
            det5.detect_batch(fr5, bx5, bs5, bb5, allow_overflow=True)
            det5.detect_batch(fr5, bx5, bs5, bb5, allow_overflow=True)
            tm5, _ = det5.last_timing()
            ms5 = det5.info("ms_screen")
            tp = float(peaks.get("bf16_tflops", 1590.0))
            extra["config4_2x_60x60"] = {
                "frames": m5, "frame": [cfg5.vid_rows, cfg5.vid_cols], "templates": "6 x 60x60 f32", "frames_per_s": m5 / dt5,
                "screen_active": int(det5.info("screen_active")), "algorithmic_gflop_per_frame": 2.0 * fma5 / 1e9,
                "whole_path_algorithmic_tflops": 2.0 * fma5 * m5 / dt5 / 1e12,
                "screen_kernel_ms_serial": ms5, "screen_kernel_algorithmic_tflops": 2.0 * fma5 * m5 / (ms5 * 1e-3) / 1e12 if ms5 > 0 else None,
                "screen_kernel_frac_of_bf16_peak": (2.0 * fma5 * m5 / (ms5 * 1e-3) / 1e12 / tp) if ms5 > 0 else None,
                "corr_stage_ms_serial": tm5["corr"], "fp32_fma_bound_frames_per_s": fp32_nominal * 1e12 / (2.0 * fma5),
                "note": "contraction-bound stress: 16x the FMAs of config 1 per frame; the exact FP32 path is bounded by fp32_fma_bound_frames_per_s, "
                        "the tensor-core screen decides the same outputs (bit-exact parity: tests/test_gpu_screen.py::test_screen_config5_upsampled_60x60)"}
            det5.close()
            del fr5
        except Exception as ex:  # pragma: no cover
            extra["config4_2x_60x60"] = {"error": repr(ex)[:300]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8+f32" if screen_on else "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": n, "method": "LocoMouse_TM",
                           "frame": [cfg.vid_rows, cfg.vid_cols], "boxes": [cfg.bb_w, cfg.bb_h_bottom, cfg.bb_h_side],
                           "templates": "6 x 30x30 f32",
                           "accumulation": ("int8 tcgen05 screen (exact integer) + fp32 FFMA re-evaluation in oracle tap order (bit-exact)"
                                            if screen_on else "fp32 FFMA, oracle tap order (bit-exact)"),
                           "parallelism": f"frame-range dp{world} (one 10k-frame video per GPU, no data-path collective)",
                           "l2": f"inputs {n * 680000 / 1e9:.1f} GB per step > 126 MB L2, no flush needed",
                           "subbatch": subb},
                "timing": {"wall_ms_per_step": wall / args.steps * 1e3, "device_event_ms_per_step": dev_ms / args.steps,
                           "stage_ms_per_step_serial": {k: v / args.steps for k, v in stage.items()},
                           "streams": n_streams, "note": "value/wall/device_event: overlapped multi-stream pipeline; stage_ms_per_step_serial and the roofline "
                                   "launch times: the same steps with the library option streams=1 (kernels strictly serial)"},
                "clocks": sampler.summary(), "gpu_launches": int(launches), "overflow_frames": overflow,
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "pass1_tm_de": pass1, "cost_builders": costs, "other_configs": extra}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
