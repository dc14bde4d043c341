"""FFV1-coded video ingest on one GPU: lm_decode_ffv1's rate, and compressed against raw end to end.

The benchmark's seeded synthetic video (synth.make_video, seed 1000, 10 000 frames of 400 x 1700 by default) is encoded by
cv2.VideoWriter with fourcc 'FFV1' (in parallel: every worker writes its own AVI of a slice of the frames that is a whole
number of GOPs, so the chunks and the record are what one writer would produce), and its chunks are read back by the host
reader (host/lm_media.hpp).  Measured, after a warm-up call of each:
  - decode kernels alone, payload resident in device memory (lm_get_info "ms_decode"): frames/s, GB/s in and out;
  - lm_decode_ffv1 from a page-locked host payload (wall clock of the call, pieces copied on the copy stream): frames/s;
  - end to end: page-locked compressed bytes -> lm_decode_ffv1 -> resident lm_detect_batch, against lm_detect_batch from
    page-locked raw frames, run alternately `--reps` times each; both paths' results are compared byte for byte.
Prints one JSON line (and writes it to --out).  Run: python tools/ffv1_ingest_check.py [--frames N] [--out FILE]"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

_FRAMES = None  # inherited by the encoder processes (fork)


def _encode(job):
    import cv2

    path, s, e = job
    h, w = _FRAMES.shape[1:]
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (w, h), False)
    for f in _FRAMES[s:e]:
        wr.write(f)
    wr.release()
    return path


def encode_ffv1(frames, tmp):
    """(record, payload uint8, offsets int64[n + 1]) of `frames` as FFV1 AVI chunks (OpenCV's writer: GOP 12)."""
    global _FRAMES
    from _ffv1_avi import read_avi_ffv1

    _FRAMES = frames
    n = frames.shape[0]
    workers = max(1, min(os.cpu_count() or 1, 64))
    step = ((n + workers - 1) // workers + 11) // 12 * 12
    jobs = [(os.path.join(tmp, f"part{k:03d}.avi"), s, min(n, s + step)) for k, s in enumerate(range(0, n, step))]
    with mp.get_context("fork").Pool(workers) as pool:
        pool.map(_encode, jobs)
    payloads, offs, base, rec = [], [np.zeros(1, np.int64)], 0, None
    for path, s, e in jobs:
        ex, p, o, dims = read_avi_ffv1(path)
        assert dims[0] == e - s and (rec is None or np.array_equal(ex, rec))
        rec = ex
        payloads.append(p)
        offs.append(o[1:] + base)
        base += int(o[-1])
        os.remove(path)
    return rec, np.concatenate(payloads), np.concatenate(offs)


def gpu_info():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip()
    except Exception as ex:  # pragma: no cover
        power = f"unavailable ({ex!r})"
    return name, power


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import Results

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, _, _, _, _ = synth.make_problem(spec, 8, seed=1000)
    dev_frames, bx, bs, bb = synth.make_video(spec, a.frames, 1000, "cuda:0", bkg)
    raw = torch.empty(tuple(dev_frames.shape), dtype=torch.uint8, pin_memory=True)
    raw.copy_(dev_frames)
    torch.cuda.synchronize()
    del dev_frames
    torch.cuda.empty_cache()
    n, fsz = raw.shape[0], raw.shape[1] * raw.shape[2]
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        rec, payload_np, offs = encode_ffv1(raw.numpy(), tmp)
        t_encode = time.perf_counter() - t0
    comp = int(offs[-1])
    payload = torch.from_numpy(payload_np).pin_memory()
    del payload_np
    det = Detector(cfg, model, bkg, calib, device=0)
    out = torch.empty(tuple(raw.shape), dtype=torch.uint8, device="cuda:0")

    # decode kernels alone, payload resident
    pdev = payload.cuda()
    det.decode_ffv1(rec, pdev, offs, out=out)
    assert torch.equal(out.cpu(), raw), "decoded frames differ from the raw frames"
    kern = []
    for _ in range(a.reps):
        det.decode_ffv1(rec, pdev, offs, out=out)
        kern.append(det.info("ms_decode"))
    del pdev
    torch.cuda.empty_cache()
    k_ms = float(np.median(kern))

    # lm_decode_ffv1 from page-locked host memory
    det.decode_ffv1(rec, payload, offs, out=out)
    host_ms = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        det.decode_ffv1(rec, payload, offs, out=out)
        host_ms.append((time.perf_counter() - t0) * 1e3)

    # end to end, alternating
    res_c = Results(n, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, pinned=True)
    res_r = Results(n, cfg.cand_cap, cfg.match_cap, cfg.n_tail_points, pinned=True)
    det.detect_batch(det.decode_ffv1(rec, payload, offs, out=out), bx, bs, bb, results=res_c)
    det.detect_batch(raw, bx, bs, bb, results=res_r)
    e2e_c, e2e_r = [], []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        det.detect_batch(det.decode_ffv1(rec, payload, offs, out=out), bx, bs, bb, results=res_c)
        e2e_c.append(n / (time.perf_counter() - t0))
        t0 = time.perf_counter()
        det.detect_batch(raw, bx, bs, bb, results=res_r)
        e2e_r.append(n / (time.perf_counter() - t0))
    equal = bool(np.array_equal(res_c.raw, res_r.raw))
    name, power = gpu_info()
    rnd = lambda v: [round(x) for x in v]
    rec = {
        "gpu": name, "power_limit": power, "frames": n, "frame_bytes": fsz, "encoder": "cv2.VideoWriter FFV1, grey",
        "encode_s": round(t_encode, 1), "compressed_bytes_per_frame": round(comp / n), "compression_ratio": round(n * fsz / comp, 3),
        "decode_kernel": {"ms": [round(x, 2) for x in kern], "frames_per_s": round(n / k_ms * 1e3), "gb_per_s_in": round(comp / k_ms / 1e6, 2),
                          "gb_per_s_out": round(n * fsz / k_ms / 1e6, 2)},
        "decode_from_pinned_host": {"ms": [round(x, 1) for x in host_ms], "frames_per_s": round(n / float(np.median(host_ms)) * 1e3)},
        "e2e_compressed_frames_per_s": rnd(e2e_c), "e2e_raw_frames_per_s": rnd(e2e_r),
        "e2e_compressed_median": round(float(np.median(e2e_c))), "e2e_raw_median": round(float(np.median(e2e_r))),
        "e2e_spread": {"compressed": round((max(e2e_c) - min(e2e_c)) / float(np.median(e2e_c)), 4),
                       "raw": round((max(e2e_r) - min(e2e_r)) / float(np.median(e2e_r)), 4)},
        "results_equal": equal, "bottom_candidates": int(res_r.n_bottom.sum()),
    }
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not equal:
        sys.exit(1)


if __name__ == "__main__":
    main()
