"""Long videos through locomouse_b200 in bounded memory (max_resident_bytes): wall time, LM_TIMING phases, windows and peak
resident bytes, and a byte-for-byte comparison of the output files.  Writes profiles/r07_stream.json (or --out).

Arms, each run --reps times alternating, medians reported:
  long      a seeded synthetic raw video of --frames frames at 400 x 1700 (LMV1, written to --dir on local disk), method 2
            (LocoMouse_TM_DE, pass 1 on the device), with the default budget (8 GiB) and with a quarter of it (2 GiB).
  config0   the 1000-frame video of the benchmark's configs[0] geometry with the default budget (one window: the path of a
            video that fits), beside the same run of --parent-exe (a locomouse_b200 built from an earlier commit) when given.
  ffv1      a --ffv1-frames FFV1-coded AVI (cv2.VideoWriter, GOP 12) in one window and in windows of --ffv1-window frames
            (batch_frames 128): every window is decoded twice, once for pass 1 and once for the frame loop.

    python tools/stream_check.py [--arms long,config0,ffv1] [--frames 40000] [--dir /tmp] [--reps 2] [--parent-exe PATH]

The arms named in --arms are (re)measured; the others are kept from an existing --out file.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import pathlib
import shutil
import signal
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
HOST = ROOT / "locomouse_cpp_b200" / "host"
GIB = 1 << 30


def log(*a):
    print(*a, flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def problem(d: pathlib.Path, extra_cfg: str):
    """Model, calibration, background and configuration of the synthetic TM_DE setup (pass 1 on the device) in d."""
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.lmfiles import write_problem_files

    spec = synth.SynthSpec(method="TM_DE")
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 8, seed=1000)
    write_problem_files(d, cfg, model, bkg, calib, frames.numpy(), bx, bs, bb, spec.side_h, with_boxes=False, extra_cfg=extra_cfg)
    (d / "video.lmv").unlink()
    return spec, bkg


def write_lmv(path: pathlib.Path, spec, bkg, n: int, seed: int, chunk: int = 500):
    """n frames of the synthetic mouse (rendered on the GPU from `seed`) as LMV1, written chunk by chunk."""
    import numpy as np

    from locomouse_cpp_b200 import synth

    cfg = spec.config()
    with open(path, "wb") as f:
        f.write(b"LMV1" + np.array([n, cfg.vid_rows, cfg.vid_cols], "<i4").tobytes())
        for s in range(0, n, chunk):
            fr = synth.make_video(spec, min(chunk, n - s), seed, "cuda", bkg, start_frame=s, total=n)[0]
            f.write(fr.cpu().numpy().tobytes())
    return cfg.vid_rows * cfg.vid_cols


def digest(out: pathlib.Path):
    return {f: hashlib.sha256((out / f).read_bytes()).hexdigest() for f in sorted(os.listdir(out))}


def run(exe, d: pathlib.Path, video: pathlib.Path, budget, tag: str):
    cfg = d / f"config_{tag}.yml"
    cfg.write_text((d / "config.yml").read_text() + (f"max_resident_bytes: {budget}\n" if budget else ""))
    out = d / f"out_{tag}"
    shutil.rmtree(out, ignore_errors=True)
    out.mkdir()
    t = time.perf_counter()
    p = subprocess.run([str(exe), "2", str(cfg), str(video), str(d / "bkg.lmi"), str(d / "model.lmm"), str(d / "calib.lmc"), "R", str(out)],
                       capture_output=True, text=True)
    wall = time.perf_counter() - t
    tl = [ln for ln in p.stdout.splitlines() if ln.startswith("LM_TIMING")]
    if p.returncode != 0 or not tl:
        raise RuntimeError(f"{tag}: {(p.stdout + p.stderr)[-600:]}")
    r = {k: float(v) for k, v in (x.split("=") for x in tl[-1].split()[1:])}
    r["wall_s"] = wall
    return r, digest(out)


def arms(exe_of, d, video, budgets, reps):
    """{tag: median LM_TIMING + wall} over reps alternating runs, and whether every run of every arm wrote the same files."""
    runs, digests = {t: [] for t in budgets}, set()
    for _ in range(reps):
        for tag, budget in budgets.items():
            r, dg = run(exe_of(tag), d, video, budget, tag)
            runs[tag].append(r)
            digests.add(json.dumps(dg, sort_keys=True))
            log(f"  {tag}: windows {r.get('windows', 1):.0f} wall {r['wall_s']:.2f} s pass1 {r['pass1_s']:.2f} s loop {r['loop_s']:.2f} s "
                f"resident {r.get('resident_bytes', float('nan')) / GIB:.2f} GiB")
    med = {t: {k: statistics.median(x[k] for x in v) for k in v[0]} for t, v in runs.items()}
    return med, len(digests) == 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=40000)
    ap.add_argument("--ffv1-frames", type=int, default=1000)
    ap.add_argument("--ffv1-window", type=int, default=256)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--dir", default=None, help="local disk for the long video (default: the system temporary directory)")
    ap.add_argument("--parent-exe", default=None)
    ap.add_argument("--arms", default="long,config0,ffv1")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r07_stream.json"))
    a = ap.parse_args()
    exe = HOST / "locomouse_b200"
    report = json.loads(pathlib.Path(a.out).read_text()) if os.path.exists(a.out) else {}
    gpu = gpu_info()
    todo = a.arms.split(",")
    signal.signal(signal.SIGTERM, lambda *_: sys.exit("terminated"))  # the finally below still removes the videos
    work = pathlib.Path(tempfile.mkdtemp(prefix="lm_stream_", dir=a.dir))
    try:
        spec, bkg = problem(work, "")
        fsz = spec.config().vid_rows * spec.config().vid_cols
        need = a.frames * fsz
    except BaseException:
        shutil.rmtree(work, ignore_errors=True)
        raise
    try:
        if "long" in todo:
            report["long"] = measure_long(a, exe, work, spec, bkg, fsz, need, gpu)
        if "config0" in todo:
            report["config0"] = measure_config0(a, exe, work, spec, bkg, gpu)
        if "ffv1" in todo:
            report["ffv1"] = measure_ffv1(a, exe, work, spec, bkg, fsz, gpu)
    finally:
        shutil.rmtree(work, ignore_errors=True)
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)
        log(json.dumps(report, indent=1)[:6000])


def measure_long(a, exe, work, spec, bkg, fsz, need, gpu):
    r = {"gpu": gpu, "frames": a.frames, "video_bytes": need}
    free = shutil.disk_usage(work).free
    r["dir"], r["disk_free_bytes"] = str(work), free
    if free < need + 4 * GIB:
        r["error"] = f"{free / GIB:.1f} GiB free, the {a.frames}-frame video needs {need / GIB:.1f} GiB: not measured"
        return r
    log(f"writing {a.frames} frames ({need / GIB:.1f} GiB) to {work}")
    t = time.perf_counter()
    write_lmv(work / "long.lmv", spec, bkg, a.frames, seed=4242)
    r["write_s"] = time.perf_counter() - t
    try:
        r["arms"], r["outputs_identical"] = arms(lambda tag: exe, work, work / "long.lmv", {"default_8GiB": None, "quarter_2GiB": 2 * GIB}, a.reps)
    finally:
        (work / "long.lmv").unlink()
    return r


def measure_config0(a, exe, work, spec, bkg, gpu):
    log("config0: 1000 frames, one window")
    write_lmv(work / "c0.lmv", spec, bkg, 1000, seed=1000)
    exe_of = lambda tag: exe if tag == "this" else pathlib.Path(a.parent_exe)
    budgets = {"this": None} | ({"parent": None} if a.parent_exe else {})
    med, same = arms(exe_of, work, work / "c0.lmv", budgets, max(a.reps, 3))
    return {"gpu": gpu, "frames": 1000, "arms": med, "outputs_identical": same}


def measure_ffv1(a, exe, work, spec, bkg, fsz, gpu):
    import cv2
    import numpy as np

    from _ffv1_avi import write_cv2_ffv1

    log(f"ffv1: {a.ffv1_frames} frames")
    fd = work / "ffv1"
    fd.mkdir()
    problem(fd, "batch_frames: 128\n")
    write_lmv(fd / "v.lmv", spec, bkg, a.ffv1_frames, seed=77)
    raw = np.fromfile(fd / "v.lmv", np.uint8, offset=16).reshape(a.ffv1_frames, spec.config().vid_rows, spec.config().vid_cols)
    assert np.array_equal(write_cv2_ffv1(cv2, fd / "v.avi", raw), raw)
    med, same = arms(lambda tag: exe, fd, fd / "v.avi", {"one_window": None, f"windows_{a.ffv1_window}": a.ffv1_window * fsz}, a.reps)
    return {"gpu": gpu, "frames": a.ffv1_frames, "arms": med, "outputs_identical": same, "file_bytes": os.path.getsize(fd / "v.avi")}


if __name__ == "__main__":
    main()
