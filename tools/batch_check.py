"""A session of config-0 videos through locomouse_b200 (once per video, what users ran before) and locomouse_b200_batch
(one GPU with 1 / 2 / 4 workers, then every GPU): whole-run seconds, videos/s, frames/s, the per-phase sums of the batch
summaries, and a byte-for-byte comparison of every output file across all arms.  Writes profiles/r06_batch.json (or --out).

Inputs: --videos seeded 400 x 1700 Y800 AVIs of --frames frames (the benchmark's synthetic mouse, each video its own seed and
background, written as PNG files), model and calibration of config 0 (method 1, LocoMouse_TM), boxes from the configuration
(use_provided_bounding_box: one configuration serves the whole session).  The FFV1 set holds the same videos as FFV1-coded
AVIs (--ffv1-videos distinct encodings, repeated under new names up to --videos).  Files are read from the page cache after
being written; caches are not dropped.

    python tools/batch_check.py --set y800 [--videos 32] [--frames 1000] [--reps 3] [--workers 1,2,4]
    python tools/batch_check.py --set ffv1 [--ffv1-workers 1,2,4,8]      (adds its arms to the same report)
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import pathlib
import shutil
import statistics
import subprocess
import sys
import tempfile
import time


ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
HOST = ROOT / "locomouse_cpp_b200" / "host"


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def log(*a):
    print(*a, flush=True)


def make_session(d: pathlib.Path, which: str, n_videos: int, n_frames: int, ffv1_distinct: int):
    import cv2
    import torch

    from _ffv1_avi import write_cv2_ffv1
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.lmfiles import write_problem_files

    spec = synth.SynthSpec(method="TM")
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 8, seed=1000)
    write_problem_files(d, cfg, model, bkg, calib, frames.numpy(), bx, bs, bb, spec.side_h, with_boxes=False)
    x0 = int(bx[0]) - cfg.bb_w
    cfg_text = (d / "config.yml").read_text() + (
        f"use_provided_bounding_box: 1\nbounding_box_bottom: [{x0}, {int(bb[0]) - cfg.bb_h_bottom}, {cfg.bb_w}, {cfg.bb_h_bottom}]\n"
        f"bounding_box_side: [{x0}, {int(bs[0]) - cfg.bb_h_side}, {cfg.bb_w}, {cfg.bb_h_side}]\n")
    (d / "config.yml").write_text(cfg_text)
    (d / which).mkdir()
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    items = []
    for i in range(n_videos):
        name, bname = f"trial{i:02d}.avi", f"bkg{i:02d}.png"
        items.append((name, bname))
        if which == "ffv1" and i >= ffv1_distinct:   # the FFV1 set repeats its distinct encodings under new names
            shutil.copy(d / which / f"trial{i % ffv1_distinct:02d}.avi", d / which / name)
            shutil.copy(d / which / f"bkg{i % ffv1_distinct:02d}.png", d / which / bname)
            continue
        seed = 7000 + 101 * i
        b = synth.make_background(spec, seed)
        cv2.imwrite(str(d / which / bname), b)
        fr = synth.make_video(spec, n_frames, seed, dev, b)[0].cpu().numpy()
        if which == "ffv1":
            write_cv2_ffv1(cv2, d / which / name, fr)
        else:
            wr = cv2.VideoWriter(str(d / which / name), cv2.VideoWriter_fourcc(*"Y800"), 30.0, (fr.shape[2], fr.shape[1]), False)
            for f in fr:
                wr.write(f)
            wr.release()
        log(f"wrote {which}/{name}")
    (d / which / "list.tsv").write_text("".join(f"{v}\t{b}\n" for v, b in items))
    return cfg_text, items


def digest(out: pathlib.Path):
    return {f.name: hashlib.sha256(f.read_bytes()).hexdigest() for f in sorted(out.iterdir()) if f.name != "batch_summary.tsv"}


def run_single(d, s, items, out):
    out.mkdir(parents=True)
    exe = str(HOST / "locomouse_b200")
    t = time.perf_counter()
    for v, b in items:
        p = subprocess.run([exe, "1", str(d / "config.yml"), str(d / s / v), str(d / s / b), str(d / "model.lmm"), str(d / "calib.lmc"), "R", str(out)],
                           capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError(p.stdout[-500:])
    return time.perf_counter() - t


def run_batch(d, s, cfg_text, workers, out, env=None):
    out.mkdir(parents=True)
    cfg = d / f"config_w{workers}.yml"
    cfg.write_text(cfg_text + f"batch_workers_per_gpu: {workers}\n")
    t = time.perf_counter()
    p = subprocess.run([str(HOST / "locomouse_b200_batch"), "1", str(cfg), str(d / s / "list.tsv"), str(d / "model.lmm"), str(d / "calib.lmc"), "R",
                        str(out)], capture_output=True, text=True, env=env)
    wall = time.perf_counter() - t
    if p.returncode != 0:
        raise RuntimeError(p.stdout[-1500:])
    rows = [r.split("\t") for r in (out / "batch_summary.tsv").read_text().splitlines()[1:]]
    phases = {k: sum(float(r[5 + j]) for r in rows) for j, k in enumerate(("load_s", "pass1_s", "loop_s", "tracks_s", "export_s"))}
    return wall, phases, sorted({int(r[3]) for r in rows})


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--set", choices=("y800", "ffv1"), default="y800")
    ap.add_argument("--videos", type=int, default=32)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workers", default="1,2,4")
    ap.add_argument("--ffv1-workers", default="1,2,4,8")
    ap.add_argument("--ffv1-videos", type=int, default=2, help="distinct FFV1 encodings (cv2's encoder is slow); the rest are copies")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_batch.json"))
    a = ap.parse_args()
    one_gpu = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    import torch

    n_gpus = torch.cuda.device_count()
    outp = pathlib.Path(a.out)
    res = json.loads(outp.read_text()) if outp.exists() else {"arms": {}}
    total_frames = a.videos * a.frames
    info = {"gpus": gpu_info(), "gpus_visible": n_gpus, "videos": a.videos, "frames_per_video": a.frames, "method": 1}
    res[a.set] = dict(info, inputs=(
        f"{a.videos} seeded 400x1700 AVIs of {a.frames} frames (config-0 geometry, method 1, the benchmark's synthetic mouse, each video "
        "its own seed and PNG background; boxes fixed by use_provided_bounding_box so one configuration serves all). "
        + ("Y800 (raw)." if a.set == "y800" else f"FFV1 written by cv2: {min(a.ffv1_videos, a.videos)} distinct encodings repeated under new names.")
        + " Files in /dev/shm, read from the page cache after being written (caches not dropped)."))
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
        d = pathlib.Path(td)
        t = time.perf_counter()
        cfg_text, items = make_session(d, a.set, a.videos, a.frames, min(a.ffv1_videos, a.videos))
        res[a.set]["setup_s"] = time.perf_counter() - t
        arms = res["arms"]

        def record(key, walls, phases=None, extra=None):
            m = statistics.median(walls)
            arms[key] = dict({"wall_s": spread(walls), "videos_per_s": a.videos / m, "frames_per_s": total_frames / m, "phase_sums_s": phases},
                             **(extra or {}))
            log(key, json.dumps(arms[key]))
            outp.parent.mkdir(parents=True, exist_ok=True)
            outp.write_text(json.dumps(res, indent=1) + "\n")

        if a.set == "y800":
            workers = [int(x) for x in a.workers.split(",")]
            walls = {"a_single": []}
            walls.update({f"b_batch_1gpu_w{w}": [] for w in workers})
            phases = {}
            ref = None
            for rep in range(a.reps):   # (a) and (b) alternated
                out = d / "out_a"
                walls["a_single"].append(run_single(d, "y800", items, out))
                ref = ref or digest(out)
                assert digest(out) == ref, "arm (a) differs between repetitions"
                shutil.rmtree(out)
                log(f"rep {rep} a_single {walls['a_single'][-1]:.2f} s")
                for w in workers:
                    out = d / "out_b"
                    wall, ph, _ = run_batch(d, "y800", cfg_text, w, out, one_gpu)
                    walls[f"b_batch_1gpu_w{w}"].append(wall)
                    phases[f"b_batch_1gpu_w{w}"] = ph
                    assert digest(out) == ref, f"batch with {w} workers differs from the single driver"
                    shutil.rmtree(out)
                    log(f"rep {rep} batch w{w} {wall:.2f} s")
            for k, xs in walls.items():
                record(k, xs, phases.get(k))
            if n_gpus > 1:
                xs, ph, devs = [], None, None
                for rep in range(a.reps):
                    out = d / "out_c"
                    wall, ph, devs = run_batch(d, "y800", cfg_text, max(workers), out)
                    xs.append(wall)
                    assert digest(out) == ref, "batch on all GPUs differs from the single driver"
                    shutil.rmtree(out)
                record("c_batch_all_gpus", xs, ph, {"devices_used": devs, "workers_per_gpu": max(workers)})
        else:
            out = d / "out_f_single"
            wall = run_single(d, "ffv1", items, out)
            ref = digest(out)
            record("ffv1_a_single", [wall])
            for w in [int(x) for x in a.ffv1_workers.split(",")]:
                out = d / f"out_f{w}"
                wall, ph, _ = run_batch(d, "ffv1", cfg_text, w, out, one_gpu)
                assert digest(out) == ref, f"FFV1 batch with {w} workers differs from the single driver"
                record(f"ffv1_batch_1gpu_w{w}", [wall], ph)
        res[a.set]["outputs_identical"] = True
    outp.write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
