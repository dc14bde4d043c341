"""locomouse_b200_batch writes, for every video of its list, the same files as locomouse_b200 run on that video alone, byte for
byte: with one and three workers per GPU, on more than one GPU when there are several, and next to a video that fails."""
import os
import subprocess

import numpy as np
import pytest

from locomouse_cpp_b200 import synth

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "locomouse_cpp_b200", "host")
METHODS = {"0": "base", "1": "TM", "2": "TM_DE"}
# (frames, container, side): 1 frame, fewer than one sub-batch, more than batch_frames (4), both sides, PNG- and FFV1-coded AVI
VIDEOS = [(1, "lmv", "R"), (3, "lmv", "L"), (9, "y800", "R"), (13, "lmv", None), (6, "mpng", "L"), (7, "ffv1", "R"), (2, "y800", "L"),
          (70, "lmv", "R")]


def _build():
    if not os.path.exists(os.path.join(ROOT, "locomouse_cpp_b200", "liblocomouse_b200.so")):
        pytest.skip("CUDA library not built")
    p = subprocess.run(["make", "-C", HOST], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    return os.path.join(HOST, "locomouse_b200"), os.path.join(HOST, "locomouse_b200_batch")


def _session(d, method):
    """Shared model / calibration / configuration and eight videos with their own backgrounds.  Boxes come from the
    configuration (use_provided_bounding_box), so one configuration serves every video."""
    from _ffv1_avi import write_cv2_ffv1
    from _png_avi import write_cv2_avi
    from test_host_cpp import write_problem_files

    spec = synth.SynthSpec(method=METHODS[method])
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 8, seed=1000)
    write_problem_files(d, cfg, model, bkg, calib, frames.numpy(), bx, bs, bb, spec.side_h, with_boxes=False)
    x0 = int(bx[0]) - cfg.bb_w   # the box's bottom-right corner is origin + size (LocoMouse_class.cpp:545-567)
    boxes = (f"use_provided_bounding_box: 1\nbatch_frames: 4\n"
             f"bounding_box_bottom: [{x0}, {int(bb[0]) - cfg.bb_h_bottom}, {cfg.bb_w}, {cfg.bb_h_bottom}]\n"
             f"bounding_box_side: [{x0}, {int(bs[0]) - cfg.bb_h_side}, {cfg.bb_w}, {cfg.bb_h_side}]\n")
    base_cfg = (d / "config.yml").read_text() + boxes
    (d / "config.yml").write_text(base_cfg)
    vids = d / "videos"
    vids.mkdir()
    lines = []
    for i, (n, kind, side) in enumerate(VIDEOS):
        seed = 5000 + 31 * i
        b = synth.make_background(spec, seed)
        fr = synth.make_video(spec, n, seed, "cpu", b)[0].numpy()
        with open(vids / f"bkg{i}.lmi", "wb") as f:
            f.write(b"LMI1" + np.array(b.shape, "<i4").tobytes() + np.ascontiguousarray(b, np.uint8).tobytes())
        name = f"trial{i}." + ("lmv" if kind == "lmv" else "avi")
        if kind == "lmv":
            with open(vids / name, "wb") as f:
                f.write(b"LMV1" + np.array(fr.shape, "<i4").tobytes() + fr.tobytes())
        elif kind == "ffv1":
            assert np.array_equal(write_cv2_ffv1(cv2, vids / name, fr), fr)
        else:
            assert np.array_equal(write_cv2_avi(cv2, vids / name, fr, {"y800": "Y800", "mpng": "MPNG"}[kind]), fr)
        lines.append((f"videos/{name}", f"videos/bkg{i}.lmi", side))
    return base_cfg, lines


def _write_list(path, lines):
    path.write_text("# video\tbackground\tside\n" + "".join("\t".join(x for x in line if x) + "\n" for line in lines))


def _single(exe, d, method, lines, out):
    """locomouse_b200 on each video alone; returns {stem: stdout}."""
    out.mkdir()
    msgs = {}
    for video, bkg, side in lines:
        p = subprocess.run([exe, method, str(d / "config.yml"), str(d / video), str(d / bkg), str(d / "model.lmm"), str(d / "calib.lmc"),
                            side or "R", str(out)], capture_output=True, text=True)
        msgs[os.path.splitext(os.path.basename(video))[0]] = (p.returncode, p.stdout)
    return msgs


def _batch(exe, d, method, lst, out, workers, base_cfg, env=None):
    out.mkdir()
    cfg = d / f"config_w{workers}.yml"
    cfg.write_text(base_cfg + f"batch_workers_per_gpu: {workers}\n")
    p = subprocess.run([exe, method, str(cfg), str(lst), str(d / "model.lmm"), str(d / "calib.lmc"), "R", str(out)], capture_output=True,
                       text=True, env=env)
    rows = [r.split("\t") for r in (out / "batch_summary.tsv").read_text().splitlines()]
    assert rows[0][:3] == ["line", "video", "status"]
    return p, rows[1:]


def _files(out):
    return {f: (out / f).read_bytes() for f in sorted(os.listdir(out)) if f != "batch_summary.tsv"}


@pytest.mark.parametrize("method", ["0", "1", "2"])
def test_batch_outputs_equal_the_single_driver(tmp_path, method):
    single_exe, batch_exe = _build()
    base_cfg, lines = _session(tmp_path, method)
    lst = tmp_path / "list.tsv"
    _write_list(lst, lines)
    msgs = _single(single_exe, tmp_path, method, lines, tmp_path / "single")
    assert all(rc == 0 for rc, _ in msgs.values()), msgs
    want = _files(tmp_path / "single")
    assert len(want) >= len(lines)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    for workers in (1, 3):
        p, rows = _batch(batch_exe, tmp_path, method, lst, tmp_path / f"batch{workers}", workers, base_cfg, env)
        assert p.returncode == 0, p.stdout + p.stderr
        assert [r[2] for r in rows] == ["ok"] * len(lines)
        assert [int(r[0]) for r in rows] == list(range(2, 2 + len(lines)))   # list line numbers (line 1 is a comment)
        assert [int(r[4]) for r in rows] == [n for n, _, _ in VIDEOS]
        got = _files(tmp_path / f"batch{workers}")
        assert got.keys() == want.keys()
        for f in want:
            assert got[f] == want[f], f"{f} differs with {workers} worker(s) per GPU"
    import torch

    if torch.cuda.device_count() > 1:
        p, rows = _batch(batch_exe, tmp_path, method, lst, tmp_path / "all_gpus", 1, base_cfg)
        assert p.returncode == 0, p.stdout + p.stderr
        assert len({r[3] for r in rows}) > 1, "the videos should spread over the GPUs"
        got = _files(tmp_path / "all_gpus")
        assert got == want


def test_a_failing_video_is_reported_and_the_others_go_on(tmp_path):
    single_exe, batch_exe = _build()
    base_cfg, lines = _session(tmp_path, "1")
    # a Y800 AVI cut inside its last frame
    src = tmp_path / lines[2][0]
    data = src.read_bytes()
    bad = tmp_path / "videos" / "broken.avi"
    bad.write_bytes(data[: len(data) - 3000])
    lines = lines[:3] + [("videos/broken.avi", lines[2][1], "R")] + lines[3:5]
    lst = tmp_path / "list.tsv"
    _write_list(lst, lines)
    msgs = _single(single_exe, tmp_path, "1", lines, tmp_path / "single")
    rc, out = msgs["broken"]
    assert rc == 1
    message = next(line for line in out.splitlines() if line.startswith("Runtime Error"))
    assert "truncated frame" in message
    p, rows = _batch(batch_exe, tmp_path, "1", lst, tmp_path / "batch", 2, base_cfg)
    assert p.returncode == 1
    assert [r[2] for r in rows] == ["ok", "ok", "ok", "runtime", "ok", "ok"]
    assert rows[3][1].endswith("broken.avi") and rows[3][-1] == message
    assert _files(tmp_path / "batch") == _files(tmp_path / "single")
