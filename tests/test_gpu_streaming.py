"""A video longer than max_resident_bytes is read, decoded and tracked in windows (LocoMouse_class.cpp useWindow): pass 1 runs
window by window, a batch_frames chunk never crosses a window, and the first chunk of a window gets the previous window's
last frame.  Every output file must equal, byte for byte, what the same inputs give in one window (the default budget):
for the three methods with pass 1 on the device and side L, with a location_prior (whose cost builders carry a one-frame
halo across every chunk boundary), for LMV, Y800, MPNG and FFV1 sources, in guard mode, for the warm loop
(LM_DRIVER_REPEAT) and through locomouse_b200_batch with one and two workers."""
import os
import subprocess

import numpy as np
import pytest

from locomouse_cpp_b200 import synth

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

N = 300
BATCH = 16
BUDGET_FRAMES = 40          # max_resident_bytes = 40 frames -> windows of 32 frames (a multiple of batch_frames)
W = 32
METHODS = {"0": "base", "1": "TM", "2": "TM_DE"}
PRIOR = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
         (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0), (0.95, 0.5, 0.6, 0.5, 1.0, 0.0, 1.0)]
PRIOR_CFG = ("location_prior: [" + ", ".join(repr(float(v)) for r in PRIOR for v in r) + "]\n"
             "max_displacement_bottom: 40\nmax_displacement_side: 25\n")


def _drivers():
    from test_host_cpp import _build_driver

    single = _build_driver()
    return single, os.path.join(os.path.dirname(single), "locomouse_b200_batch")


def _pass1_cfg(d, method, spec, cfg):
    """Configuration that makes pass 1 run on the device for `method`."""
    if method == "0":
        return "pass1_integer_sums: 1\n"
    if method == "1":
        y, x = np.mgrid[-5:6, -5:6]
        disk = ((x * x + y * y) <= 5.5 ** 2).astype(np.float64)
        fs = cv2.FileStorage(str(d / "diskfilter.yml"), cv2.FILE_STORAGE_WRITE)
        fs.write("H", (disk / disk.sum()).astype(np.float32))
        fs.release()
        return (f"pass1_integer_sums: 1\nbw_threshold_bottom: 40\nbw_threshold_side: 40\nmin_pixel_count: 25\nzero_col_pre: 0\n"
                f"zero_col_post: {cfg.n_cols}\nzero_row_pre: 0\nzero_row_post: {spec.side_h}\ndisk_filter_file: {d / 'diskfilter.yml'}\n")
    return ""


def _problem(d, method, source, prior, n=N):
    """Problem files in d, the video as `source`; returns (video path, frame bytes)."""
    from _ffv1_avi import write_cv2_ffv1
    from _png_avi import write_cv2_avi
    from test_host_cpp import write_problem_files

    spec = synth.SynthSpec(method=METHODS[method], flip=True)
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=1000, device="cuda")
    frames = frames.cpu().numpy()
    extra = f"batch_frames: {BATCH}\n" + _pass1_cfg(d, method, spec, cfg) + (PRIOR_CFG if prior else "")
    write_problem_files(d, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, extra_cfg=extra, with_boxes=False)
    video = d / "video.lmv"
    if source == "ffv1":
        video = d / "video.avi"
        assert np.array_equal(write_cv2_ffv1(cv2, video, frames), frames)
    elif source in ("y800", "mpng"):
        video = d / "video.avi"
        assert np.array_equal(write_cv2_avi(cv2, video, frames, source.upper()), frames)
    return video, frames.shape[1] * frames.shape[2]


def _timing(stdout):
    line = [ln for ln in stdout.splitlines() if ln.startswith("LM_TIMING")][-1]
    return {k: float(v) for k, v in (x.split("=") for x in line.split()[1:])}


def _files(out):
    return {f: (out / f).read_bytes() for f in sorted(os.listdir(out)) if f != "batch_summary.tsv"}


def _run(exe, d, method, video, budget, name, env=None):
    """locomouse_b200 with max_resident_bytes = budget (None: the default) into d/name; returns (files, LM_TIMING)."""
    cfg = d / f"config_{name}.yml"
    cfg.write_text((d / "config.yml").read_text() + (f"max_resident_bytes: {budget}\n" if budget else ""))
    out = d / name
    out.mkdir()
    p = subprocess.run([exe, method, str(cfg), str(video), str(d / "bkg.lmi"), str(d / "model.lmm"), str(d / "calib.lmc"), "L", str(out)],
                       capture_output=True, text=True, env=None if env is None else dict(os.environ, **env))
    assert p.returncode == 0, p.stdout + p.stderr
    return _files(out), _timing(p.stdout)


def _check_streamed(d, method, video, fsz, prior, env=None):
    exe, _ = _drivers()
    want, t1 = _run(exe, d, method, video, None, "one_window")
    got, tw = _run(exe, d, method, video, BUDGET_FRAMES * fsz, "windows", env)
    assert t1["windows"] == 1 and tw["windows"] > 1
    assert tw["resident_bytes"] <= 3 * W * fsz + fsz, tw
    assert t1["resident_bytes"] >= N * fsz
    assert "output_video.lmo" in want and got.keys() == want.keys()
    for f in want:
        assert got[f] == want[f], f"{f} differs when the video is streamed in {tw['windows']:.0f} windows"
    if prior:
        assert b"paw_tracks0" in want["output_video.yml"] and "costs_video.lmo" in want
    return tw


@pytest.mark.parametrize("prior", [False, True], ids=["no_prior", "location_prior"])
@pytest.mark.parametrize("method", ["0", "1", "2"])
def test_streamed_raw_video_equals_one_window(tmp_path, method, prior):
    video, fsz = _problem(tmp_path, method, "lmv", prior)
    tw = _check_streamed(tmp_path, method, video, fsz, prior)
    assert tw["windows"] == -(-N // W)


@pytest.mark.parametrize("source", ["y800", "mpng", "ffv1"])
def test_streamed_avi_sources_equal_one_window(tmp_path, source):
    video, fsz = _problem(tmp_path, "2", source, True)
    tw = _check_streamed(tmp_path, "2", video, fsz, True)
    if source == "ffv1":
        # windows end just before a keyframe, and the cv2 writer's GOP does not divide the 32-frame window
        assert tw["windows"] > -(-N // W)


def test_streamed_ffv1_in_guard_mode_and_warm_loop(tmp_path):
    video, fsz = _problem(tmp_path, "1", "ffv1", True)
    tw = _check_streamed(tmp_path, "1", video, fsz, True, env={"LM_GUARD": "1", "LM_DRIVER_REPEAT": "1"})
    assert tw["guard_violations"] == 0
    assert tw["warm_loop_s"] > 0


def test_batch_driver_streams_like_the_single_driver(tmp_path):
    """locomouse_b200_batch on a list of long videos with a small budget: the files of the single driver, byte for byte, with
    one and two workers."""
    from _ffv1_avi import write_cv2_ffv1
    from _png_avi import write_cv2_avi
    from test_host_cpp import write_problem_files

    single, batch = _drivers()
    spec = synth.SynthSpec(method="TM_DE", flip=True)
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 8, seed=1000)
    fsz = cfg.vid_rows * cfg.vid_cols
    write_problem_files(tmp_path, cfg, model, bkg, calib, frames.numpy(), bx, bs, bb, spec.side_h, with_boxes=False,
                        extra_cfg=f"batch_frames: {BATCH}\n" + PRIOR_CFG + f"max_resident_bytes: {BUDGET_FRAMES * fsz}\n")
    vids = tmp_path / "videos"
    vids.mkdir()
    lines = []
    for i, (n, kind) in enumerate([(N, "lmv"), (150, "ffv1"), (70, "y800"), (20, "lmv")]):
        b = synth.make_background(spec, 7000 + i)
        fr = synth.make_video(spec, n, 7000 + i, "cuda", b)[0].cpu().numpy()
        with open(vids / f"bkg{i}.lmi", "wb") as f:
            f.write(b"LMI1" + np.array(b.shape, "<i4").tobytes() + np.ascontiguousarray(b, np.uint8).tobytes())
        name = f"trial{i}." + ("lmv" if kind == "lmv" else "avi")
        if kind == "lmv":
            with open(vids / name, "wb") as f:
                f.write(b"LMV1" + np.array(fr.shape, "<i4").tobytes() + fr.tobytes())
        elif kind == "ffv1":
            assert np.array_equal(write_cv2_ffv1(cv2, vids / name, fr), fr)
        else:
            assert np.array_equal(write_cv2_avi(cv2, vids / name, fr, "Y800"), fr)
        lines.append((f"videos/{name}", f"videos/bkg{i}.lmi"))
    (tmp_path / "list.tsv").write_text("".join(f"{v}\t{b}\n" for v, b in lines))
    want = tmp_path / "single"
    want.mkdir()
    for v, b in lines:
        p = subprocess.run([single, "2", str(tmp_path / "config.yml"), str(tmp_path / v), str(tmp_path / b), str(tmp_path / "model.lmm"),
                            str(tmp_path / "calib.lmc"), "L", str(want)], capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
    assert _timing(p.stdout)["windows"] == 1   # the 20-frame video fits in one window
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    for workers in (1, 2):
        cfgw = tmp_path / f"config_w{workers}.yml"
        cfgw.write_text((tmp_path / "config.yml").read_text() + f"batch_workers_per_gpu: {workers}\n")
        out = tmp_path / f"batch{workers}"
        out.mkdir()
        p = subprocess.run([batch, "2", str(cfgw), str(tmp_path / "list.tsv"), str(tmp_path / "model.lmm"), str(tmp_path / "calib.lmc"), "L",
                            str(out)], capture_output=True, text=True, env=env)
        assert p.returncode == 0, p.stdout + p.stderr
        rows = [r.split("\t") for r in (out / "batch_summary.tsv").read_text().splitlines()[1:]]
        assert [r[2] for r in rows] == ["ok"] * len(lines)
        assert _files(out) == _files(want), f"{workers} worker(s)"
