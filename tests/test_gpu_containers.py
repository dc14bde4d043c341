"""Matroska and QuickTime / MP4 video on the device (host/lm_containers.hpp feeding the unchanged device path):
- lm_decode_png / lm_decode_ffv1 on chunks indexed from MKV / MOV / MP4 equal cv2.VideoCapture + extractChannel(0);
- locomouse_b200 on each container writes output_<stem>.yml and the candidates file byte-identical to its output on the Y800 AVI
  of the frames VideoCapture reads, once in guard mode with no guard byte touched;
- an FFV1 Matroska video streamed through several windows gives the bytes of one window;
- locomouse_b200_batch on a list mixing .avi, .mkv and .mov trials writes each video's files as the single driver does.
Needs a B200: pytest -m gpu."""
import os
import subprocess

import numpy as np
import pytest

from _containers import box, mkv, mov, write_cv2
from _ffv1_avi import Encoder, read_avi_ffv1
from _png_avi import capture, read_avi_png, write_cv2_avi
from locomouse_cpp_b200 import synth
from test_gpu_png_ingest import _detector

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

SOURCES = [("mkv", "FFV1"), ("mkv", "png "), ("mkv", "Y800"), ("mov", "png "), ("mov", "FFV1"), ("mov", "Y800"), ("mp4", "png ")]


def _frames(seed, n, h, w, colour):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = rng.integers(0, 256, (h, w, 3) if colour else (h, w), dtype=np.uint8)
    return np.stack([np.roll(base, 3 * i, axis=1) + rng.integers(0, 3, base.shape, dtype=np.uint8) for i in range(n)])


@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("ext,fourcc", [s for s in SOURCES if s[1] != "Y800"], ids=[f"{e}-{f.strip()}" for e, f in SOURCES if f != "Y800"])
def test_device_decode_of_indexed_chunks(tmp_path, ext, fourcc, colour):
    path = tmp_path / f"v.{ext}"
    want = write_cv2(cv2, path, _frames(len(ext) + colour, 30, 40, 64, colour), fourcc)
    det = _detector(40, 64)
    if fourcc == "FFV1":
        ex, payload, offs, _ = read_avi_ffv1(path)
        got = det.decode_ffv1(ex, payload, offs)
    else:
        payload, offs, _ = read_avi_png(path)
        got = det.decode_png(payload, offs)
    assert np.array_equal(got.cpu().numpy(), want)


def test_device_decode_of_hand_written_containers(tmp_path):
    """FFV1 with a GOP in an MKV of unknown-size clusters and in a MOV whose record is in 'glbl'; PNG in an mp4v MP4."""
    from _containers import esds_png, png_frames

    g = _frames(5, 26, 24, 40, False)
    rec, fr = Encoder(False, slices=(2, 2), gop=7).encode(g)
    (tmp_path / "a.mkv").write_bytes(mkv(fr, "V_FFV1", 40, 24, private=rec, unknown_sizes=True, block_group=True, audio_first=True))
    (tmp_path / "b.mov").write_bytes(mov(fr, b"FFV1", 40, 24, children=box(b"glbl", rec), chunks=[9, 9, 8], co64=True, moov_first=True))
    c = _frames(6, 10, 24, 40, True)
    (tmp_path / "c.mp4").write_bytes(mov(png_frames(cv2, c), b"mp4v", 40, 24, children=esds_png(), mp4=True, chunks=[3, 7]))
    det = _detector(24, 40)
    for name in ("a.mkv", "b.mov"):
        assert np.array_equal(capture(cv2, tmp_path / name), g)
        ex, payload, offs, _ = read_avi_ffv1(tmp_path / name)
        assert np.array_equal(det.decode_ffv1(ex, payload, offs).cpu().numpy(), g), name
    assert np.array_equal(capture(cv2, tmp_path / "c.mp4"), c[..., 0])
    payload, offs, _ = read_avi_png(tmp_path / "c.mp4")
    assert np.array_equal(det.decode_png(payload, offs).cpu().numpy(), c[..., 0])


def _timing(stdout):
    line = [ln for ln in stdout.splitlines() if ln.startswith("LM_TIMING")][-1]
    return {k: float(v) for k, v in (x.split("=") for x in line.split()[1:])}


def _drive(exe, d, method, video, out, env=None):
    out.mkdir()
    p = subprocess.run([exe, method, str(d / "config.yml"), str(video), str(d / "bkg.lmi"), str(d / "model.lmm"), str(d / "calib.lmc"), "R",
                        str(out)], capture_output=True, text=True, env=None if env is None else dict(os.environ, **env))
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


def test_driver_output_on_every_container_equals_y800_avi(tmp_path):
    """locomouse_b200 (method 2, a location prior so the tracker runs) on each container: output_video.yml and output_video.lmo
    byte-identical to its output on the Y800 AVI of the frames VideoCapture reads from that container."""
    from test_host_cpp import _build_driver, write_problem_files
    from test_gpu_streaming import PRIOR_CFG

    exe = _build_driver()
    spec = synth.SynthSpec(method="TM_DE")
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    frames = frames.numpy()
    write_problem_files(tmp_path, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, with_boxes=False,
                        extra_cfg="batch_frames: 16\n" + PRIOR_CFG)
    for i, (ext, fourcc) in enumerate(SOURCES):
        d = tmp_path / f"{ext}_{fourcc.strip()}"
        d.mkdir()
        got = write_cv2(cv2, d / f"video.{ext}", frames, fourcc)
        assert got.shape == frames.shape
        assert np.array_equal(write_cv2_avi(cv2, d / "video.avi", got, "Y800"), got)
        env = {"LM_GUARD": "1"} if i == 0 else None
        t = _timing(_drive(exe, tmp_path, "2", d / f"video.{ext}", d / "container", env))
        _drive(exe, tmp_path, "2", d / "video.avi", d / "avi")
        if env:
            assert t["guard_violations"] == 0
        for f in ("output_video.yml", "output_video.lmo"):
            assert (d / "container" / f).read_bytes() == (d / "avi" / f).read_bytes(), f"{f} differs for .{ext} '{fourcc}'"
        assert b"paw_tracks0" in (d / "container" / "output_video.yml").read_bytes()


def test_streamed_ffv1_matroska_equals_one_window(tmp_path):
    """A 300-frame FFV1 Matroska video with a 40-frame budget streams through several windows that end before keyframes, in
    guard mode, and gives every output file of a one-window run byte for byte."""
    from test_gpu_streaming import _check_streamed, _problem

    _, fsz = _problem(tmp_path, "2", "lmv", True)
    n, rows, cols = np.frombuffer((tmp_path / "video.lmv").read_bytes()[4:16], "<i4")
    frames = np.fromfile(tmp_path / "video.lmv", np.uint8, offset=16).reshape(n, rows, cols)
    video = tmp_path / "video.mkv"
    assert np.array_equal(write_cv2(cv2, video, frames, "FFV1"), frames)
    tw = _check_streamed(tmp_path, "2", video, fsz, True, env={"LM_GUARD": "1"})
    assert tw["windows"] > 1 and tw["guard_violations"] == 0


def test_batch_driver_mixes_containers(tmp_path):
    """locomouse_b200_batch on .avi, .mkv and .mov trials: each video's files as the single driver writes them, every row ok."""
    from test_gpu_streaming import BATCH, PRIOR_CFG, _drivers, _files
    from test_host_cpp import write_problem_files

    single, batch = _drivers()
    spec = synth.SynthSpec(method="TM_DE", flip=True)
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 8, seed=1000)
    write_problem_files(tmp_path, cfg, model, bkg, calib, frames.numpy(), bx, bs, bb, spec.side_h, with_boxes=False,
                        extra_cfg=f"batch_frames: {BATCH}\n" + PRIOR_CFG)
    vids = tmp_path / "videos"
    vids.mkdir()
    lines = []
    for i, (n, ext, fourcc) in enumerate([(30, "avi", "FFV1"), (45, "mkv", "FFV1"), (20, "mov", "png "), (25, "mkv", "Y800"),
                                          (18, "mp4", "png "), (33, "mov", "FFV1"), (12, "avi", "Y800")]):
        b = synth.make_background(spec, 7100 + i)
        fr = synth.make_video(spec, n, 7100 + i, "cpu", b)[0].numpy()
        with open(vids / f"bkg{i}.lmi", "wb") as f:
            f.write(b"LMI1" + np.array(b.shape, "<i4").tobytes() + np.ascontiguousarray(b, np.uint8).tobytes())
        name = f"trial{i}.{ext}"
        assert np.array_equal(write_cv2(cv2, vids / name, fr, fourcc), fr)
        lines.append((f"videos/{name}", f"videos/bkg{i}.lmi"))
    (tmp_path / "list.tsv").write_text("".join(f"{v}\t{b}\n" for v, b in lines))
    want = tmp_path / "single"
    want.mkdir()
    for v, b in lines:
        p = subprocess.run([single, "2", str(tmp_path / "config.yml"), str(tmp_path / v), str(tmp_path / b), str(tmp_path / "model.lmm"),
                            str(tmp_path / "calib.lmc"), "L", str(want)], capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    out = tmp_path / "batch"
    out.mkdir()
    cfgw = tmp_path / "config_w2.yml"
    cfgw.write_text((tmp_path / "config.yml").read_text() + "batch_workers_per_gpu: 2\n")
    p = subprocess.run([batch, "2", str(cfgw), str(tmp_path / "list.tsv"), str(tmp_path / "model.lmm"), str(tmp_path / "calib.lmc"), "L", str(out)],
                       capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stdout + p.stderr
    rows = [r.split("\t") for r in (out / "batch_summary.tsv").read_text().splitlines()[1:]]
    assert [r[2] for r in rows] == ["ok"] * len(lines)
    got = _files(out)
    assert got.keys() == _files(want).keys() and all(f"output_trial{i}.yml" in got for i in range(len(lines)))
    assert got == _files(want)
