"""MPEG-4 Part 2 on the device (lm_decode_mpeg4, k_mpeg4.cu):
- the device decode equals the CPU decode (mpeg4_format.h) and cv2.VideoCapture's channel 0 on cv2-written 'XVID' / 'mp4v'
  video in AVI, MP4 and Matroska, grey and colour, 400 x 1700 included;
- the test encoder's random-syntax streams decode on the device as VideoCapture reads them;
- a 2 100-frame video decodes the same from pageable, page-locked and device payloads, whose pieces end inside GOPs (host)
  and at the 2 048-frame limit (device);
- malformed frames in any piece raise LM_ERR_INVALID naming the frame, in guard mode with no guard byte touched;
- detection and the three pass-1 entry points on decoded frames equal the raw path on cv2's decoded frames;
- locomouse_b200 with decode_mpeg4: 1 on an XVID AVI, an MP4 and an MKV (the AVI also in windows) and locomouse_b200_batch
  write output_<stem>.yml byte-identical to the run on the Y800 AVI of cv2's decoded frames.
Needs a B200: pytest -m gpu."""
import subprocess

import numpy as np
import pytest

from _containers import write_cv2
from _mpeg4_avi import decode_cpu, frames_of, read_video_mpeg4, split, write_cv2_mpeg4
from test_gpu_mjpeg_ingest import _memories
from test_gpu_png_ingest import _detector
from test_mpeg4_avi import _frames

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _gpu(path, det=None):
    payload, offs, extra, _, (n, h, w) = read_video_mpeg4(path)
    det = det or _detector(h, w)
    got = det.decode_mpeg4(extra, payload, offs).cpu().numpy()
    assert np.array_equal(got, decode_cpu(extra, payload, offs, h, w))
    return got


KINDS = [("avi", "XVID"), ("mp4", "mp4v"), ("mkv", "XVID")]


@pytest.mark.parametrize("ext,fourcc", KINDS, ids=[f"{e}-{f}" for e, f in KINDS])
@pytest.mark.parametrize("colour", [False, True], ids=["grey", "colour"])
@pytest.mark.parametrize("h,w,n,noise", [(400, 1700, 14, 8.0), (48, 64, 40, 30.0), (36, 44, 30, 2.0)])
def test_cv2_written_equals_videocapture(tmp_path, ext, fourcc, colour, h, w, n, noise):
    want = write_cv2_mpeg4(cv2, tmp_path / f"v.{ext}", _frames(h + n, n, h, w, colour, noise), fourcc)
    assert np.array_equal(_gpu(tmp_path / f"v.{ext}"), want)


@pytest.mark.parametrize("h,w", [(48, 64), (18, 30), (2, 31), (50, 17)])
def test_random_syntax_streams(tmp_path, h, w):
    from _mpeg4_avi import mpeg4_avi
    from _png_avi import capture
    from test_mpeg4_avi import fuzz_stream

    for seed in range(3):
        _, frames = fuzz_stream(h, w, seed)
        (tmp_path / "f.avi").write_bytes(mpeg4_avi(frames, w, h, fourcc=b"FMP4"))
        assert np.array_equal(_gpu(tmp_path / "f.avi"), capture(cv2, tmp_path / "f.avi"))


@pytest.fixture(scope="module")
def long_video(tmp_path_factory):
    path = tmp_path_factory.mktemp("long") / "v.avi"
    want = write_cv2_mpeg4(cv2, path, _frames(77, 2100, 32, 48, False, 6.0), "XVID")
    payload, offs, extra, ivop, _ = read_video_mpeg4(path)
    return want, payload, offs, extra


def test_every_payload_memory_and_piece(long_video):
    want, payload, offs, extra = long_video
    det = _detector(32, 48)
    for name, p in _memories(payload).items():
        assert np.array_equal(det.decode_mpeg4(extra, p, offs).cpu().numpy(), want), name
    assert det.info("ms_decode") > 0


def test_malformed_frames_are_named_in_every_piece(monkeypatch, long_video):
    monkeypatch.setenv("LM_GUARD", "1")
    want, payload, offs, extra = long_video
    frames = frames_of(payload, offs)
    det = _detector(32, 48)
    for at in (1, 600, 2099):
        start = frames[at].index(b"\0\0\1\xb6") + 12
        for bad in (frames[at][:start] + bytes(len(frames[at]) - start), frames[at][:start + 2]):
            p, o = split(frames[:at] + [bad] + frames[at + 1:])
            words = f"frame {at}: (the frame's data ends|invalid VLC|coefficient run|intra DC|marker bit)"
            with pytest.raises(ValueError, match=words):
                decode_cpu(extra, p, o, 32, 48)
            for name, m in _memories(p).items():
                with pytest.raises(ValueError, match=words):
                    det.decode_mpeg4(extra, m, o)
    for name, m in _memories(payload).items():
        assert np.array_equal(det.decode_mpeg4(extra, m, offs).cpu().numpy(), want), name
    assert det.info("guard_regions") > 0
    assert det.info("guard_violations") == 0


def test_detection_on_decoded_frames_is_unchanged(tmp_path):
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import bb_base_params, bb_de_params, bb_tm_params

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    ref_frames = write_cv2_mpeg4(cv2, tmp_path / "v.avi", frames.numpy(), "XVID")
    payload, offs, extra, _, _ = read_video_mpeg4(tmp_path / "v.avi")
    det = Detector(cfg, model, bkg, calib, device=0)
    dev = det.decode_mpeg4(extra, payload, offs)
    assert np.array_equal(dev.cpu().numpy(), ref_frames)
    got = det.detect_batch(dev, bx, bs, bb)
    ref = det.detect_batch(ref_frames, bx, bs, bb)
    assert int(ref.n_bottom.sum()) > 0
    assert np.array_equal(got.raw, ref.raw)
    y, x = np.mgrid[-2:3, -2:3]
    disk = ((x * x + y * y) <= 6.25).astype(np.float32)
    for fn, p in ((det.bounding_box_tm_de, bb_de_params(cfg, side_h=spec.side_h)), (det.bounding_box_base, bb_base_params(cfg, side_h=spec.side_h)),
                  (det.bounding_box_tm, bb_tm_params(cfg, disk / disk.sum(), side_h=spec.side_h, sums_as_float=0))):
        a, b = fn(dev, p), fn(ref_frames, p)
        assert all(np.array_equal(np.ascontiguousarray(u).view(np.uint8), np.ascontiguousarray(v).view(np.uint8)) for u, v in zip(a, b))


@pytest.mark.parametrize("method", ["1"])
def test_driver_output_on_mpeg4_equals_y800(tmp_path, method):
    """host/locomouse_b200 with decode_mpeg4: 1 on an XVID AVI, an mp4v MP4 and an XVID MKV (and the AVI in windows of 16
    frames, which end before I-VOPs) writes the same output_<stem>.yml and candidates file, byte for byte, as on the Y800 AVI
    of the frames VideoCapture reads from it; so does locomouse_b200_batch on a list holding the MP4.  Method 2 (TM_DE) is
    not run: on cv2's MPEG-4 frames of this synthetic video its pass-1 box leaves the image, in the Y800 run as well."""
    from _png_avi import write_cv2_avi
    from locomouse_cpp_b200 import synth
    from test_host_cpp import _build_driver, write_problem_files

    exe = _build_driver()
    spec = synth.SynthSpec(method={"1": "TM", "2": "TM_DE"}[method])
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 60, seed=1000)
    frames = frames.numpy()
    rows = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
            (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0), (0.95, 0.5, 0.6, 0.5, 1.0, 0.0, 1.0)]
    flat = ", ".join(repr(float(v)) for r in rows for v in r)
    fsz = frames.shape[1] * frames.shape[2]
    runs = [("y800", "avi", "XVID", ""), ("avi", "avi", "XVID", ""), ("mp4", "mp4", "mp4v", ""), ("mkv", "mkv", "XVID", ""),
            ("win", "avi", "XVID", f"max_resident_bytes: {16 * fsz}\n")]
    outs = {}
    decoded = None
    for name, ext, fourcc, extra in runs:
        d = tmp_path / name
        d.mkdir()
        write_problem_files(d, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, with_boxes=method == "1",
                            extra_cfg=f"batch_frames: 4\ndecode_mpeg4: 1\nlocation_prior: [{flat}]\nmax_displacement_bottom: 40\n"
                                      f"max_displacement_side: 25\n" + extra)
        if name == "y800":
            continue
        got = write_cv2(cv2, d / f"video.{ext}", frames, fourcc)
        decoded = got if decoded is None else decoded
        assert np.array_equal(got, decoded)
    assert np.array_equal(write_cv2_avi(cv2, tmp_path / "y800" / "video.avi", decoded, "Y800"), decoded)
    for name, ext, _, _ in runs:
        d = tmp_path / name
        p = subprocess.run([exe, method, str(d / "config.yml"), str(d / f"video.{ext}"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                            str(d / "calib.lmc"), "R", str(d)], capture_output=True, text=True)
        assert p.returncode == 0, name + p.stdout + p.stderr
        outs[name] = ((d / "output_video.yml").read_bytes(), (d / "output_video.lmo").read_bytes())
    assert b"paw_tracks0" in outs["y800"][0]
    for name in outs:
        assert outs[name] == outs["y800"], name
    from test_gpu_streaming import _drivers

    batch = _drivers()[1]
    (tmp_path / "list.tsv").write_text("mp4/video.mp4\tmp4/bkg.lmi\n")
    (tmp_path / "batch").mkdir()
    d = tmp_path / "mp4"
    p = subprocess.run([batch, method, str(d / "config.yml"), str(tmp_path / "list.tsv"), str(d / "model.lmm"), str(d / "calib.lmc"), "R",
                        str(tmp_path / "batch")], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    assert (tmp_path / "batch" / "output_video.yml").read_bytes() == outs["y800"][0]
    # the same video without the option keeps today's refusal, which names the option
    (tmp_path / "off").mkdir()
    cfg_text = (tmp_path / "avi" / "config.yml").read_text().replace("decode_mpeg4: 1", "decode_mpeg4: 0")
    (tmp_path / "off" / "config.yml").write_text(cfg_text)
    d = tmp_path / "avi"
    p = subprocess.run([exe, method, str(tmp_path / "off" / "config.yml"), str(d / "video.avi"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                        str(d / "calib.lmc"), "R", str(tmp_path / "off")], capture_output=True, text=True)
    assert p.returncode != 0 and "outside this library" in p.stdout + p.stderr and "decode_mpeg4" in p.stdout + p.stderr
