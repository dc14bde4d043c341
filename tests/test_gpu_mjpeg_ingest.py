"""Motion-JPEG on the device (lm_decode_mjpeg, k_mjpeg.cu):
- the device decode equals the CPU decode (mjpeg_format.h) and cv2.VideoCapture's channel 0 on cv2-written video, the test
  encoder's streams (with and without restart intervals) and the frame of every (Y, Cb) pair; restart-interval streams and
  the (Y, Cb) frame from pageable, page-locked and device payloads;
- malformed streams, and a frame that leaves out frame 0's DHT tables (in any piece), raise LM_ERR_INVALID naming the frame,
  in guard mode with no guard byte touched;
- detection and the three pass-1 entry points on decoded frames equal the raw path on cv2's decoded frames;
- locomouse_b200 with decode_mjpeg: 1 on an MJPEG AVI, MKV and MOV (also in 32-frame windows) and locomouse_b200_batch write
  output_<stem>.yml byte-identical to the run on the Y800 AVI of cv2's decoded frames.
Needs a B200: pytest -m gpu."""
import subprocess

import numpy as np
import pytest

from _containers import write_cv2
from _mjpeg_avi import Jpeg, decode_cpu, mjpeg_file, read_video_mjpeg, split, write_cv2_mjpeg
from test_gpu_png_ingest import _detector
from test_mjpeg_avi import HAND, _frames, dc_pairs_frame

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _gpu(path, det=None):
    payload, offs, (n, h, w) = read_video_mjpeg(path)
    det = det or _detector(h, w)
    got = det.decode_mjpeg(payload, offs).cpu().numpy()
    assert np.array_equal(got, decode_cpu(payload, offs, h, w))
    return got


@pytest.mark.parametrize("colour", [False, True], ids=["grey", "colour"])
@pytest.mark.parametrize("writer,quality", [("ffmpeg", None), ("opencv", 50), ("opencv", 90)])
@pytest.mark.parametrize("h,w,n", [(400, 1700, 5), (48, 64, 40)])
def test_cv2_written_equals_videocapture(tmp_path, writer, quality, colour, h, w, n):
    api = cv2.CAP_OPENCV_MJPEG if writer == "opencv" else None
    want = write_cv2_mjpeg(cv2, tmp_path / "v.avi", _frames(h + n, n, h, w, colour), api=api, quality=quality)
    assert np.array_equal(_gpu(tmp_path / "v.avi"), want)


@pytest.mark.parametrize("kw", HAND, ids=[",".join(f"{k}={v}" for k, v in kw.items()) for kw in HAND])
@pytest.mark.parametrize("h,w", [(2, 31), (18, 17), (66, 97)])
def test_hand_built_streams(tmp_path, kw, h, w):
    rng = np.random.Generator(np.random.PCG64(h + w))
    J = Jpeg(**kw)
    hs, vs = J.hv
    jpegs = [J.encode(rng.integers(0, 256, (h, w), dtype=np.uint8), *(rng.integers(0, 256, (-(-h // vs), -(-w // hs)), dtype=np.uint8)
                                                                      for _ in range(2))) for _ in range(5)]
    want = mjpeg_file(cv2, tmp_path / "v.avi", jpegs, w, h)
    assert np.array_equal(_gpu(tmp_path / "v.avi"), want)


def test_every_y_cb_pair_and_payload_memory(tmp_path):
    import torch

    jpeg, _, _ = dc_pairs_frame()
    want = mjpeg_file(cv2, tmp_path / "v.avi", [jpeg] * 3, 2048, 2048)
    payload, offs = split([jpeg] * 3)
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import Config, Model

    # the frame is larger than the tracker's boxes may be: a small box, only the decoder is used
    cfg = Config(vid_rows=2048, vid_cols=2048, n_rows=64, n_cols=64, bb_w=64, bb_h_bottom=32, bb_h_side=32, cand_cap=64, det_cap=64, match_cap=64)
    w = np.zeros((1, 1), np.float32)
    det = Detector(cfg, Model(w=[[w, w, w], [w, w, w]], rho=[[1.0] * 3, [1.0] * 3]), np.zeros((2048, 2048), np.uint8),
                   np.arange(64 * 64, dtype=np.int32).reshape(64, 64), device=0)
    pinned = torch.from_numpy(payload).pin_memory()
    for p in (payload, torch.from_numpy(payload), pinned, pinned.cuda()):
        assert np.array_equal(det.decode_mjpeg(p, offs).cpu().numpy(), want)
    out = torch.zeros((3, 2048, 2048), dtype=torch.uint8, device="cuda:0")
    assert det.decode_mjpeg(pinned, offs, out=out) is out and np.array_equal(out.cpu().numpy(), want)
    assert det.info("ms_decode") > 0


def _memories(payload):
    """the payload as pageable numpy, pageable torch, page-locked and device memory"""
    import torch

    pinned = torch.from_numpy(payload).pin_memory()
    return {"pageable": payload, "torch": torch.from_numpy(payload), "pinned": pinned, "device": pinned.cuda()}


RESTART = [dict(comps=3, hv=(2, 2), dri=2), dict(comps=1, dri=3, fill=True), dict(comps=3, hv=(2, 1), dri=1, custom_huffman=True)]


@pytest.mark.parametrize("kw", RESTART, ids=[",".join(f"{k}={v}" for k, v in kw.items()) for kw in RESTART])
def test_restart_intervals_from_every_payload_memory(tmp_path, kw):
    rng = np.random.Generator(np.random.PCG64(len(kw)))
    J = Jpeg(**kw)
    hs, vs = J.hv
    h, w = 34, 45
    jpegs = [J.encode(rng.integers(0, 256, (h, w), dtype=np.uint8), *(rng.integers(0, 256, (-(-h // vs), -(-w // hs)), dtype=np.uint8)
                                                                      for _ in range(2))) for _ in range(6)]
    want = mjpeg_file(cv2, tmp_path / "v.avi", jpegs, w, h)
    payload, offs = split(jpegs)
    det = _detector(h, w)
    for name, p in _memories(payload).items():
        assert np.array_equal(det.decode_mjpeg(p, offs).cpu().numpy(), want), name


def test_table_carry_is_refused_in_every_piece(monkeypatch):
    """A frame that leaves out the DHT tables frame 0 defines is refused on the device as on the CPU, wherever it lies: the
    2 100 frames of pageable and page-locked payloads are decoded in three pieces, and the frame is in the first, the second
    or the last."""
    monkeypatch.setenv("LM_GUARD", "1")
    rng = np.random.Generator(np.random.PCG64(13))
    ys = [rng.integers(0, 256, (16, 32), dtype=np.uint8) for _ in range(3)]
    J = Jpeg(comps=1, custom_huffman=True)
    jpegs = [J.encode(y) for y in ys] * 700
    det = _detector(16, 32)
    payload, offs = split(jpegs)
    want = decode_cpu(payload, offs, 16, 32)
    for at in (1, 1500, 2099):
        bad = list(jpegs)
        bad[at] = Jpeg(comps=1, custom_huffman=True, omit_dht=True).encode(ys[at % 3])
        payload, offs = split(bad)
        words = f"frame {at}: the frame defines other Huffman tables"
        with pytest.raises(ValueError, match=words):
            decode_cpu(payload, offs, 16, 32)
        for name, p in _memories(payload).items():
            with pytest.raises(ValueError, match=words):
                det.decode_mjpeg(p, offs)
    payload, offs = split(jpegs)
    for name, p in _memories(payload).items():
        assert np.array_equal(det.decode_mjpeg(p, offs).cpu().numpy(), want), name
    assert det.info("guard_violations") == 0


def test_malformed_streams_name_the_frame(monkeypatch):
    monkeypatch.setenv("LM_GUARD", "1")
    rng = np.random.Generator(np.random.PCG64(8))
    y = rng.integers(0, 256, (32, 48), dtype=np.uint8)
    good = Jpeg(comps=1, quality=90).encode(y)
    ecs = good.index(b"\xff\xda") + 10
    det = _detector(32, 48)
    cases = [(good[:ecs + (len(good) - ecs) // 2] + b"\xff\xd9", "the entropy-coded data ends"),
             (good[:ecs] + b"\xff\x00" * 8 + good[ecs + 8:], "invalid Huffman code"),
             (Jpeg(comps=1, dri=2).encode(y).replace(b"\xff\xd0", b"\xff\xfe\x00\x02", 1), "restart marker missing"),
             (Jpeg(comps=1).encode(y[:16]), "the frame's SOF size differs")]
    # a run past coefficient 63: after the DC of the first block, AC symbols of run 15 / size 1 ('0xF1') until the run overflows
    from _mjpeg_avi import AC_LUMA, _Bits, _codes, DC_LUMA
    dc, ac = _codes(*DC_LUMA), _codes(*AC_LUMA)
    bw = _Bits()
    bw.put(*dc[0])
    for _ in range(5):
        bw.put(*ac[0xF1])
        bw.put(1, 1)
    bw.flush()
    cases.append((good[:ecs] + bytes(bw.out) + b"\xff\xd9", "AC run past coefficient 63"))
    for bad, words in cases:
        payload, offs = split([good, good, bad, good])
        with pytest.raises(ValueError, match="frame 2: " + words):
            det.decode_mjpeg(payload, offs)
    payload, offs = split([good] * 4)
    assert np.array_equal(det.decode_mjpeg(payload, offs).cpu().numpy(), decode_cpu(payload, offs, 32, 48))
    assert det.info("guard_regions") > 0
    assert det.info("guard_violations") == 0


def test_detection_on_decoded_frames_is_unchanged(tmp_path):
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import bb_base_params, bb_de_params, bb_tm_params

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    ref_frames = write_cv2_mjpeg(cv2, tmp_path / "v.avi", frames.numpy())
    payload, offs, _ = read_video_mjpeg(tmp_path / "v.avi")
    det = Detector(cfg, model, bkg, calib, device=0)
    dev = det.decode_mjpeg(payload, offs)
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


@pytest.mark.parametrize("method", ["1", "2"])
def test_driver_output_on_mjpeg_equals_y800(tmp_path, method):
    """host/locomouse_b200 with decode_mjpeg: 1 on MJPEG in AVI, MKV and MOV (and the AVI in 32-frame windows) writes the same
    output_<stem>.yml and candidates file, byte for byte, as on the Y800 AVI of the frames VideoCapture reads from it; so does
    locomouse_b200_batch on a list holding the MKV."""
    from _png_avi import write_cv2_avi
    from locomouse_cpp_b200 import synth
    from test_host_cpp import _build_driver, write_problem_files

    exe = _build_driver()
    spec = synth.SynthSpec(method={"1": "TM", "2": "TM_DE"}[method])
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 80, seed=1000)
    frames = frames.numpy()
    rows = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
            (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0), (0.95, 0.5, 0.6, 0.5, 1.0, 0.0, 1.0)]
    flat = ", ".join(repr(float(v)) for r in rows for v in r)
    fsz = frames.shape[1] * frames.shape[2]
    runs = [("y800", "avi", ""), ("avi", "avi", ""), ("mkv", "mkv", ""), ("mov", "mov", ""), ("win", "avi", f"max_resident_bytes: {32 * fsz}\n")]
    outs = {}
    decoded = None
    for name, ext, extra in runs:
        d = tmp_path / name
        d.mkdir()
        write_problem_files(d, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, with_boxes=method == "1",
                            extra_cfg=f"batch_frames: 16\ndecode_mjpeg: 1\nlocation_prior: [{flat}]\nmax_displacement_bottom: 40\n"
                                      f"max_displacement_side: 25\n" + extra)
        video = d / f"video.{ext}"
        if name == "y800":
            continue
        got = write_cv2(cv2, video, frames, "MJPG")
        decoded = got if decoded is None else decoded
        assert np.array_equal(got, decoded)
    assert np.array_equal(write_cv2_avi(cv2, tmp_path / "y800" / "video.avi", decoded, "Y800"), decoded)
    for name, ext, _ in runs:
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
    (tmp_path / "list.tsv").write_text("mkv/video.mkv\tmkv/bkg.lmi\n")
    (tmp_path / "batch").mkdir()
    d = tmp_path / "mkv"
    p = subprocess.run([batch, method, str(d / "config.yml"), str(tmp_path / "list.tsv"), str(d / "model.lmm"), str(d / "calib.lmc"), "R",
                        str(tmp_path / "batch")], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    assert (tmp_path / "batch" / "output_video.yml").read_bytes() == outs["y800"][0]
    # the same video without the option keeps today's refusal
    (tmp_path / "off").mkdir()
    cfg_text = (tmp_path / "avi" / "config.yml").read_text().replace("decode_mjpeg: 1", "decode_mjpeg: 0")
    (tmp_path / "off" / "config.yml").write_text(cfg_text)
    d = tmp_path / "avi"
    p = subprocess.run([exe, method, str(tmp_path / "off" / "config.yml"), str(d / "video.avi"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                        str(d / "calib.lmc"), "R", str(tmp_path / "off")], capture_output=True, text=True)
    assert p.returncode != 0 and "outside this library" in p.stdout + p.stderr
