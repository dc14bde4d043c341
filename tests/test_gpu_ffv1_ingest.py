"""lm_decode_ffv1 / Detector.decode_ffv1: FFV1-coded AVI frames decoded on the device (csrc/k_ffv1.cu), one thread per
(GOP, slice) chain.

- Decoded frames equal cv2.VideoCapture + extractChannel(0) for cv2-written grey and colour video (1700 x 400, and small
  sizes over one, several and partial GOPs: n = 1, 12, 13, 50), and for streams of the test encoder: widths 1 and 31,
  range coders with the default and a custom state table, the large context model (work memory in global slots),
  intra-only, coded initial states and uneven slice grids.
- Payloads in pageable, pinned and device memory.
- Malformed streams (a truncated slice, a CRC mismatch, a footer size running past the chunk, a run of Golomb-Rice
  escapes that outlasts its slice) fail with ValueError naming frame and slice, in guard mode with no guard byte touched.
- Detection and pass 1 on decoded, resident frames equal the same calls on the raw frames; the driver's output from an
  FFV1 AVI is byte-identical to its output from the Y800 AVI of the same frames.
Needs a B200: pytest -m gpu."""
import numpy as np
import pytest

from _ffv1_avi import LARGE, Encoder, decode_cpu, encode_avi, make_slice, read_avi_ffv1, split_slices, write_cv2_ffv1
from test_gpu_png_ingest import _detector

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _frames(seed, n, h, w, colour):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = rng.integers(0, 256, (h, w, 3) if colour else (h, w), dtype=np.uint8)
    base[h // 3: h // 2] = 40
    return np.stack([np.roll(base, 2 * i, axis=1) + rng.integers(0, 3, base.shape, dtype=np.uint8) for i in range(n)])


def _gpu(path, det=None):
    ex, payload, offs, (n, h, w) = read_avi_ffv1(path)
    det = det or _detector(h, w)
    return det.decode_ffv1(ex, payload, offs).cpu().numpy()


@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("w,h,n", [(1700, 400, 1), (1700, 400, 13), (64, 24, 12), (64, 24, 50), (36, 10, 13)])
def test_cv2_written_equals_videocapture(tmp_path, colour, w, h, n):
    want = write_cv2_ffv1(cv2, tmp_path / "v.avi", _frames(w + n, n, h, w, colour))
    assert np.array_equal(_gpu(tmp_path / "v.avi"), want)


@pytest.mark.parametrize("kw", [dict(), dict(coder=1), dict(coder=2), dict(model=LARGE), dict(model=LARGE, coder=2), dict(gop=1),
                                dict(coder=1, initial_states=True), dict(slices=(3, 5)), dict(slices=(1, 2), gop=5)],
                         ids=["golomb", "range", "range-custom", "large", "large-range", "intra", "initial-states", "grid-3x5", "grid-1x2"])
@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("w", [1, 31])
def test_hand_built_streams(tmp_path, kw, colour, w):
    if w == 1 and kw.get("slices", (4, 2))[0] > 1:
        kw = dict(kw, slices=(1, 3))
    _, _, want = encode_avi(cv2, tmp_path / "v.avi", _frames(3, 13, 21, w, colour), **kw)
    assert np.array_equal(_gpu(tmp_path / "v.avi"), want)


def test_payload_in_pageable_pinned_and_device_memory(tmp_path):
    import torch

    want = write_cv2_ffv1(cv2, tmp_path / "v.avi", _frames(5, 30, 40, 64, False))
    ex, payload, offs, (n, h, w) = read_avi_ffv1(tmp_path / "v.avi")
    det = _detector(h, w)
    pinned = torch.from_numpy(payload).pin_memory()
    for p in (payload, torch.from_numpy(payload), pinned, pinned.cuda()):
        assert np.array_equal(det.decode_ffv1(ex, p, offs).cpu().numpy(), want)
    out = torch.zeros((n, h, w), dtype=torch.uint8, device="cuda:0")
    assert det.decode_ffv1(bytes(ex), pinned, offs, out=out) is out and np.array_equal(out.cpu().numpy(), want)
    assert det.info("ms_decode") > 0


def test_malformed_streams_name_frame_and_slice(monkeypatch):
    monkeypatch.setenv("LM_GUARD", "1")
    frames = _frames(9, 6, 16, 24, False)
    enc = Encoder(False)
    rec, good = enc.encode(frames[:2])
    head = enc.head_bytes[2]  # slice 2 of frame 1
    rec, good = enc.encode(frames)
    ex = np.frombuffer(rec, np.uint8)
    det = _detector(16, 24)
    assert det.info("guard_violations") == 0

    def run(fr):
        pay = np.frombuffer(b"".join(fr), np.uint8)
        offs = np.concatenate([[0], np.cumsum([len(f) for f in fr])]).astype(np.int64)
        return det.decode_ffv1(ex, pay, offs).cpu().numpy()

    def patched(frame, s, fn):
        fr = list(good)
        sl = split_slices(fr[frame], 8)
        sl[s] = fn(sl[s])
        fr[frame] = b"".join(sl)
        return fr

    cases = [
        (patched(3, 4, lambda b: make_slice(b[:(len(b) - 8) // 2])), r"frame 3, slice 4: the slice data ends"),
        (patched(2, 6, lambda b: b[:10] + bytes([b[10] ^ 0x40]) + b[11:]), r"frame 2, slice 6: slice CRC mismatch"),
        (patched(4, 7, lambda b: b[:-8] + b"\xff\xff\xff" + b[-5:]), r"frame 4, slice 0: the slice footers"),
        # the header kept, then all-zero bits: Golomb-Rice escapes (12 zeros + 8 bits each) that outlast the slice
        (patched(1, 2, lambda b: make_slice(b[:head] + bytes(len(b) - 8 - head))), r"frame 1, slice 2: the slice data ends"),
    ]
    for fr, words in cases:
        with pytest.raises(ValueError, match=words):
            run(fr)
    assert np.array_equal(run(good), frames)
    assert det.info("guard_regions") > 0
    assert det.info("guard_violations") == 0


def test_detection_on_decoded_frames_is_unchanged(tmp_path):
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import bb_base_params, bb_de_params, bb_tm_params

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    frames = frames.numpy()
    assert np.array_equal(write_cv2_ffv1(cv2, tmp_path / "v.avi", frames), frames)
    ex, payload, offs, _ = read_avi_ffv1(tmp_path / "v.avi")
    det = Detector(cfg, model, bkg, calib, device=0)
    dev = det.decode_ffv1(ex, payload, offs)
    assert np.array_equal(dev.cpu().numpy(), frames)
    assert np.array_equal(decode_cpu(ex, payload, offs, frames.shape[1], frames.shape[2]), frames)
    got = det.detect_batch(dev, bx, bs, bb)
    ref = det.detect_batch(frames, bx, bs, bb)
    assert int(ref.n_bottom.sum()) > 0
    assert np.array_equal(got.raw, ref.raw)
    y, x = np.mgrid[-2:3, -2:3]
    disk = ((x * x + y * y) <= 6.25).astype(np.float32)
    for fn, p in ((det.bounding_box_tm_de, bb_de_params(cfg, side_h=spec.side_h)), (det.bounding_box_base, bb_base_params(cfg, side_h=spec.side_h)),
                  (det.bounding_box_tm, bb_tm_params(cfg, disk / disk.sum(), side_h=spec.side_h, sums_as_float=0))):
        a, b = fn(dev, p), fn(frames, p)
        assert all(np.array_equal(np.ascontiguousarray(u).view(np.uint8), np.ascontiguousarray(v).view(np.uint8)) for u, v in zip(a, b))


@pytest.mark.parametrize("method", ["1", "2"])
def test_driver_output_on_ffv1_equals_y800(tmp_path, method):
    """host/locomouse_b200 on an FFV1 AVI (decoded once into device memory) writes the same output_<stem>.yml and candidates
    file, byte for byte, as on the Y800 AVI of the same frames."""
    import subprocess

    from _png_avi import write_cv2_avi
    from locomouse_cpp_b200 import synth
    from test_host_cpp import _build_driver, write_problem_files

    exe = _build_driver()
    spec = synth.SynthSpec(method={"1": "TM", "2": "TM_DE"}[method])
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    frames = frames.numpy()
    rows = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
            (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0), (0.95, 0.5, 0.6, 0.5, 1.0, 0.0, 1.0)]
    flat = ", ".join(repr(float(v)) for r in rows for v in r)
    outs = []
    for fourcc in ("Y800", "FFV1"):
        d = tmp_path / fourcc
        d.mkdir()
        write_problem_files(d, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, with_boxes=method == "1",
                            extra_cfg=f"batch_frames: 16\nlocation_prior: [{flat}]\nmax_displacement_bottom: 40\nmax_displacement_side: 25\n")
        want = write_cv2_ffv1(cv2, d / "video.avi", frames) if fourcc == "FFV1" else write_cv2_avi(cv2, d / "video.avi", frames, "Y800")
        assert np.array_equal(want, frames)
        p = subprocess.run([exe, method, str(d / "config.yml"), str(d / "video.avi"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                            str(d / "calib.lmc"), "R", str(d)], capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
        outs.append(((d / "output_video.yml").read_bytes(), (d / "output_video.lmo").read_bytes()))
    assert outs[0][0] == outs[1][0] and outs[0][1] == outs[1][1]
    assert b"paw_tracks0" in outs[0][0]
