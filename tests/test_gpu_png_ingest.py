"""lm_decode_png / Detector.decode_png: PNG-coded AVI frames inflated and unfiltered on the device (csrc/k_png.cu).

- Decoded frames equal cv2.VideoCapture + extractChannel(0) on AVIs written by cv2.VideoWriter ('MPNG' / 'png ', grey and
  colour) and on hand-built AVIs of cv2.imencode PNGs (widths 1 and 31, which the writer cannot produce).
- PNGs built here from numpy filtering and Python's zlib cover every row filter, stored / fixed / dynamic blocks (the
  zlib strategies and level 0, a stored block across IDAT chunks), 1-byte IDAT chunks, colour types 0 / 2 / 6, a
  hand-written fixed-Huffman stream with matches of length 258 at distance 32768, and payloads in pageable, pinned and
  device memory.
- Malformed streams fail with LM_ERR_INVALID (ValueError) naming the frame, in guard mode with no guard byte touched.
- Detection and pass 1 on decoded, resident frames equal the same calls on the raw frames from host memory.
Needs a B200: pytest -m gpu."""
import zlib

import numpy as np
import pytest

from _png_avi import BitWriter, capture, make_png, png_avi, png_from_zlib, read_avi_png, write_cv2_avi
from locomouse_cpp_b200.types import Config, Model

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def _detector(rows, cols):
    from locomouse_cpp_b200.api import Detector

    cfg = Config(vid_rows=rows, vid_cols=cols, n_rows=rows, n_cols=cols, bb_w=cols, bb_h_bottom=rows, bb_h_side=rows,
                 cand_cap=64, det_cap=64, match_cap=64)
    w = np.zeros((1, 1), np.float32)
    model = Model(w=[[w, w, w], [w, w, w]], rho=[[1.0] * 3, [1.0] * 3])
    return Detector(cfg, model, np.zeros((rows, cols), np.uint8), np.arange(rows * cols, dtype=np.int32).reshape(rows, cols), device=0)


def _decode(pngs, rows, cols, det=None):
    payload = np.frombuffer(b"".join(pngs), np.uint8)
    offs = np.concatenate([[0], np.cumsum([len(p) for p in pngs])]).astype(np.int64)
    det = det or _detector(rows, cols)
    return det.decode_png(payload, offs).cpu().numpy()


def _channel0(img):
    """What VideoCapture's BGR frame gives as channel 0: grey itself, blue (third byte) of RGB / RGBA."""
    return img if img.ndim == 2 else img[..., 2]


VIDEOS = [("MPNG", False, 2, 1), ("MPNG", False, 32, 50), ("png ", False, 32, 50), ("MPNG", True, 32, 50), ("png ", True, 2, 1),
          ("MPNG", False, 1700, 50), ("MPNG", True, 1700, 1)]


@pytest.mark.parametrize("fourcc,colour,width,n", VIDEOS)
def test_decode_equals_videocapture(tmp_path, fourcc, colour, width, n):
    rng = np.random.Generator(np.random.PCG64(width + n))
    h = 400 if width == 1700 else 24
    base = rng.integers(0, 256, (h, width, 3) if colour else (h, width), dtype=np.uint8)
    frames = np.stack([np.roll(base, 3 * i, axis=0) for i in range(n)])
    want = write_cv2_avi(cv2, tmp_path / "v.avi", frames, fourcc)
    payload, offs, dims = read_avi_png(tmp_path / "v.avi")
    assert dims == want.shape
    got = _decode([payload[offs[i]:offs[i + 1]].tobytes() for i in range(n)], h, width)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("width,colour", [(1, False), (31, False), (31, True), (1, True)])
def test_decode_equals_videocapture_hand_built(tmp_path, width, colour):
    rng = np.random.Generator(np.random.PCG64(7 + width))
    h, n = 17, 5
    frames = rng.integers(0, 256, (n, h, width, 3) if colour else (n, h, width), dtype=np.uint8)
    pngs = [cv2.imencode(".png", f)[1].tobytes() for f in frames]
    (tmp_path / "v.avi").write_bytes(png_avi(pngs, width, h))
    want = capture(cv2, tmp_path / "v.avi")
    payload, offs, dims = read_avi_png(tmp_path / "v.avi")
    assert dims == want.shape == (n, h, width)
    got = _decode([payload[offs[i]:offs[i + 1]].tobytes() for i in range(n)], h, width)
    assert np.array_equal(got, want)


def _images(rng, h, w):
    grey = rng.integers(0, 256, (h, w), dtype=np.uint8)
    smooth = (np.add.outer(np.arange(h), np.arange(w)) % 256).astype(np.uint8)
    return grey, smooth


def test_every_filter_strategy_and_chunking():
    rng = np.random.Generator(np.random.PCG64(3))
    h, w = 45, 70
    grey, smooth = _images(rng, h, w)
    rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    rgba = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    mix = rng.integers(0, 5, h).tolist()
    cases = []
    for img in (grey, smooth, rgb, rgba):
        for filters in (mix, [0] * h, [1] * h, [2] * h, [3] * h, [4] * h):
            cases.append((img, dict(filters=filters)))
    for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_RLE, zlib.Z_HUFFMAN_ONLY, zlib.Z_FILTERED):
        for img in (grey, smooth, rgb):
            cases.append((img, dict(filters=mix, strategy=strategy)))
    for level in (0, 1, 9):
        cases.append((smooth, dict(filters=mix, level=level)))
    cases.append((smooth, dict(filters=mix, level=0, idat_split=1000)))   # stored blocks continue across IDAT chunks
    cases.append((grey, dict(filters=mix, idat_split=1)))                  # every byte in a chunk of its own
    cases.append((rgba, dict(filters=mix, level=0, idat_split=7)))
    big = rng.integers(0, 256, (200, 600), dtype=np.uint8)                 # level 0 of > 64 kB: several stored blocks
    for img, kw in cases:
        got = _decode([make_png(img, **kw)], h, w)
        assert np.array_equal(got[0], _channel0(img)), kw
    got = _decode([make_png(big, filters=[4] * 200, level=0, idat_split=4096)], 200, 600)
    assert np.array_equal(got[0], big)


def _far_match_png():
    """A fixed-Huffman block of matches of length 258 at distance 32768 (zlib never emits a distance above 32506): rows of
    255 pixels + the filter byte, 256 rows = 2 x 32768 bytes, rows 128..255 repeat rows 0..127."""
    rng = np.random.Generator(np.random.PCG64(11))
    top = rng.integers(0, 256, (128, 255), dtype=np.uint8)
    img = np.concatenate([top, top])
    raw = np.concatenate([np.zeros((256, 1), np.uint8), img], axis=1).tobytes()
    bw = BitWriter()
    bw.put(0x78, 8), bw.put(0x01, 8)
    for k in range(0, 32768, 16384):          # stored blocks with the first 32768 bytes
        bw.put(0, 1), bw.put(0, 2)
        bw.align()
        bw.put(16384, 16), bw.put(16384 ^ 0xFFFF, 16)
        bw.raw(raw[k:k + 16384])
    bw.put(1, 1), bw.put(1, 2)                # final block, fixed codes
    for _ in range(127):                      # 127 x 258 = 32766 bytes
        bw.fixed_literal(285)                 # length 258
        bw.code(29, 5)                        # distance code 29: 24577 + 13 extra bits
        bw.put(32768 - 24577, 13)
    for v in raw[-2:]:
        bw.fixed_literal(v)
    bw.fixed_literal(256)
    z = bw.bytes() + zlib.adler32(raw).to_bytes(4, "big")
    return png_from_zlib(z, 255, 256), img


def test_match_of_length_258_at_distance_32768():
    png, img = _far_match_png()
    assert np.array_equal(cv2.imdecode(np.frombuffer(png, np.uint8), cv2.IMREAD_UNCHANGED), img)
    assert np.array_equal(_decode([png], 256, 255)[0], img)


def test_payload_in_pageable_pinned_and_device_memory():
    import torch

    rng = np.random.Generator(np.random.PCG64(5))
    h, w, n = 30, 41, 9
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if i % 3 == 1 else rng.integers(0, 256, (h, w), dtype=np.uint8) for i in range(n)]
    pngs = [make_png(im, filters=rng.integers(0, 5, h).tolist(), idat_split=97) for im in imgs]
    payload = np.frombuffer(b"".join(pngs), np.uint8).copy()
    offs = np.concatenate([[0], np.cumsum([len(p) for p in pngs])]).astype(np.int64)
    want = np.stack([_channel0(im) for im in imgs])
    det = _detector(h, w)
    pinned = torch.from_numpy(payload).pin_memory()
    for p in (payload, torch.from_numpy(payload), pinned, pinned.cuda()):
        assert np.array_equal(det.decode_png(p, offs).cpu().numpy(), want)
    out = torch.zeros((n, h, w), dtype=torch.uint8, device="cuda:0")
    assert det.decode_png(pinned, offs, out=out) is out and np.array_equal(out.cpu().numpy(), want)
    assert det.info("ms_decode") > 0


def _malformed(raw, w, h):
    """(name, zlib stream, expected words of the message) for a frame whose filtered stream is `raw`."""
    good = zlib.compress(raw)
    hdr = b"\x78\x01"
    bw = BitWriter()                          # dynamic block whose 19 code-length codes all have length 1
    bw.put(1, 1), bw.put(2, 2), bw.put(0, 5), bw.put(0, 5), bw.put(15, 4)
    for _ in range(19):
        bw.put(1, 3)
    oversub = hdr + bw.bytes() + b"\0" * 8
    bw = BitWriter()                          # literal, then a match of length 3 at distance 2
    bw.put(1, 1), bw.put(1, 2)
    bw.fixed_literal(0)
    bw.fixed_literal(257)
    bw.code(1, 5)
    bw.fixed_literal(256)
    far = hdr + bw.bytes()
    return [
        ("truncated", good[:len(good) // 2], "ends early"),
        ("block type 3", hdr + b"\x07" + b"\0" * 8, "block type"),
        ("over-subscribed", oversub, "code lengths"),
        ("distance before start", far, "before the start"),
        ("too short", zlib.compress(raw[:-1]), "shorter"),
        ("too long", zlib.compress(raw + b"\0"), "longer"),
        ("preset dictionary", b"\x78\xbb" + good[2:], "zlib header"),
        ("bad filter type", zlib.compress(b"\x05" + raw[1:]), "filter"),
    ]


def test_malformed_streams_name_the_frame(monkeypatch):
    monkeypatch.setenv("LM_GUARD", "1")
    rng = np.random.Generator(np.random.PCG64(9))
    h, w = 12, 20
    img = rng.integers(0, 256, (h, w), dtype=np.uint8)
    raw = np.concatenate([np.zeros((h, 1), np.uint8), img], axis=1).tobytes()
    good = png_from_zlib(zlib.compress(raw), w, h)
    det = _detector(h, w)
    assert det.info("guard_violations") == 0
    for name, z, words in _malformed(raw, w, h):
        with pytest.raises(ValueError, match=r"frame 2: .*" + words):
            _decode([good, good, png_from_zlib(z, w, h), good], h, w, det)
    for bad, words in ((png_from_zlib(zlib.compress(raw), w + 1, h), "pixels"), (good[:30], "not a PNG"),
                       (png_from_zlib(zlib.compress(raw), w, h, depth=16), "bit depth"),
                       (png_from_zlib(zlib.compress(raw), w, h, interlace=1), "interlaced")):
        with pytest.raises(ValueError, match=r"frame 1: .*" + words):
            _decode([good, bad], h, w, det)
    assert np.array_equal(_decode([good], h, w, det)[0], img)
    assert det.info("guard_regions") > 0
    assert det.info("guard_violations") == 0


def test_detection_on_decoded_frames_is_unchanged():
    import torch

    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.api import Detector
    from locomouse_cpp_b200.types import bb_base_params, bb_de_params, bb_tm_params

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40, seed=1000)
    frames = frames.numpy()
    pngs = [cv2.imencode(".png", f)[1].tobytes() for f in frames]
    det = Detector(cfg, model, bkg, calib, device=0)
    payload = torch.from_numpy(np.frombuffer(b"".join(pngs), np.uint8).copy()).pin_memory()
    offs = np.concatenate([[0], np.cumsum([len(p) for p in pngs])]).astype(np.int64)
    dev = det.decode_png(payload, offs)
    assert np.array_equal(dev.cpu().numpy(), frames)
    got = det.detect_batch(dev, bx, bs, bb)
    ref = det.detect_batch(frames, bx, bs, bb)
    assert int(ref.n_bottom.sum()) > 0
    assert np.array_equal(got.raw, ref.raw)    # every lm_results array, scores as their f64 bit patterns
    y, x = np.mgrid[-2:3, -2:3]
    disk = ((x * x + y * y) <= 6.25).astype(np.float32)
    for fn, p in ((det.bounding_box_tm_de, bb_de_params(cfg, side_h=spec.side_h)), (det.bounding_box_base, bb_base_params(cfg, side_h=spec.side_h)),
                  (det.bounding_box_tm, bb_tm_params(cfg, disk / disk.sum(), side_h=spec.side_h, sums_as_float=0))):
        a, b = fn(dev, p), fn(frames, p)
        assert all(np.array_equal(np.ascontiguousarray(u).view(np.uint8), np.ascontiguousarray(v).view(np.uint8)) for u, v in zip(a, b))


@pytest.mark.parametrize("method", ["1", "2"])
def test_driver_output_on_mpng_equals_y800(tmp_path, method):
    """host/locomouse_b200 on an MPNG AVI (frames decoded once into device memory, pass 1 and detection on resident frames)
    writes the same output_<stem>.yml and candidates file, byte for byte, as on the Y800 AVI of the same frames.
    Method 2 (TM_DE) runs pass 1 on the device; method 1 (TM) reads the pass-1 boxes file."""
    import subprocess

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
    for fourcc in ("Y800", "MPNG"):
        d = tmp_path / fourcc.strip()
        d.mkdir()
        write_problem_files(d, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h, with_boxes=method == "1",
                            extra_cfg=f"batch_frames: 16\nlocation_prior: [{flat}]\nmax_displacement_bottom: 40\nmax_displacement_side: 25\n")
        want = write_cv2_avi(cv2, d / "video.avi", frames, fourcc if fourcc == "MPNG" else "Y800")
        assert np.array_equal(want, frames)
        p = subprocess.run([exe, method, str(d / "config.yml"), str(d / "video.avi"), str(d / "bkg.lmi"), str(d / "model.lmm"),
                            str(d / "calib.lmc"), "R", str(d)], capture_output=True, text=True)
        assert p.returncode == 0, p.stdout + p.stderr
        outs.append(((d / "output_video.yml").read_bytes(), (d / "output_video.lmo").read_bytes()))
    assert outs[0][0] == outs[1][0] and outs[0][1] == outs[1][1]
    assert b"paw_tracks0" in outs[0][0]
