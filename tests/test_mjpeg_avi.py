"""Motion-JPEG video read by host/lm_media.hpp with decode_mjpeg on (lmh_read_video_mjpeg) and decoded by
csrc/mjpeg_format.h run on the CPU (lmh_decode_mjpeg, the code k_mjpeg.cu runs on the device): frames equal
cv2.VideoCapture's channel 0 for cv2-written video (FFmpeg's and OpenCV's own MJPEG writers, grey and colour) and for streams
of the test encoder (1 and 3 components, 4:2:0 and 4:2:2, restart intervals, custom tables, omitted DHT, fill bytes, odd
widths); one frame of DC-only blocks pins the blue rule on all 65 536 (Y, Cb) pairs.  What the decoder does not decode is
refused with the reason, and with the option off Motion-JPEG keeps its "outside this library" refusal.  CPU only."""
import struct

import numpy as np
import pytest

from _containers import bitmapinfo, box, full, mkv, mov, write_cv2
from _mjpeg_avi import Jpeg, decode_cpu, mjpeg_avi, mjpeg_file, read_video_mjpeg, split, write_cv2_mjpeg
from _png_avi import capture
from test_avi_ranges import read_range

cv2 = pytest.importorskip("cv2")


def _frames(seed, n, h, w, colour):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3) if colour else (h, w), dtype=np.uint8), (7, 7), 2)
    return np.stack([np.roll(base, 3 * i, axis=1) for i in range(n)])


def _decoded(path):
    payload, offs, (n, h, w) = read_video_mjpeg(path)
    return decode_cpu(payload, offs, h, w)


@pytest.mark.parametrize("colour", [False, True], ids=["grey", "colour"])
@pytest.mark.parametrize("writer,quality", [("ffmpeg", None), ("opencv", 50), ("opencv", 75), ("opencv", 90)])
@pytest.mark.parametrize("h,w", [(400, 1700), (48, 64), (30, 250)])
def test_cv2_written_avi(tmp_path, writer, quality, colour, h, w):
    api = cv2.CAP_OPENCV_MJPEG if writer == "opencv" else None
    want = write_cv2_mjpeg(cv2, tmp_path / "v.avi", _frames(h + w, 3, h, w, colour), api=api, quality=quality)
    assert want.shape == (3, h, w)
    assert np.array_equal(_decoded(tmp_path / "v.avi"), want)


HAND = [dict(comps=1), dict(comps=1, quality=30), dict(comps=3, hv=(2, 2)), dict(comps=3, hv=(2, 1)), dict(comps=1, dri=3),
        dict(comps=3, hv=(2, 2), dri=2), dict(comps=3, hv=(2, 1), dri=1, custom_huffman=True), dict(comps=1, custom_huffman=True, quality=95),
        dict(comps=1, omit_dht=True), dict(comps=3, omit_dht=True, fill=True, quality=98), dict(comps=1, fill=True, dri=5)]


@pytest.mark.parametrize("kw", HAND, ids=[",".join(f"{k}={v}" for k, v in kw.items()) for kw in HAND])
@pytest.mark.parametrize("h,w", [(16, 16), (2, 31), (18, 17), (64, 1), (66, 97)])
def test_hand_built_streams(tmp_path, kw, h, w):
    rng = np.random.Generator(np.random.PCG64(h * w))
    J = Jpeg(**kw)
    hs, vs = J.hv
    jpegs = []
    for i in range(3):
        y = rng.integers(0, 256, (h, w), dtype=np.uint8)
        if i == 1:
            y = np.full((h, w), 255, np.uint8)  # saturated blocks: large coefficients, many FF bytes to stuff
        cb, cr = (rng.integers(0, 256, (-(-h // vs), -(-w // hs)), dtype=np.uint8) for _ in range(2))
        jpegs.append(J.encode(y, cb, cr))
    want = mjpeg_file(cv2, tmp_path / "v.avi", jpegs, w, h)
    payload, offs = split(jpegs)
    assert np.array_equal(decode_cpu(payload, offs, h, w), want)
    assert np.array_equal(_decoded(tmp_path / "v.avi"), want)


def dc_pairs_frame():
    """One 4:2:0 frame of DC-only blocks whose four Y blocks and one Cb block per MCU cover every (Y, Cb) pair: Y block value
    v needs a dequantised DC of 8 v (the IDCT gives (16383 (64 v + 32)) >> 20 = v), so q[0] = 8 and the coded DC is v - 128."""
    J = Jpeg(comps=3, hv=(2, 2), q=[np.full(64, 8), np.full(64, 8)])
    mx, my = 128, 128  # 16 384 MCUs x 4 Y blocks = 65 536 pairs; pair p: Cb = p >> 8, Y = p & 255, MCU p // 4 (one Cb per MCU)
    pair = np.arange(65536)
    yv, cv = pair & 255, pair >> 8
    m, k = pair // 4, pair % 4
    yb = np.zeros((2 * my, 2 * mx, 64), np.int64)
    cb = np.zeros((my, mx, 64), np.int64)
    yb[2 * (m // mx) + k // 2, 2 * (m % mx) + k % 2, 0] = yv - 128
    cb[m // mx, m % mx, 0] = cv - 128
    cr = np.zeros_like(cb)
    return J.encode_blocks((16 * my, 16 * mx), [yb, cb, cr]), yv, cv


def test_every_y_cb_pair(tmp_path):
    jpeg, yv, cv = dc_pairs_frame()
    want = mjpeg_file(cv2, tmp_path / "v.avi", [jpeg], 2048, 2048)[0]
    payload, offs = split([jpeg])
    got = decode_cpu(payload, offs, 2048, 2048)[0]
    assert np.array_equal(got, want)
    # the pairs really are all there: each Y block is flat at its v, and blue follows the restated rule
    blocks = got.reshape(256, 8, 256, 8).transpose(0, 2, 1, 3).reshape(256, 256, 64)
    ys = blocks.reshape(-1, 64)
    assert len({(int(a), int(b)) for a, b in zip(yv, cv)}) == 65536
    expect = np.clip((yv * 8192 + (cv - 128) * 14516) >> 13, 0, 255)
    by, bx = np.divmod(np.arange(65536) // 4, 128)
    k = np.arange(65536) % 4
    assert np.array_equal(blocks[2 * by + k // 2, 2 * bx + k % 2, 0], expect)
    assert (ys == ys[:, :1]).all()


def _refused(path, words, opt_in=True):
    with pytest.raises(RuntimeError, match=words):
        if opt_in:
            read_video_mjpeg(path)
        else:
            read_range(path, 0, 0)


def _patched(jpeg, marker, fn):
    """jpeg with the payload of its first `marker` segment passed through fn"""
    at = jpeg.index(bytes([0xFF, marker]))
    n = struct.unpack(">H", jpeg[at + 2:at + 4])[0]
    body = fn(jpeg[at + 4:at + 2 + n])
    return jpeg[:at + 2] + struct.pack(">H", len(body) + 2) + body + jpeg[at + 2 + n:]


def test_refusals(tmp_path):
    rng = np.random.Generator(np.random.PCG64(7))
    y = rng.integers(0, 256, (16, 32), dtype=np.uint8)
    good = Jpeg(comps=1).encode(y)
    colour = Jpeg(comps=3).encode(y, np.full((8, 16), 100, np.uint8), np.full((8, 16), 100, np.uint8))
    cases = [
        (good.replace(b"\xff\xc0", b"\xff\xc2", 1), "progressive"),
        (good.replace(b"\xff\xc0", b"\xff\xc9", 1), "arithmetic"),
        (good.replace(b"\xff\xc0", b"\xff\xc3", 1), "lossless"),
        (_patched(good, 0xC0, lambda b: bytes([12]) + b[1:]), "12-bit"),
        (_patched(good, 0xDB, lambda b: bytes([0x10]) + b[1:] + b[1:]), "16-bit quantisation"),
        (_patched(good, 0xC0, lambda b: b[:5] + bytes([4]) + b[6:] + bytes([2, 0x11, 0, 3, 0x11, 0, 4, 0x11, 0])), "only 1-component"),
        (_patched(colour, 0xC0, lambda b: b[:6] + b"R" + b[7:9] + b"G" + b[10:12] + b"B" + b[13:]), "RGB-coded"),
        (Jpeg(comps=3, hv=(1, 1)).encode(y, y, y), "chroma layout"),
    ]
    for i, (jpeg, words) in enumerate(cases):
        (tmp_path / f"r{i}.avi").write_bytes(mjpeg_avi([jpeg], 32, 16))
        _refused(tmp_path / f"r{i}.avi", r"frame 0: .*" + words)
    # an AVI1 interlaced pair: each field is a JPEG of half the height, so the chunk's SOF is not the video's size
    field = Jpeg(comps=1).encode(y[:8])
    (tmp_path / "i.avi").write_bytes(mjpeg_avi([good, field + field], 32, 16))
    _refused(tmp_path / "i.avi", r"frame 1: the frame's SOF size differs")
    (tmp_path / "l.avi").write_bytes(mjpeg_avi([good], 32, 16, fourcc=b"LJPG"))
    _refused(tmp_path / "l.avi", "outside this library")


def _avi1(jpeg):
    """jpeg with an 'AVI1' APP0 segment after its SOI, as the fields of interlaced AVI files carry"""
    return jpeg[:2] + b"\xff\xe0" + struct.pack(">H", 12) + b"AVI1" + bytes(6) + jpeg[2:]


@pytest.mark.parametrize("kind", ["avi", "mkv", "mov"])
def test_interlaced_field_pairs_are_refused(tmp_path, kind):
    """Every chunk two fields of half the height: VideoCapture weaves them into frames of the container's size; the reader
    refuses the video at frame 0 instead of reading the fields as frames of half the height."""
    rng = np.random.Generator(np.random.PCG64(11))
    J = Jpeg(comps=1)
    chunks = [_avi1(J.encode(rng.integers(0, 256, (16, 64), dtype=np.uint8))) + _avi1(J.encode(rng.integers(0, 256, (16, 64), dtype=np.uint8)))
              for _ in range(3)]
    path = tmp_path / f"v.{kind}"
    path.write_bytes({"avi": lambda: mjpeg_avi(chunks, 64, 32), "mkv": lambda: mkv(chunks, "V_MJPEG", 64, 32),
                      "mov": lambda: mov(chunks, b"jpeg", 64, 32)}[kind]())
    assert capture(cv2, path).shape == (3, 32, 64)
    _refused(path, r"frame 0: the frame's SOF size differs.*the frame is 64 x 16 pixels \(SOF\), the video 64 x 32")


def test_tables_carried_from_an_earlier_frame_are_refused(tmp_path):
    """libavcodec keeps DHT and DQT tables from frame to frame; a frame that leaves out a table an earlier frame defined is
    refused, by the reader and by the decoder, instead of being decoded with the wrong table."""
    rng = np.random.Generator(np.random.PCG64(12))
    ys = [rng.integers(0, 256, (16, 32), dtype=np.uint8) for _ in range(3)]
    custom = [Jpeg(comps=1, custom_huffman=True, omit_dht=i > 0).encode(y) for i, y in enumerate(ys)]
    no_dqt = [Jpeg(comps=1, quality=40, omit_dqt=i > 0).encode(y) for i, y in enumerate(ys)]
    for name, jpegs, words in (("dht", custom, r"frame 1: the frame defines other Huffman tables \(DHT\) than the video's first frame"),
                               ("dqt", no_dqt, r"frame 1: a component's quantisation table is not defined in the frame")):
        path = tmp_path / f"{name}.avi"
        path.write_bytes(mjpeg_avi(jpegs, 32, 16))
        assert capture(cv2, path).shape == (3, 16, 32)
        _refused(path, words)
        payload, offs = split(jpegs)
        with pytest.raises(ValueError, match=words):
            decode_cpu(payload, offs, 16, 32)
    # tables defined by frame 0 and by no other frame are the Annex K defaults: frames that all leave out DHT are read
    plain = [Jpeg(comps=1, omit_dht=True).encode(y) for y in ys]
    want = mjpeg_file(cv2, tmp_path / "plain.avi", plain, 32, 16)
    assert np.array_equal(_decoded(tmp_path / "plain.avi"), want)
    # frame 0 without DHT and a later frame with it is refused too (the set of defined tables differs)
    mixed = plain[:1] + [Jpeg(comps=1).encode(y) for y in ys[1:]]
    (tmp_path / "mixed.avi").write_bytes(mjpeg_avi(mixed, 32, 16))
    _refused(tmp_path / "mixed.avi", r"frame 1: the frame defines other Huffman tables")


def test_option_off_keeps_the_refusal(tmp_path):
    write_cv2_mjpeg(cv2, tmp_path / "v.avi", _frames(1, 2, 16, 24, True))
    _refused(tmp_path / "v.avi", "outside this library", opt_in=False)
    assert read_video_mjpeg(tmp_path / "v.avi")[2] == (2, 16, 24)


def test_malformed_entropy_data_names_the_frame():
    rng = np.random.Generator(np.random.PCG64(8))
    y = rng.integers(0, 256, (32, 48), dtype=np.uint8)
    good = Jpeg(comps=1, quality=90).encode(y)
    ecs = good.index(b"\xff\xda") + 2 + 8 + 2
    bad = [good[:ecs + (len(good) - ecs) // 2] + b"\xff\xd9",             # truncated entropy data
           good[:ecs] + b"\xff\x00" * 8 + good[ecs + 8:],                  # all-ones: no code of either table
           Jpeg(comps=1, dri=2).encode(y).replace(b"\xff\xd0", b"\xff\xfe\x00\x02", 1)]  # a restart marker replaced
    for i, b in enumerate(bad):
        payload, offs = split([good, good, b])
        with pytest.raises(ValueError, match=r"frame 2: (the entropy-coded data ends|invalid Huffman code|restart marker missing)"):
            decode_cpu(payload, offs, 32, 48)


@pytest.mark.parametrize("kind", ["mkv", "mov", "mkv-vfw", "mp4-6c"])
def test_containers(tmp_path, kind):
    if kind in ("mkv", "mov"):
        path = tmp_path / f"v.{kind}"
        want = write_cv2(cv2, path, _frames(2, 5, 24, 40, True), "MJPG")
    else:
        rng = np.random.Generator(np.random.PCG64(9))
        jpegs = [Jpeg(comps=1).encode(rng.integers(0, 256, (24, 40), dtype=np.uint8)) for _ in range(4)]
        if kind == "mkv-vfw":
            path = tmp_path / "v.mkv"
            path.write_bytes(mkv(jpegs, "V_MS/VFW/FOURCC", 40, 24, private=bitmapinfo(40, 24, b"MJPG", 24)))
        else:
            def descr(tag, body):
                return bytes([tag, 0x80, 0x80, 0x80, len(body)]) + body
            esds = full(b"esds", descr(3, struct.pack(">HB", 1, 0) + descr(4, bytes([0x6C, 0x11, 0, 0, 0]) + struct.pack(">II", 0, 0)) +
                                        descr(6, b"\x02")))
            path = tmp_path / "v.mp4"
            path.write_bytes(mov(jpegs, b"mp4v", 40, 24, children=esds, mp4=True))
        want = capture(cv2, path)
        assert want.shape == (4, 24, 40)
    assert np.array_equal(_decoded(path), want)
    _refused(path, "outside this library", opt_in=False)
