"""Frame ranges of a video file (host/lm_media.hpp: index_video + read_frames, the reader LocoMouse streams a long video
through): ranges joined at arbitrary cuts are byte-identical to the whole read, for every container and pixel format the
reader takes; window plans of lmmedia::plan_windows end on FFV1 keyframes; a truncated chunk is refused when the file is
indexed, before any frame is used, with the message of a whole read."""
import ctypes as C
import struct

import numpy as np
import pytest

from _ffv1_avi import encode_avi, read_avi_ffv1
from _png_avi import _riff, read_avi_png, write_cv2_avi
from test_host_media import _dib_avi, _read
from test_match2nd import _host

cv2 = pytest.importorskip("cv2")
CODECS = {0: "raw", 1: "png", 2: "ffv1"}


def read_range(path, first, count):
    """(dims, bytes, offsets) of frames [first, first + count): dims = (n, rows, cols, codec, bytes of the range)."""
    fn = _host().lmh_read_avi_range
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    dims = np.zeros(5, np.int64)
    msg = C.create_string_buffer(512)
    if fn(str(path).encode(), first, count, dims.ctypes.data, None, None, msg, 512) != 0:
        raise RuntimeError(msg.value.decode())
    out = np.zeros(max(int(dims[4]), 1), np.uint8)
    offs = np.zeros(count + 1, np.int64)
    assert fn(str(path).encode(), first, count, dims.ctypes.data, out.ctypes.data, offs.ctypes.data, msg, 512) == 0
    return dims, out[:int(dims[4])], offs


def plan(path, max_bytes, batch_frames):
    fn = _host().lmh_plan_windows
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int]
    starts = np.zeros(4096, np.int32)
    msg = C.create_string_buffer(512)
    k = fn(str(path).encode(), max_bytes, batch_frames, starts.ctypes.data, starts.size, msg, 512)
    if k < 0:
        raise RuntimeError(msg.value.decode())
    return starts[:k + 1].tolist()


def joined(path, cuts):
    """The ranges between consecutive cuts, joined: raw pixels, or (payload, offsets) of coded frames."""
    parts, offs = [], [0]
    for a, b in zip(cuts[:-1], cuts[1:]):
        dims, data, o = read_range(path, a, b - a)
        parts.append(data)
        offs += [offs[-1] + int(v) for v in o[1:]]
    return CODECS[int(dims[3])], np.concatenate(parts), np.array(offs, np.int64)


def random_cuts(rng, n, k):
    return [0] + sorted(rng.choice(np.arange(1, n), size=min(k, n - 1), replace=False).tolist()) + [n]


def _frames(seed, n, h, w, *extra):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = rng.integers(0, 256, (n, h, w) + extra, dtype=np.uint8)
    return np.where(rng.random((n, h, w) + extra) < 0.7, base // 32 * 32, base).astype(np.uint8)   # compressible, not trivial


def _opendml_avi(frames, split):
    """A grey AVI whose frames continue in an OpenDML 'AVIX' RIFF after the first 'split' frames (with an idx1 and an ix00
    index chunk the walk must step over)."""
    n, h, w = frames.shape
    bih = struct.pack("<IiiHHIIiiII", 40, w, h, 1, 8, struct.unpack("<I", b"Y800")[0], w * h, 0, 0, 0, 0)
    strh = b"vids" + b"Y800" + b"\0" * 48
    odml = _riff(b"LIST", b"odml" + _riff(b"dmlh", struct.pack("<I", n) + b"\0" * 244))
    hdrl = b"hdrl" + _riff(b"avih", b"\0" * 56) + _riff(b"LIST", b"strl" + _riff(b"strh", strh) + _riff(b"strf", bih)) + odml
    movi = lambda fr: _riff(b"LIST", b"movi" + _riff(b"ix00", b"\0" * 24) + b"".join(_riff(b"00db", f.tobytes()) for f in fr))
    body0 = b"AVI " + _riff(b"LIST", hdrl) + movi(frames[:split]) + _riff(b"idx1", b"\0" * 16 * split)
    body1 = b"AVIX" + movi(frames[split:])
    return b"RIFF" + struct.pack("<I", len(body0)) + body0 + b"RIFF" + struct.pack("<I", len(body1)) + body1


def _videos(d):
    """{name: (path, channel 0 of every frame)} for every kind of video the reader takes."""
    out = {}
    grey = _frames(1, 23, 12, 20)
    write_cv2_avi(cv2, d / "y800.avi", grey, "Y800")
    out["y800"] = (d / "y800.avi", grey)
    bgr = _frames(2, 17, 9, 13, 3)
    (d / "bgr24.avi").write_bytes(_dib_avi(bgr, 24))              # bottom-up, rows padded to 4 bytes
    out["bgr24_bottom_up"] = (d / "bgr24.avi", bgr[..., 0])
    bgra = _frames(3, 11, 6, 10, 4)
    (d / "bgra32.avi").write_bytes(_dib_avi(bgra, 32, top_down=True))
    out["bgra32_top_down"] = (d / "bgra32.avi", bgra[..., 0])
    idx = _frames(4, 13, 5, 7)
    pal = [(int(v), 0, 0) for v in np.random.Generator(np.random.PCG64(5)).integers(0, 256, 256)]
    (d / "pal8.avi").write_bytes(_dib_avi(idx, 8, palette=pal))
    out["palettised"] = (d / "pal8.avi", np.array([p[0] for p in pal], np.uint8)[idx])
    odml = _frames(6, 19, 8, 16)
    (d / "odml.avi").write_bytes(_opendml_avi(odml, 7))
    out["opendml"] = (d / "odml.avi", odml)
    lmv = _frames(7, 15, 10, 14)
    (d / "v.lmv").write_bytes(b"LMV1" + struct.pack("<iii", *lmv.shape) + lmv.tobytes())
    out["lmv"] = (d / "v.lmv", lmv)
    return out


def test_raw_ranges_join_to_the_whole_read(tmp_path):
    rng = np.random.Generator(np.random.PCG64(11))
    for name, (path, want) in _videos(tmp_path).items():
        n = want.shape[0]
        if name != "lmv":
            assert np.array_equal(_read("lmh_read_avi", path), want), name
        for k in (1, 3, n - 1):
            codec, data, _ = joined(path, random_cuts(rng, n, k))
            assert codec == "raw"
            assert data.tobytes() == want.tobytes(), f"{name}, {k} cut(s)"
        dims, one, _ = read_range(path, n - 1, 1)
        assert tuple(dims[:3]) == want.shape and one.tobytes() == want[-1].tobytes()


@pytest.mark.parametrize("kind", ["mpng", "ffv1_gop12", "ffv1_intra", "ffv1_cv2"])
def test_coded_ranges_join_to_the_whole_read(tmp_path, kind):
    rng = np.random.Generator(np.random.PCG64(12))
    path = tmp_path / "v.avi"
    if kind == "mpng":
        frames = _frames(8, 21, 16, 24)
        write_cv2_avi(cv2, path, frames, "MPNG")
        whole = read_avi_png(path)
    elif kind == "ffv1_cv2":
        from _ffv1_avi import write_cv2_ffv1

        frames = _frames(9, 30, 16, 24)
        write_cv2_ffv1(cv2, path, frames)
        whole = read_avi_ffv1(path)[1:3]
    else:
        frames = _frames(9, 30, 16, 24)
        encode_avi(cv2, path, frames, slices=(2, 2), gop=12 if kind == "ffv1_gop12" else 1)
        whole = read_avi_ffv1(path)[1:3]
    payload, offsets = whole[0], whole[1]
    n = frames.shape[0]
    for k in (1, 4, n - 1):
        codec, data, offs = joined(path, random_cuts(rng, n, k))
        assert codec == ("png" if kind == "mpng" else "ffv1")
        assert data.tobytes() == np.asarray(payload).tobytes(), f"{k} cut(s)"
        assert np.array_equal(offs, np.asarray(offsets)), f"{k} cut(s)"


def test_window_plans(tmp_path):
    frames = _frames(10, 40, 8, 12)
    fsz = 8 * 12
    write_cv2_avi(cv2, tmp_path / "y800.avi", frames, "Y800")
    # W = budget / frame bytes, rounded down to a multiple of batch_frames, at least batch_frames
    assert plan(tmp_path / "y800.avi", 48 * fsz, 16) == [0, 40]                      # fits: one window, today's path
    assert plan(tmp_path / "y800.avi", 40 * fsz, 16) == [0, 32, 40]
    assert plan(tmp_path / "y800.avi", 39 * fsz, 16) == [0, 32, 40]
    assert plan(tmp_path / "y800.avi", 10 * fsz + 5, 4) == [0, 8, 16, 24, 32, 40]
    assert plan(tmp_path / "y800.avi", 3 * fsz, 4) == [0, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40]
    assert plan(tmp_path / "y800.avi", 1, 16) == [0, 16, 32, 40]
    # FFV1, GOP 12: a window ends just before a keyframe
    encode_avi(cv2, tmp_path / "gop12.avi", frames, slices=(1, 1), gop=12)
    s = plan(tmp_path / "gop12.avi", 32 * fsz, 16)
    assert s == [0, 24, 40]
    assert all(a % 12 == 0 for a in s[:-1])
    assert plan(tmp_path / "gop12.avi", 16 * fsz, 4) == [0, 12, 24, 40]
    # a GOP longer than W widens its window to the GOP
    assert plan(tmp_path / "gop12.avi", 8 * fsz, 4) == [0, 12, 24, 36, 40]
    assert plan(tmp_path / "gop12.avi", 4 * fsz, 4) == [0, 12, 24, 36, 40]
    # intra-only: every frame is a keyframe, so windows are W long
    encode_avi(cv2, tmp_path / "intra.avi", frames, slices=(1, 1), gop=1)
    assert plan(tmp_path / "intra.avi", 16 * fsz, 8) == [0, 16, 32, 40]


@pytest.mark.parametrize("kind", ["y800", "bgr24", "mpng", "ffv1"])
def test_truncated_chunk_in_the_last_window_is_refused_at_index_time(tmp_path, kind):
    frames = _frames(13, 12, 16, 24)
    path = tmp_path / "v.avi"
    if kind == "bgr24":
        path.write_bytes(_dib_avi(np.repeat(frames[..., None], 3, axis=3), 24))
    elif kind == "ffv1":
        encode_avi(cv2, path, frames, slices=(1, 1), gop=4)
    else:
        write_cv2_avi(cv2, path, frames, {"y800": "Y800", "mpng": "MPNG"}[kind])
    data = path.read_bytes()
    idx1 = data.rfind(b"idx1")                    # the index after 'movi' names the frame chunks too
    idx1 = idx1 if idx1 >= 0 else len(data)
    last = max(data.rfind(b"00db", 0, idx1), data.rfind(b"00dc", 0, idx1))
    size = struct.unpack("<I", data[last + 4:last + 8])[0]
    bad = tmp_path / "bad.avi"
    bad.write_bytes(data[:last + 8 + size // 2])   # cut inside the last frame chunk
    with pytest.raises(RuntimeError, match="truncated frame"):
        read_range(bad, 0, 1)                     # only frame 0 is asked for
    with pytest.raises(RuntimeError, match="truncated frame"):
        plan(bad, 1, 1)
    dims, _, _ = read_range(path, 0, 1)
    assert int(dims[0]) == 12


def test_range_outside_the_video_is_refused(tmp_path):
    frames = _frames(14, 5, 4, 6)
    write_cv2_avi(cv2, tmp_path / "v.avi", frames, "Y800")
    with pytest.raises(RuntimeError, match="outside the video"):
        read_range(tmp_path / "v.avi", 3, 3)
