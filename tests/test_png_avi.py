"""PNG-coded AVI ('MPNG' / 'png ') frame chunks read by host/lm_media.hpp (lmh_read_avi_png): as many frames as
cv2.VideoCapture reads, each payload slice a PNG that cv2.imdecode turns into that frame; frames lm_decode_png cannot decode
(16-bit, palette, interlaced, a size other than frame 0's) refused with a message.  CPU only."""
import struct
import zlib

import numpy as np
import pytest

from _png_avi import capture, png_avi, png_from_zlib, read_avi_png, write_cv2_avi

cv2 = pytest.importorskip("cv2")


def _check_slices(path, want):
    payload, offs, dims = read_avi_png(path)
    assert dims == want.shape[:3] and offs.size == want.shape[0] + 1 and offs[-1] == payload.size
    for i in range(dims[0]):
        im = cv2.imdecode(payload[offs[i]:offs[i + 1]], cv2.IMREAD_COLOR if want.ndim == 4 else cv2.IMREAD_UNCHANGED)
        assert np.array_equal(im if want.ndim == 4 else im.reshape(want.shape[1:]), want[i])


@pytest.mark.parametrize("fourcc", ["MPNG", "png "])
@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("width,n", [(2, 1), (32, 50), (1700, 1), (1700, 50)])
def test_cv2_written_avi(tmp_path, fourcc, colour, width, n):
    rng = np.random.Generator(np.random.PCG64(width * 100 + n))
    h = 40 if width == 1700 and n == 50 else 17
    shape = (n, h, width, 3) if colour else (n, h, width)
    frames = rng.integers(0, 256, shape, dtype=np.uint8)
    write_cv2_avi(cv2, tmp_path / "v.avi", frames, fourcc)
    cap = cv2.VideoCapture(str(tmp_path / "v.avi"))
    read = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        read.append(f if colour else f[..., 0])
    assert len(read) == n
    _check_slices(tmp_path / "v.avi", np.stack(read))


@pytest.mark.parametrize("width", [1, 31])
@pytest.mark.parametrize("colour", [False, True])
def test_hand_built_avi_with_widths_the_writer_cannot_produce(tmp_path, width, colour):
    rng = np.random.Generator(np.random.PCG64(width))
    frames = rng.integers(0, 256, (6, 9, width, 3) if colour else (6, 9, width), dtype=np.uint8)
    pngs = [cv2.imencode(".png", f)[1].tobytes() for f in frames]
    (tmp_path / "v.avi").write_bytes(png_avi(pngs, width, 9, fourcc=b"png ", empty_at=(3,)))   # zero-size chunks are skipped
    assert capture(cv2, tmp_path / "v.avi").shape[0] == 6
    _check_slices(tmp_path / "v.avi", frames)


def _raw(h, w, bpp=1):
    return zlib.compress(b"".join(b"\0" + bytes(w * bpp) for _ in range(h)))


def _plte_png(w, h):
    png = png_from_zlib(_raw(h, w), w, h, ctype=3)
    plte = struct.pack(">I", 6) + b"PLTE" + bytes(6) + struct.pack(">I", zlib.crc32(b"PLTE" + bytes(6)))
    return png[:33] + plte + png[33:]


@pytest.mark.parametrize("make,words", [
    (lambda: png_from_zlib(_raw(5, 8, 2), 8, 5, depth=16), "bit depth 16"),
    (lambda: _plte_png(8, 5), "colour type 3"),
    (lambda: png_from_zlib(_raw(5, 8), 8, 5, interlace=1), "interlaced"),
    (lambda: png_from_zlib(_raw(6, 8), 8, 6), "frame 0 has 8 x 5"),
    (lambda: b"not a png at all" * 4, "not a PNG"),
])
def test_undecodable_frames_are_refused(tmp_path, make, words):
    good = png_from_zlib(_raw(5, 8), 8, 5)
    (tmp_path / "v.avi").write_bytes(png_avi([good, good, make()], 8, 5))
    with pytest.raises(RuntimeError, match=r"frame 2: .*" + words):
        read_avi_png(tmp_path / "v.avi")


def test_raw_reader_points_png_streams_elsewhere(tmp_path):
    from test_host_media import _read

    good = png_from_zlib(_raw(5, 8), 8, 5)
    (tmp_path / "v.avi").write_bytes(png_avi([good], 8, 5))
    with pytest.raises(RuntimeError, match="PNG-coded"):
        _read("lmh_read_avi", tmp_path / "v.avi")
