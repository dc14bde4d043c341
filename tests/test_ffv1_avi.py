"""FFV1-coded AVI ('FFV1') read by host/lm_media.hpp (lmh_read_avi_ffv1) and decoded by csrc/ffv1_format.h run on the CPU
(lmh_decode_ffv1, the same code k_ffv1.cu runs per thread): frames equal cv2.VideoCapture's channel 0 for cv2-written
grey and colour video and for streams of the test encoder (range coders with the default and a custom table, the large
context model, coded initial states, intra-only, uneven slice grids); the configuration record is checked and what the
device decoder does not decode is refused with the reason.  CPU only."""
import numpy as np
import pytest

from _ffv1_avi import LARGE, Encoder, decode_cpu, encode_avi, ffv1_avi, make_slice, read_avi_ffv1, split_slices, strf_record, write_cv2_ffv1

cv2 = pytest.importorskip("cv2")


def _frames(seed, n, h, w, colour):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = rng.integers(0, 256, (h, w, 3) if colour else (h, w), dtype=np.uint8)
    base[h // 3: h // 2] = 40  # a flat band: run mode (Golomb-Rice) and context 0
    return np.stack([np.roll(base, 2 * i, axis=1) + rng.integers(0, 3, base.shape, dtype=np.uint8) for i in range(n)])


@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("w,h,n", [(1700, 400, 1), (64, 24, 13), (36, 10, 50)])
def test_cv2_written_avi(tmp_path, colour, w, h, n):
    want = write_cv2_ffv1(cv2, tmp_path / "v.avi", _frames(w + n, n, h, w, colour))
    ex, payload, offs, dims = read_avi_ffv1(tmp_path / "v.avi")
    assert dims == want.shape and offs[-1] == payload.size and len(ex) == 42
    assert np.array_equal(decode_cpu(ex, payload, offs, h, w), want)


@pytest.mark.parametrize("kw", [dict(coder=1), dict(coder=2), dict(model=LARGE), dict(model=LARGE, coder=1), dict(gop=1),
                                dict(coder=1, initial_states=True), dict(slices=(3, 5)), dict(slices=(1, 1), gop=4)],
                         ids=["range", "range-custom", "large", "large-range", "intra", "initial-states", "grid-3x5", "one-slice"])
@pytest.mark.parametrize("colour", [False, True])
def test_hand_built_streams(tmp_path, kw, colour):
    frames = _frames(3, 14, 21, 31, colour)
    _, _, want = encode_avi(cv2, tmp_path / "v.avi", frames, **kw)
    ex, payload, offs, dims = read_avi_ffv1(tmp_path / "v.avi")
    assert dims == want.shape
    assert np.array_equal(decode_cpu(ex, payload, offs, 21, 31), want)


def test_width_one_and_empty_chunks(tmp_path):
    frames = _frames(4, 5, 9, 1, False)
    rec, fr = Encoder(False, slices=(1, 3), gop=3).encode(frames)
    (tmp_path / "v.avi").write_bytes(ffv1_avi(fr, 1, 9, rec, empty_at=(2,)))
    ex, payload, offs, dims = read_avi_ffv1(tmp_path / "v.avi")
    assert dims == (5, 9, 1)
    assert np.array_equal(decode_cpu(ex, payload, offs, 9, 1), frames)


def _refused(tmp_path, rec, frames, w, h, words):
    (tmp_path / "v.avi").write_bytes(ffv1_avi(frames, w, h, rec))
    with pytest.raises(RuntimeError, match=words):
        read_avi_ffv1(tmp_path / "v.avi")


def test_refusals(tmp_path):
    frames = _frames(5, 3, 8, 12, False)
    enc = Encoder(False, slices=(2, 2))
    _, fr = enc.encode(frames)
    _refused(tmp_path, enc.record(colorspace=0, chroma_planes=1), fr, 12, 8, "YUV with chroma planes")
    _refused(tmp_path, enc.record(bits=16), fr, 12, 8, "16 bits per sample")
    _refused(tmp_path, enc.record(version=2), fr, 12, 8, "version 2")
    _refused(tmp_path, enc.record(version=4), fr, 12, 8, "version 4")
    bad = bytearray(enc.record())
    bad[5] ^= 0x10
    _refused(tmp_path, bytes(bad), fr, 12, 8, "CRC mismatch")
    _refused(tmp_path, b"", fr, 12, 8, "versions 0 and 1")
    _refused(tmp_path, enc.record(), fr[1:], 12, 8, "not a keyframe")


def test_record_of_cv2_writer(tmp_path):
    """The record OpenCV writes parses (version 3, Golomb-Rice, 4 x 2 slices, ec) and a flipped bit anywhere is refused."""
    write_cv2_ffv1(cv2, tmp_path / "v.avi", _frames(6, 2, 400, 1700, True))
    data = (tmp_path / "v.avi").read_bytes()
    rec, at = strf_record(data)
    assert len(rec) == 42
    ex, payload, offs, _ = read_avi_ffv1(tmp_path / "v.avi")
    assert len(split_slices(payload[offs[0]:offs[1]].tobytes(), 8)) == 8
    for i in (0, 20, 41):
        b = bytearray(data)
        b[at + i] ^= 1
        (tmp_path / "b.avi").write_bytes(bytes(b))
        with pytest.raises(RuntimeError, match="configuration record"):
            read_avi_ffv1(tmp_path / "b.avi")


def test_cpu_decoder_names_a_bad_slice(tmp_path):
    frames = _frames(8, 4, 16, 24, False)
    rec, fr = Encoder(False).encode(frames)
    sl = split_slices(fr[2], 8)
    sl[5] = sl[5][:-1] + bytes([sl[5][-1] ^ 1])
    fr[2] = b"".join(sl)
    pay = np.frombuffer(b"".join(fr), np.uint8)
    offs = np.concatenate([[0], np.cumsum([len(f) for f in fr])]).astype(np.int64)
    with pytest.raises(ValueError, match="frame 2, slice 5: slice CRC mismatch"):
        decode_cpu(np.frombuffer(rec, np.uint8), pay, offs, 16, 24)
    enc = Encoder(False)
    head = (enc.encode(frames[:2]), enc.head_bytes[3])[1]
    sl = split_slices(fr[1], 8)
    sl[3] = make_slice(sl[3][:head] + bytes(len(sl[3]) - 8 - head))  # the header, then a run of Golomb escapes that outlasts the slice
    fr[1], fr[2] = b"".join(sl), Encoder(False).encode(frames)[1][2]
    pay = np.frombuffer(b"".join(fr), np.uint8)
    offs = np.concatenate([[0], np.cumsum([len(f) for f in fr])]).astype(np.int64)
    with pytest.raises(ValueError, match="frame 1, slice 3: the slice data ends"):
        decode_cpu(np.frombuffer(rec, np.uint8), pay, offs, 16, 24)
