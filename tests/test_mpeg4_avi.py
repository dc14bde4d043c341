"""MPEG-4 Part 2 video read by host/lm_media.hpp with decode_mpeg4 on (lmh_read_video_mpeg4) and decoded by
csrc/mpeg4_format.h run on the CPU (lmh_decode_mpeg4, the code k_mpeg4.cu runs on the device): frames equal
cv2.VideoCapture's channel 0 for cv2-written 'XVID' / 'mp4v' video in AVI, Matroska and MP4, grey and colour, at several
sizes and quantisers; the colour rule holds for all 65 536 (Y, Cb) pairs and for frames whose sizes are not multiples of
16; every VLC table is a prefix code whose unused words all lie in the start-code region; what the decoder does not decode
is refused with the reason, malformed frames are named, and with the option off MPEG-4 keeps its "outside this library"
refusal.  The reader's I-VOP bits end the windows a long video is streamed through.  CPU only."""
import struct

import numpy as np
import pytest

from _containers import bitmapinfo, full, mkv, mov
from _mpeg4_avi import (T_DC_LUM, T_DC_CHROM, T_CBPY, T_MCBPC_I, Bits, Mpeg4Fuzz, before_vop, blue_table, decode_cpu, frames_of, mpeg4_avi, plan_mpeg4, read_video_mpeg4, segments, split, user_data,
                        vlc_table, vol, vop_type, with_vol, write_cv2_mpeg4)
from _png_avi import capture
from test_avi_ranges import read_range

cv2 = pytest.importorskip("cv2")


def _frames(seed, n, h, w, colour, noise=8.0, speed=3):
    """a smooth pattern drifting by `speed` pixels a frame, plus noise: more noise, coarser quantisers"""
    rng = np.random.Generator(np.random.PCG64(seed))
    yy, xx = np.mgrid[0:h, 0:w]
    out = []
    for i in range(n):
        f = 128 + 70 * np.sin((xx + speed * i) / 9.0) * np.cos((yy - 2 * i) / 7.0) + rng.normal(0, noise, (h, w))
        f = f.clip(0, 255).astype(np.uint8)
        out.append(np.dstack([f, np.roll(f, 5, 1), np.roll(f, -7, 0)]) if colour else f)
    return np.stack(out)


def _decoded(path):
    payload, offs, extra, _, (n, h, w) = read_video_mpeg4(path)
    return decode_cpu(extra, payload, offs, h, w)


KINDS = [("avi", "XVID"), ("avi", "mp4v"), ("mp4", "mp4v"), ("mkv", "XVID")]


@pytest.mark.parametrize("ext,fourcc", KINDS, ids=[f"{e}-{f}" for e, f in KINDS])
@pytest.mark.parametrize("colour", [False, True], ids=["grey", "colour"])
@pytest.mark.parametrize("h,w,noise,speed", [(400, 1700, 8.0, 3), (48, 64, 0.0, 1), (48, 64, 40.0, 7), (36, 44, 20.0, 5), (18, 30, 4.0, 2)])
def test_cv2_written(tmp_path, ext, fourcc, colour, h, w, noise, speed):
    n = 8 if w > 1000 else 30
    want = write_cv2_mpeg4(cv2, tmp_path / f"v.{ext}", _frames(h + w + int(noise), n, h, w, colour, noise, speed), fourcc)
    assert want.shape == (n, h, w)
    assert np.array_equal(_decoded(tmp_path / f"v.{ext}"), want)


def _y4m(path, y, cb):
    """one 4:2:0 frame as a .y4m file (C420jpeg); Cr is 128"""
    h, w = y.shape
    cr = np.full_like(cb, 128)
    path.write_bytes(f"YUV4MPEG2 W{w} H{h} F30:1 Ip A1:1 C420jpeg\n".encode() + b"FRAME\n" + y.tobytes() + cb.tobytes() + cr.tobytes())


def test_every_y_cb_pair(tmp_path):
    """VideoCapture's blue for 4:2:0 video is table(Y, Cb) with Cb nearest: one 512 x 512 frame holds all 65 536 pairs (each
    Cb sample over four Y samples), and the restated rule gives every one of them."""
    yy, xx = np.mgrid[0:512, 0:512]
    y = (((yy // 2) * 4 + (yy % 2) * 2 + (xx % 2)) % 256).astype(np.uint8)
    cb = np.tile(np.arange(256, dtype=np.uint8), (256, 1))
    _y4m(tmp_path / "all.y4m", y, cb)
    got = capture(cv2, tmp_path / "all.y4m")[0]
    cbf = np.repeat(np.repeat(cb, 2, 0), 2, 1)
    seen = np.zeros((256, 256), bool)
    seen[y, cbf] = True
    assert seen.all()
    assert np.array_equal(blue_table()[y, cbf], got)


@pytest.mark.parametrize("h,w", [(402, 1698), (400, 1712), (50, 34), (18, 30), (2, 2)])
def test_colour_rule_on_odd_tails(tmp_path, h, w):
    rng = np.random.Generator(np.random.PCG64(h * w))
    y = rng.integers(0, 256, (h, w), dtype=np.uint8)
    cb = rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8)
    _y4m(tmp_path / "r.y4m", y, cb)
    got = capture(cv2, tmp_path / "r.y4m")[0]
    assert np.array_equal(blue_table()[y, np.repeat(np.repeat(cb, 2, 0), 2, 1)], got)


# table id: (its entries, unused words of its longest length, leading zeros every unused word has)
TABLES = {0: (9, 7, 6), 1: (21, 1, 9), 2: (16, 2, 5), 3: (33, 2, 11), 4: (13, 1, 11), 5: (13, 1, 12), 6: (103, 8, 9), 7: (103, 8, 9)}


@pytest.mark.parametrize("t", sorted(TABLES), ids=["mcbpc_i", "mcbpc_p", "cbpy", "mvd", "dc_lum", "dc_chrom", "tcoef_intra", "tcoef_inter"])
def test_vlc_tables_are_prefix_codes(t):
    """No code is a prefix of another, and the only words no code covers are the zero runs that start codes need."""
    tab = vlc_table(t)
    count, holes, zeros = TABLES[t]
    assert len(tab) == count
    L = max(l for _, l in tab)
    cover = np.zeros(1 << L, np.int32)
    for c, l in tab:
        assert 0 <= c < (1 << l)
        cover[c << (L - l):(c + 1) << (L - l)] += 1
    assert cover.max() == 1
    unused = np.flatnonzero(cover == 0)
    assert unused.size == holes
    assert all(u < (1 << (L - zeros)) for u in unused)


def _cv2_avi(tmp_path, n=26, h=32, w=48, fourcc="XVID"):
    path = tmp_path / "base.avi"
    want = write_cv2_mpeg4(cv2, path, _frames(5, n, h, w, False, 10.0), fourcc)
    payload, offs, extra, ivop, dims = read_video_mpeg4(path)
    assert extra.size > 0  # the headers in front of frame 0's VOP: VOS, VO, VOL, user data
    return frames_of(payload, offs), want


def _refused(path, words):
    with pytest.raises(RuntimeError, match=words):
        read_video_mpeg4(path)


def test_refusals(tmp_path):
    frames, want = _cv2_avi(tmp_path)
    h, w = want.shape[1:]
    cases = [(dict(interlaced=1), "interlaced"), (dict(shape=1), "rectangular"), (dict(not_8_bit=1), "8-bit"), (dict(quant_type=1), "quant_type 1"),
             (dict(sprite=1), "sprites"), (dict(ver_id=2, qpel=1), "quarter-pel"), (dict(complexity_disable=0), "complexity estimation"),
             (dict(resync_disable=0), "resync markers"), (dict(partitioned=1), "data partitioning"), (dict(ver_id=2, newpred=1), "newpred"),
             (dict(ver_id=2, reduced=1), "reduced-resolution"), (dict(scalability=1), "scalable")]
    for i, (kw, words) in enumerate(cases):
        bad = [with_vol(f, vol(w, h, **kw)) for f in frames]
        (tmp_path / f"r{i}.avi").write_bytes(mpeg4_avi(bad, w, h))
        _refused(tmp_path / f"r{i}.avi", "frame 0: .*" + words)
        payload, offs = split(bad)
        with pytest.raises(ValueError, match="frame 0: .*" + words):
            decode_cpu(b"", payload, offs, h, w)
    # a VOL of another size than the container's, and a later VOL that differs from the first
    (tmp_path / "size.avi").write_bytes(mpeg4_avi([with_vol(f, vol(w + 16, h)) for f in frames], w, h))
    _refused(tmp_path / "size.avi", "frame 0: the VOL's frame size differs")
    changed = list(frames)
    changed[12] = with_vol(frames[12], vol(w, h, res=25))
    (tmp_path / "change.avi").write_bytes(mpeg4_avi(changed, w, h))
    _refused(tmp_path / "change.avi", "frame 12: the frame carries a VOL that differs")
    # B- and S-VOPs: the VOP's coding type
    for t, words in ((2, "B-VOPs"), (3, "S-VOPs")):
        bad = list(frames)
        at = bad[1].index(b"\0\0\1\xb6") + 4
        bad[1] = bad[1][:at] + bytes([(bad[1][at] & 0x3F) | (t << 6)]) + bad[1][at + 1:]
        (tmp_path / f"t{t}.avi").write_bytes(mpeg4_avi(bad, w, h))
        _refused(tmp_path / f"t{t}.avi", "frame 1: " + words)
    # short-header (H.263) frames, and a first frame that is not an I-VOP
    payload, offs = split([b"\0\0\x80\x02" + bytes(40)] + frames[1:])
    with pytest.raises(ValueError, match="frame 0: short-header"):
        decode_cpu(b"", payload, offs, h, w)
    extra = [frames[0][a:e] for c, a, e in segments(frames[0]) if 0x20 <= c <= 0x2F][0]
    payload, offs = split(frames[1:])
    with pytest.raises(ValueError, match="frame 0: the first frame is not an I-VOP"):
        decode_cpu(extra, payload, offs, h, w)
    # user data of encoders for which libavcodec changes its decoding
    for text in (b"XviD0050", b"DivX503b1393p", b"FFmpeg0.4.9-pre1b4718", b"Lavc0.0.1"):
        bad = [before_vop(frames[0], user_data(text))] + frames[1:]
        (tmp_path / "ud.avi").write_bytes(mpeg4_avi(bad, w, h))
        _refused(tmp_path / "ud.avi", "frame 0: the stream's user data names XviD, DivX or an old libavcodec")
    # an 'XVID' stream without libavcodec's user data is decoded by libavcodec with XviD's IDCT
    plain = [b"".join(f[a:e] for c, a, e in segments(f) if c != 0xB2) for f in frames]
    (tmp_path / "plain.avi").write_bytes(mpeg4_avi(plain, w, h))
    _refused(tmp_path / "plain.avi", "'XVID' MPEG-4 video without libavcodec's user data")
    (tmp_path / "plain_mp4v.avi").write_bytes(mpeg4_avi(plain, w, h, fourcc=b"FMP4"))
    assert np.array_equal(_decoded(tmp_path / "plain_mp4v.avi"), capture(cv2, tmp_path / "plain_mp4v.avi"))


def test_option_off_keeps_the_refusal(tmp_path):
    write_cv2_mpeg4(cv2, tmp_path / "v.avi", _frames(1, 3, 16, 32, True), "XVID")
    with pytest.raises(RuntimeError, match="outside this library.*decode_mpeg4: 1"):
        read_range(tmp_path / "v.avi", 0, 0)
    assert read_video_mpeg4(tmp_path / "v.avi")[4] == (3, 16, 32)


def test_malformed_frames_are_named(tmp_path):
    frames, want = _cv2_avi(tmp_path)
    h, w = want.shape[1:]
    start = frames[2].index(b"\0\0\1\xb6") + 12
    cases = [frames[2][:start + (len(frames[2]) - start) // 3],  # truncated
             frames[2][:start] + bytes(len(frames[2]) - start),  # zeros: no code of the MCBPC / CBPY / TCOEF tables
             frames[2][:start] + b"\xff" * (len(frames[2]) - start)]
    for bad in cases:
        payload, offs = split(frames[:2] + [bad] + frames[3:])
        with pytest.raises(ValueError, match="frame 2: (the frame's data ends|invalid VLC|coefficient run|intra DC|marker bit)"):
            decode_cpu(b"", payload, offs, h, w)
    payload, offs = split(frames)
    assert np.array_equal(decode_cpu(b"", payload, offs, h, w), want)


def _not_coded_vop(increment):
    """a P-VOP header with vop_coded 0 (30 ticks a second: 5 bits of time increment)"""
    b = Bits()
    b.put(1, 2), b.put(0, 1), b.put(1, 1), b.put(increment, 5), b.put(1, 1), b.put(0, 1)
    return b"\0\0\1\xb6" + b.stuffed()


def test_not_coded_vops_are_left_out(tmp_path):
    """VideoCapture returns no frame for a not-coded VOP: the reader leaves it out, so the frames stay one for one; the
    decoder refuses one it is given."""
    frames, want = _cv2_avi(tmp_path, n=20)
    h, w = want.shape[1:]
    with_n = frames[:6] + [_not_coded_vop(6)] + frames[6:]
    (tmp_path / "n.avi").write_bytes(mpeg4_avi(with_n, w, h))
    assert np.array_equal(capture(cv2, tmp_path / "n.avi"), want)
    assert np.array_equal(_decoded(tmp_path / "n.avi"), want)
    payload, offs = split(with_n)
    with pytest.raises(ValueError, match="frame 6: not-coded VOP"):
        decode_cpu(b"", payload, offs, h, w)


def test_ivop_bits_and_windows(tmp_path):
    """cv2 writes GOPs of 12 (I then 11 P-VOPs); the reader records each frame's I-VOP bit, and windows end before an I-VOP."""
    path = tmp_path / "v.avi"
    want = write_cv2_mpeg4(cv2, path, _frames(2, 40, 32, 48, False), "XVID")
    payload, offs, extra, ivop, (n, h, w) = read_video_mpeg4(path)
    types = [vop_type(f) for f in frames_of(payload, offs)]
    assert types == [0 if i % 12 == 0 else 1 for i in range(40)]
    assert list(ivop) == [int(t == 0) for t in types]
    assert plan_mpeg4(path, 20 * h * w, 4) == [0, 12, 24, 40]  # the last window holds the rest
    assert plan_mpeg4(path, 8 * h * w, 4) == [0, 12, 24, 36, 40]  # a GOP longer than a window is one window
    # each GOP decodes on its own with the VOL the reader keeps
    for a, b in ((0, 12), (12, 24), (24, 36), (36, 40)):
        p, o = split(frames_of(payload, offs)[a:b])
        assert np.array_equal(decode_cpu(extra, p, o, h, w), want[a:b])


@pytest.mark.parametrize("kind", ["mkv-vfw", "mp4-esds"])
def test_hand_written_containers(tmp_path, kind):
    """The frames of a cv2-written AVI (VOL in frame 0) in a Matroska V_MS/VFW/FOURCC track, and in an MP4 'mp4v' track whose
    esds holds the VOL (DecoderSpecificInfo) and whose frames do not."""
    frames, want = _cv2_avi(tmp_path, n=14)
    h, w = want.shape[1:]
    if kind == "mkv-vfw":
        path = tmp_path / "v.mkv"
        path.write_bytes(mkv(frames, "V_MS/VFW/FOURCC", w, h, private=bitmapinfo(w, h, b"XVID", 24)))
    else:
        head = [f[:f.index(b"\0\0\1\xb6")] for f in frames]
        dsi = head[0]
        bare = [f[len(hd):] for f, hd in zip(frames, head)]

        def descr(tag, body):
            return bytes([tag, 0x80, 0x80, 0x80, len(body)]) + body
        esds = full(b"esds", descr(3, struct.pack(">HB", 1, 0) + descr(4, bytes([0x20, 0x11, 0, 0, 0]) + struct.pack(">II", 0, 0) + descr(5, dsi)) +
                                    descr(6, b"\x02")))
        path = tmp_path / "v.mp4"
        path.write_bytes(mov(bare, b"mp4v", w, h, children=esds, mp4=True))
    assert np.array_equal(capture(cv2, path), want)
    assert np.array_equal(_decoded(path), want)


FUZZ_SIZES = [(16, 16), (32, 48), (48, 64), (18, 30), (2, 2), (2, 31), (8, 1), (34, 45), (50, 17), (64, 96)]


def fuzz_stream(h, w, seed):
    """two GOPs (I + 7 P, I + 3 P) of random syntax; levels up to 3, see DESIGN §8 on larger ones"""
    F = Mpeg4Fuzz(w, h, seed, levels=3)
    frames = [F.headers() + F.vop(0)] + [F.vop(1) for _ in range(7)] + [F.headers() + F.vop(0)] + [F.vop(1) for _ in range(3)]
    return F, frames


@pytest.mark.parametrize("h,w", FUZZ_SIZES, ids=[f"{h}x{w}" for h, w in FUZZ_SIZES])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_syntax_streams(tmp_path, h, w, seed):
    """The test encoder's streams (dquant, ac_pred beside other quantisers, DC in the TCOEF table, all escapes, every
    f_code, wrapping vectors past every edge, intra and not_coded macroblocks in P-VOPs, both rounding types, widths 1-31):
    read back through VideoCapture, both decoders give its frames."""
    F, frames = fuzz_stream(h, w, seed)
    (tmp_path / "f.avi").write_bytes(mpeg4_avi(frames, w, h, fourcc=b"FMP4"))
    want = capture(cv2, tmp_path / "f.avi")
    assert want.shape == (len(frames), h, w)
    payload, offs = split(frames)
    assert np.array_equal(decode_cpu(b"", payload, offs, h, w), want)
    assert np.array_equal(_decoded(tmp_path / "f.avi"), want)
    if (h, w) == (48, 64):
        u = F.used
        assert all(u[k] > 0 for k in ("dquant", "ac_pred", "dc_in_tcoef", "esc1", "esc2", "esc3", "intra_in_p", "not_coded")), u
        assert u["rounding"] == {0, 1} and len(u["fcodes"]) >= 4, u


def test_negative_intra_dc_is_an_error(tmp_path):
    """libavcodec treats an intra DC that predicts below 0 as an error (and conceals the frame); it is refused here."""
    F = Mpeg4Fuzz(16, 16, 0)
    b = Bits()
    b.put(0, 2), b.put(0, 1), b.put(1, 1), b.put(0, 5), b.put(1, 1), b.put(1, 1), b.put(0, 3), b.put(2, 5)
    F._put(b, T_MCBPC_I, 0), b.put(0, 1), F._put(b, T_CBPY, 0)
    F._put(b, T_DC_LUM, 8), b.put(126, 8)  # -129: below the predictor 128
    for k in range(1, 6):
        F._put(b, T_DC_LUM if k < 4 else T_DC_CHROM, 0)
    payload, offs = split([F.headers() + b"\0\0\1\xb6" + b.stuffed()])
    with pytest.raises(ValueError, match="frame 0: intra DC .*negative"):
        decode_cpu(b"", payload, offs, 16, 16)


def test_lowercase_xvid_without_libavcodec_user_data_is_refused(tmp_path):
    """libavcodec upper-cases the codec tag before it picks XviD's decoding for a stream without its user data"""
    frames, want = _cv2_avi(tmp_path)
    h, w = want.shape[1:]
    plain = [b"".join(f[a:e] for c, a, e in segments(f) if c != 0xB2) for f in frames]
    for fourcc in (b"xvid",):
        (tmp_path / "p.avi").write_bytes(mpeg4_avi(plain, w, h, fourcc=fourcc))
        _refused(tmp_path / "p.avi", "MPEG-4 video without libavcodec's user data")


def test_odd_heights_are_refused(tmp_path):
    F, frames = fuzz_stream(16, 16, 0)
    bad = [with_vol(f, vol(16, 15)) for f in frames]
    (tmp_path / "o.avi").write_bytes(mpeg4_avi(bad, 16, 15, fourcc=b"FMP4"))
    _refused(tmp_path / "o.avi", "frame 0: odd frame heights")
