"""Matroska and QuickTime / MP4 video (host/lm_containers.hpp, through lmmedia::index_video): every accepted file gives the
frame count cv2.VideoCapture reports and reads, and the frames VideoCapture + extractChannel(0) gives -- raw frames from the
reader, PNG chunks through cv2.imdecode, FFV1 chunks through the CPU build of ffv1_format.h.  Ranges and window plans agree
with the whole read.  Every refusal names the file and the reason.  The container is chosen by signature, not extension."""
import numpy as np
import pytest

from _containers import (bitmapinfo, box, check_capture, esds_png, frame_count, mkv, mov, png_frames, write_cv2)
from _ffv1_avi import Encoder, decode_cpu, read_avi_ffv1
from _png_avi import capture, write_cv2_avi
from test_avi_ranges import joined, plan, random_cuts, read_range

cv2 = pytest.importorskip("cv2")

# the rows of cv2.VideoWriter files: (extension, fourcc, colour allowed)
CV2_ROWS = [("mkv", "FFV1", True), ("mkv", "png ", True), ("mkv", "Y800", False), ("mov", "png ", True), ("mov", "FFV1", True),
            ("mov", "Y800", False), ("mp4", "png ", True)]


def _frames(seed, n, h, w, colour=False):
    rng = np.random.Generator(np.random.PCG64(seed))
    shape = (n, h, w, 3) if colour else (n, h, w)
    base = rng.integers(0, 256, shape, dtype=np.uint8)
    return np.where(rng.random(shape) < 0.6, base // 32 * 32, base).astype(np.uint8)


def decoded(path):
    """Channel 0 of every frame as this library reads the file: raw pixels, or the coded chunks decoded on the CPU."""
    dims = read_range(path, 0, 0)[0]
    n, rows, cols, codec = (int(v) for v in dims[:4])
    _, data, offs = read_range(path, 0, n)
    if codec == 0:
        return data.reshape(n, rows, cols)
    if codec == 1:
        out = []
        for a, b in zip(offs[:-1], offs[1:]):
            img = cv2.imdecode(data[a:b], cv2.IMREAD_UNCHANGED)
            out.append(img if img.ndim == 2 else img[..., 0])
        return np.stack(out)
    ex, payload, offsets, (n2, r2, c2) = read_avi_ffv1(path)
    assert (n2, r2, c2) == (n, rows, cols) and np.array_equal(payload, data) and np.array_equal(offsets, offs)
    return decode_cpu(ex, payload, offsets, rows, cols)


def check_accepted(path):
    """The index count equals CAP_PROP_FRAME_COUNT and the frames VideoCapture reads, and so do the frames."""
    want = capture(cv2, path)
    n = int(read_range(path, 0, 0)[0][0])
    assert n == frame_count(cv2, path) == want.shape[0], path
    got = decoded(path)
    assert got.shape == want.shape and np.array_equal(got, want), path
    return want


@pytest.mark.parametrize("n", [1, 25])
@pytest.mark.parametrize("fps", [30000 / 1001, 400.0, 1.0], ids=["29.97", "400", "1"])
@pytest.mark.parametrize("colour", [False, True], ids=["grey", "colour"])
@pytest.mark.parametrize("ext,fourcc", [(e, f) for e, f, _ in CV2_ROWS], ids=[f"{e}-{f.strip()}" for e, f, _ in CV2_ROWS])
def test_cv2_written_files(tmp_path, ext, fourcc, colour, fps, n):
    if colour and not dict(((e, f), c) for e, f, c in CV2_ROWS)[(ext, fourcc)]:
        pytest.skip("cv2 writes colour Y800 as planar YUV")
    path = tmp_path / f"v.{ext}"
    frames = _frames(n + int(fps), n, 24, 40, colour)
    want = write_cv2(cv2, path, frames, fourcc, fps)
    got = check_accepted(path)
    expect = frames[..., 0] if colour else frames   # grey 'raw ' in QuickTime is stored inverted (255 - v) and read back so
    assert np.array_equal(got, expect) and np.array_equal(want, expect)


def test_opencv_frame_count_rule_is_pinned(tmp_path):
    """OpenCV's estimate floor(duration * fps + 0.5) from the segment Duration and av_reduce(1e9, DefaultDuration, 30000):
    at every rate and length here it equals the frames in the file, and the index agrees."""
    for fps in (30000 / 1001, 400.0, 1.0, 25.0, 59.94, 1000.0, 0.5):
        for n in (1, 2, 7, 101):
            path = tmp_path / f"v{fps}_{n}.mkv"
            write_cv2(cv2, path, _frames(n, n, 8, 16), "FFV1", fps)
            assert int(read_range(path, 0, 0)[0][0]) == frame_count(cv2, path) == n, (fps, n)


def _gop_mkv(path, frames, gop, **kw):
    rec, fr = Encoder(frames.ndim == 4, slices=(1, 1), gop=gop).encode(frames)
    h, w = frames.shape[1:3]
    path.write_bytes(mkv(fr, "V_FFV1", w, h, private=rec, **kw))
    check_capture(cv2, path, frames)


HAND_WRITTEN = ["mkv_unknown_sizes", "mkv_block_group", "mkv_audio_first", "mkv_void_crc", "mkv_all", "mkv_vfw_y800", "mkv_vfw_bgr",
                "mkv_vfw_ffv1", "mkv_unc_bgr24", "mkv_unc_rgb24", "mkv_unc_grey_padded", "mov_co64", "mov_stsc_runs", "mov_moov_first",
                "mov_moov_last_large_mdat", "mov_single_size", "mov_raw_rgb24", "mov_raw_grey_padded", "mov_ffv1_glbl", "mp4_mp4v_png",
                "mov_no_edit_list"]


@pytest.mark.parametrize("kind", HAND_WRITTEN)
def test_hand_written_files(tmp_path, kind):
    g, c = _frames(3, 12, 9, 13), _frames(4, 12, 9, 13, True)
    pngs = png_frames(cv2, c)
    vfw_png = dict(private=bitmapinfo(13, 9, b"png ", 24))
    pad = lambda f: np.pad(f.reshape(9, -1), ((0, 0), (0, -f.reshape(9, -1).shape[1] % 4))).tobytes()   # rows to 4 bytes
    path = tmp_path / ("v." + kind[:3])
    want = c[..., 0]
    layouts = {"mkv_unknown_sizes": dict(unknown_sizes=True), "mkv_block_group": dict(block_group=True), "mkv_audio_first": dict(audio_first=True),
               "mkv_void_crc": dict(void_crc=True), "mkv_all": dict(unknown_sizes=True, block_group=True, audio_first=True, void_crc=True)}
    if kind in layouts:
        data = mkv(pngs, "V_MS/VFW/FOURCC", 13, 9, cluster_frames=5, **vfw_png, **layouts[kind])
    elif kind == "mkv_vfw_y800":
        data, want = mkv([f.tobytes() for f in g], "V_MS/VFW/FOURCC", 13, 9, private=bitmapinfo(13, 9, b"Y800", 8)), g
    elif kind == "mkv_vfw_bgr":
        data = mkv([pad(f) for f in c], "V_MS/VFW/FOURCC", 13, 9, private=bitmapinfo(13, 9, 0, 24))
    elif kind == "mkv_vfw_ffv1":
        rec, fr = Encoder(False, slices=(2, 1), gop=5).encode(g)
        data, want = mkv(fr, "V_MS/VFW/FOURCC", 13, 9, private=bitmapinfo(13, 9, b"FFV1", 24, rec)), g
    elif kind == "mkv_unc_bgr24":
        data = mkv([f.tobytes() for f in c], "V_UNCOMPRESSED", 13, 9, colour=b"BGR\x18")
    elif kind == "mkv_unc_rgb24":
        data = mkv([f[..., ::-1].tobytes() for f in c], "V_UNCOMPRESSED", 13, 9, colour=b"RGB\x18", block_group=True)
    elif kind == "mkv_unc_grey_padded":
        data, want = mkv([pad(f) for f in g], "V_UNCOMPRESSED", 13, 9, colour=b"Y800"), g
    elif kind == "mov_co64":
        data = mov(pngs, b"png ", 13, 9, co64=True, chunks=[5, 5, 2])
    elif kind == "mov_stsc_runs":
        data = mov(pngs, b"MPNG", 13, 9, chunks=[3, 3, 1, 1, 2, 2])
    elif kind == "mov_moov_first":
        data = mov(pngs, b"png ", 13, 9, moov_first=True, chunks=[4, 4, 4])
    elif kind == "mov_moov_last_large_mdat":
        data = mov(pngs, b"png ", 13, 9, large_mdat=True, co64=True, chunks=[7, 5])
    elif kind == "mov_single_size":
        same = [pngs[0]] * 12
        data, want = mov(same, b"png ", 13, 9, single_size=True, chunks=[6, 6]), np.repeat(c[:1, ..., 0], 12, 0)
    elif kind == "mov_raw_rgb24":
        data = mov([pad(f[..., ::-1]) for f in c], b"raw ", 13, 9, depth=24, chunks=[2] * 6)
    elif kind == "mov_raw_grey_padded":
        data, want = mov([pad(f) for f in g], b"raw ", 13, 9, depth=40), 255 - g
    elif kind == "mov_ffv1_glbl":
        rec, fr = Encoder(True, slices=(1, 2), gop=4).encode(c)
        data = mov(fr, b"FFV1", 13, 9, children=box(b"glbl", rec), chunks=[4, 4, 4], moov_first=True)
    elif kind == "mp4_mp4v_png":
        data = mov(pngs, b"mp4v", 13, 9, children=esds_png(), mp4=True, chunks=[6, 6])
    elif kind == "mov_no_edit_list":
        data = mov(pngs, b"png ", 13, 9, edit=None)
    path.write_bytes(data)
    check_capture(cv2, path, want)
    check_accepted(path)


def test_ranges_and_window_plans_agree_with_the_whole_read(tmp_path):
    rng = np.random.Generator(np.random.PCG64(21))
    frames = _frames(5, 40, 8, 12)
    _gop_mkv(tmp_path / "gop12.mkv", frames, 12, unknown_sizes=True, cluster_frames=7)
    tmp = tmp_path / "gop12.mov"
    rec, fr = Encoder(False, slices=(1, 1), gop=12).encode(frames)
    tmp.write_bytes(mov(fr, b"FFV1", 12, 8, children=box(b"glbl", rec), chunks=[9, 9, 9, 9, 4]))
    for path in (tmp_path / "gop12.mkv", tmp):
        whole = joined(path, [0, 40])
        for k in (1, 5, 39):
            part = joined(path, random_cuts(rng, 40, k))
            assert part[0] == "ffv1" and part[1].tobytes() == whole[1].tobytes() and np.array_equal(part[2], whole[2])
        fsz = 8 * 12
        assert plan(path, 32 * fsz, 16) == [0, 24, 40]          # windows end just before a keyframe
        assert plan(path, 16 * fsz, 4) == [0, 12, 24, 40]
        assert plan(path, 4 * fsz, 4) == [0, 12, 24, 36, 40]    # a GOP longer than a window is one window
    raw = tmp_path / "raw.mov"
    g = _frames(6, 30, 9, 13)
    raw.write_bytes(mov([f.tobytes() for f in g], b"raw ", 13, 9, depth=40, chunks=[7, 7, 7, 9]))
    for k in (1, 4, 29):
        assert joined(raw, random_cuts(rng, 30, k))[1].tobytes() == (255 - g).tobytes()
    assert plan(raw, 10 * 9 * 13, 4) == [0, 8, 16, 24, 30]


def _refused(path, *words):
    with pytest.raises(RuntimeError) as e:
        read_range(path, 0, 1)
    msg = str(e.value)
    assert str(path) in msg, msg
    for w in words:
        assert w in msg, msg
    with pytest.raises(RuntimeError):
        plan(path, 1, 1)
    return msg


def test_refusals_name_the_file_and_the_reason(tmp_path):
    c = _frames(7, 10, 9, 13, True)
    pngs = png_frames(cv2, c)
    vfw = dict(private=bitmapinfo(13, 9, b"png ", 24))
    cases = {
        "laced.mkv": (mkv(pngs, "V_MS/VFW/FOURCC", 13, 9, laced_at=3, **vfw), ["frame 3", "laced"]),
        # a gap in the timestamps: OpenCV counts 13 frames from the duration, but reads 10
        "gap.mkv": (mkv(pngs, "V_MS/VFW/FOURCC", 13, 9, timecodes_ms=[0, 33, 67, 100, 133, 167, 200, 234, 267, 400], **vfw),
                    ["holds 10 frames", "OpenCV would count 13"]),
        "no_duration.mkv": (mkv(pngs, "V_MS/VFW/FOURCC", 13, 9, with_duration=False, **vfw), ["no segment Duration"]),
        "encoded.mkv": (mkv(pngs, "V_MS/VFW/FOURCC", 13, 9, content_encoding=True, **vfw), ["ContentEncoding"]),
        "yuv.mkv": (mkv([b"\0" * 176] * 10, "V_UNCOMPRESSED", 13, 9, colour=b"I420"), ["ColourSpace 'I420'", "outside this library"]),
        "edit_offset.mov": (mov(pngs, b"png ", 13, 9, edit=[(334, 1001)]), ["edit list"]),
        "edit_short.mov": (mov(pngs, b"png ", 13, 9, edit=[(200, 0)]), ["edit list"]),
        "edit_two.mov": (mov(pngs, b"png ", 13, 9, edit=[(100, 0), (234, 3003)]), ["edit list"]),
        "fragmented.mp4": (mov(pngs, b"png ", 13, 9, moof=True, mp4=True), ["fragmented"]),
        "ctts.mov": (mov(pngs, b"png ", 13, 9, ctts=[0, 2002] * 5), ["ctts"]),
        "mp4v_mpeg4.mp4": (mov(pngs, b"mp4v", 13, 9, mp4=True, children=esds_png().replace(bytes([0x6D, 0x11]), bytes([0x20, 0x11]))),
                           ["'mp4v' with object type 32", "outside this library"]),
        "raw_pal8.mov": (mov([b"\0" * 117] * 10, b"raw ", 13, 9, depth=8), ["depth 8", "outside this library"]),
    }
    for name, (data, words) in cases.items():
        (tmp_path / name).write_bytes(data)
        _refused(tmp_path / name, *words)
    # the non-identity edit lists drop frames in VideoCapture; the gap makes its count differ from the frames it reads
    for name in ("edit_offset.mov", "edit_short.mov"):
        assert capture(cv2, tmp_path / name).shape[0] < 10
    assert frame_count(cv2, tmp_path / "gap.mkv") == 13 and capture(cv2, tmp_path / "gap.mkv").shape[0] == 10


@pytest.mark.parametrize("ext", ["mkv", "mov"])
def test_mjpeg_is_outside_this_library(tmp_path, ext):
    path = tmp_path / f"v.{ext}"
    write_cv2(cv2, path, _frames(8, 5, 16, 24, True), "MJPG")
    _refused(path, "outside this library", "V_MJPEG" if ext == "mkv" else "'jpeg'")


@pytest.mark.parametrize("kind", ["mkv_cv2", "mkv_unknown_sizes", "mov_cv2", "mov_moov_first", "mp4_cv2"])
def test_truncation_anywhere_is_refused_at_index_time(tmp_path, kind):
    frames = _frames(9, 12, 16, 24)
    path = tmp_path / ("v." + kind[:3])
    if kind == "mkv_unknown_sizes":
        _gop_mkv(path, frames, 4, unknown_sizes=True)
    elif kind == "mov_moov_first":
        rec, fr = Encoder(False, slices=(1, 1), gop=4).encode(frames)
        path.write_bytes(mov(fr, b"FFV1", 24, 16, children=box(b"glbl", rec), moov_first=True, chunks=[4, 4, 4]))
    else:
        write_cv2(cv2, path, frames, "FFV1" if kind != "mp4_cv2" else "png ")
    data = path.read_bytes()
    assert int(read_range(path, 0, 1)[0][0]) == 12
    rng = np.random.Generator(np.random.PCG64(len(data)))
    cuts = sorted(set(rng.integers(8, len(data) - 1, 40).tolist()) | {len(data) - 1, len(data) // 2, 9})   # past the signature
    bad = tmp_path / ("bad." + kind[:3])
    for cut in cuts:
        bad.write_bytes(data[:cut])
        with pytest.raises(RuntimeError) as e:
            read_range(bad, 0, 1)
        msg = str(e.value)
        assert str(bad) in msg and ("truncated" in msg or "no 'moov' box" in msg), (cut, msg)


def test_container_is_chosen_by_signature(tmp_path):
    frames = _frames(10, 6, 16, 24)
    write_cv2(cv2, tmp_path / "a.mkv", frames, "FFV1")
    write_cv2(cv2, tmp_path / "b.mov", frames, "png ")
    write_cv2_avi(cv2, tmp_path / "c.avi", frames, "Y800")
    for src, dst, codec in (("a.mkv", "a.avi", 2), ("b.mov", "b.mkv", 1), ("c.avi", "c.mov", 0)):
        (tmp_path / dst).write_bytes((tmp_path / src).read_bytes())
        dims = read_range(tmp_path / dst, 0, 0)[0]
        assert int(dims[0]) == 6 and int(dims[3]) == codec, dst
        assert np.array_equal(decoded(tmp_path / dst), frames)
    (tmp_path / "x.mkv").write_bytes(b"GIF89a" + b"\0" * 64)
    msg = _refused(tmp_path / "x.mkv", "unrecognised container")
    for name in ("AVI", "Matroska", "QuickTime / MP4", "LMV1"):
        assert name in msg
    # an EBML file that is not Matroska
    (tmp_path / "w.webm").write_bytes(mkv(png_frames(cv2, frames), "V_MS/VFW/FOURCC", 24, 16, private=bitmapinfo(24, 16, b"png ", 8)).replace(b"matroska", b"webm\0\0\0\0"))
    _refused(tmp_path / "w.webm", "DocType 'webm'")


def test_index_cost_on_the_cpu(tmp_path):
    """The index walk is host work: a 10 000-frame FFV1 Matroska file against the same frames as AVI (page cache warm)."""
    import time

    from _ffv1_avi import ffv1_avi

    rec, fr = Encoder(False, slices=(1, 1), gop=12).encode(_frames(11, 12, 8, 16))
    frames = [fr[i % 12] for i in range(10000)]
    (tmp_path / "v.mkv").write_bytes(mkv(frames, "V_FFV1", 16, 8, private=rec, cluster_frames=64))
    (tmp_path / "v.avi").write_bytes(ffv1_avi(frames, 16, 8, rec))
    best = {}
    for name in ("v.avi", "v.mkv"):
        read_range(tmp_path / name, 0, 0)
        t = []
        for _ in range(5):
            t0 = time.perf_counter()
            assert int(read_range(tmp_path / name, 0, 0)[0][0]) == 10000
            t.append(time.perf_counter() - t0)
        best[name] = min(t)
    print(f"index walk, 10 000 FFV1 frames: AVI {best['v.avi'] * 1e3:.1f} ms, Matroska {best['v.mkv'] * 1e3:.1f} ms")
    assert best["v.mkv"] < 1.0


def test_batch_list_refuses_one_stem_in_two_containers(tmp_path):
    """t01.avi and t01.mkv would both write output_t01.yml: the batch driver's pre-flight refuses the list."""
    import os
    import subprocess

    from test_batch_list import HOST, ROOT, _run, _touch

    if not os.path.exists(os.path.join(ROOT, "locomouse_cpp_b200", "liblocomouse_b200.so")):
        pytest.skip("CUDA library not built")
    p = subprocess.run(["make", "-C", HOST, "locomouse_b200_batch"], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    b = _touch(tmp_path / "bkg.lmi")
    v1, v2, v3 = _touch(tmp_path / "t01.avi"), _touch(tmp_path / "t02.mov"), _touch(tmp_path / "t01.mkv")
    p = _run(os.path.join(HOST, "locomouse_b200_batch"), tmp_path, [f"{v1}\t{b}", f"{v2}\t{b}", f"{v3}\t{b}"])
    assert p.returncode == 1
    assert "list line 3: output stem 't01' is also the stem of line 1" in p.stdout
    assert "list line 2" not in p.stdout
