"""Matroska and QuickTime / MP4 test data (host/lm_containers.hpp): videos written by cv2.VideoWriter, and small hand-written
Matroska and ISO BMFF writers for the structures cv2 does not produce (unknown element sizes, BlockGroup, an audio track before
the video track, Void and CRC-32 elements, co64, several chunks with stsc runs, moov before or after mdat, 64-bit box sizes,
raw RGB samples).  Every hand-written file a test expects to be accepted is first decoded with cv2.VideoCapture and must give
the intended frames (check_capture)."""
import struct
import zlib

import numpy as np

from _png_avi import capture

DD_2997 = 33366700          # DefaultDuration (ns) FFmpeg writes for 30000 / 1001 frames/s


def write_cv2(cv2, path, frames, fourcc, fps=30000 / 1001):
    """frames [n, h, w] grey or [n, h, w, 3] BGR through cv2.VideoWriter; returns what VideoCapture + channel 0 reads back."""
    n, h, w = frames.shape[:3]
    wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*fourcc), fps, (w, h), frames.ndim == 4)
    assert wr.isOpened(), (path, fourcc)
    for f in frames:
        wr.write(f)
    wr.release()
    return capture(cv2, path)


def frame_count(cv2, path):
    cap = cv2.VideoCapture(str(path))
    n = int(cap.get(cv2.CAP_PROP_FRAME_COUNT))
    cap.release()
    return n


def check_capture(cv2, path, want):
    got = capture(cv2, path)
    assert got.shape == want.shape and np.array_equal(got, want), f"cv2.VideoCapture does not read {path} as intended"
    return got


def png_frames(cv2, frames):
    """Each frame as a PNG file (cv2.imencode: grey, or BGR stored as RGB)."""
    return [cv2.imencode(".png", f)[1].tobytes() for f in frames]


# ---- Matroska -------------------------------------------------------------------------------------------------------------

UNKNOWN = b"\x01\xff\xff\xff\xff\xff\xff\xff"


def _id(i):
    return i.to_bytes((i.bit_length() + 7) // 8, "big")


def _size(n):
    for k in range(1, 9):
        if n < (1 << (7 * k)) - 1:
            return ((1 << (7 * k)) | n).to_bytes(k, "big")   # marker bit, then the value
    raise ValueError(n)


def el(i, payload=b"", unknown=False):
    return _id(i) + (UNKNOWN if unknown else _size(len(payload))) + payload


def uint_el(i, v):
    return el(i, v.to_bytes(max(1, (v.bit_length() + 7) // 8), "big"))


def master(i, children, crc=False, unknown=False):
    """A master element; crc puts a CRC-32 element (IEEE, little-endian, over the other children) first."""
    body = b"".join(children)
    if crc:
        body = el(0xBF, struct.pack("<I", zlib.crc32(body) & 0xFFFFFFFF)) + body
    return el(i, body, unknown)


def mkv(payloads, codec_id, w, h, private=None, colour=None, default_duration=DD_2997, duration_ms=None, timecodes_ms=None,
        unknown_sizes=False, block_group=False, audio_first=False, void_crc=False, laced_at=None, content_encoding=False,
        cluster_frames=8, with_duration=True):
    """A Matroska file whose video track holds one frame per payload, in clusters of cluster_frames.  Timecodes are
    i * default_duration by default; the segment Duration is the last timecode plus one frame unless given."""
    n = len(payloads)
    tc = timecodes_ms if timecodes_ms is not None else [round(i * default_duration / 1e6) for i in range(n)]
    if duration_ms is None:
        duration_ms = (tc[-1] if n else 0) + default_duration / 1e6
    vt = 2 if audio_first else 1
    ebml = master(0x1A45DFA3, [uint_el(0x4286, 1), uint_el(0x42F7, 1), uint_el(0x42F2, 4), uint_el(0x42F3, 8), el(0x4282, b"matroska"),
                               uint_el(0x4287, 4), uint_el(0x4285, 2)])
    info = [uint_el(0x2AD7B1, 1000000), el(0x4D80, b"lm-test"), el(0x5741, b"lm-test")]
    if with_duration:
        info.append(el(0x4489, struct.pack(">d", duration_ms)))
    video = [uint_el(0xB0, w), uint_el(0xBA, h)] + ([el(0x2EB524, colour)] if colour is not None else [])
    entry = [uint_el(0xD7, vt), uint_el(0x73C5, 1000 + vt), uint_el(0x9C, 0), el(0x86, codec_id.encode()), uint_el(0x83, 1),
             uint_el(0x23E383, default_duration), master(0xE0, video)]
    if private is not None:
        entry.append(el(0x63A2, bytes(private)))
    if content_encoding:
        entry.append(master(0x6D80, [master(0x6240, [uint_el(0x5031, 0), uint_el(0x5032, 1), uint_el(0x5033, 1),
                                                     master(0x5034, [uint_el(0x4254, 0)])])]))
    if void_crc:
        entry.append(el(0xEC, b"\0" * 5))
    tracks = [master(0xAE, entry, crc=void_crc)]
    if audio_first:
        audio = master(0xE1, [el(0xB5, struct.pack(">d", 8000.0)), uint_el(0x9F, 1), uint_el(0x6264, 16)])
        tracks.insert(0, master(0xAE, [uint_el(0xD7, 1), uint_el(0x73C5, 1001), el(0x86, b"A_PCM/INT/LIT"), uint_el(0x83, 2), audio]))
    segment = [master(0x1549A966, info, crc=void_crc)]
    if void_crc:
        segment.append(el(0xEC, b"\0" * 30))
    segment.append(master(0x1654AE6B, tracks, crc=void_crc))
    for c0 in range(0, n, cluster_frames):
        kids = [uint_el(0xE7, tc[c0])]
        if void_crc:
            kids.append(el(0xEC, b"\0" * 3))
        for i in range(c0, min(n, c0 + cluster_frames)):
            rel = struct.pack(">h", tc[i] - tc[c0])
            flags = 0x02 if laced_at == i else 0
            if audio_first:   # an audio block of track 1 beside every video frame
                kids.append(el(0xA3, b"\x81" + rel + b"\x80" + b"\0" * 64))
            if block_group:
                kids.append(master(0xA0, [el(0xA1, bytes([0x80 | vt]) + rel + bytes([flags]) + payloads[i]),
                                          uint_el(0x9B, max(1, round(default_duration / 1e6)))]))
            else:
                kids.append(el(0xA3, bytes([0x80 | vt]) + rel + bytes([0x80 | flags]) + payloads[i]))
        segment.append(master(0x1F43B675, kids, crc=void_crc, unknown=unknown_sizes))
    return ebml + master(0x18538067, segment, unknown=unknown_sizes)


def bitmapinfo(w, h, fourcc, bits, extra=b""):
    return struct.pack("<IiiHHIIiiII", 40 + len(extra), w, h, 1, bits, struct.unpack("<I", fourcc)[0] if isinstance(fourcc, bytes) else fourcc,
                       w * h * max(bits // 8, 1), 0, 0, 0, 0) + extra


# ---- ISO BMFF (QuickTime / MP4) ---------------------------------------------------------------------------------------------


def box(t, payload, large=False):
    if large:
        return struct.pack(">I", 1) + t + struct.pack(">Q", 16 + len(payload)) + payload
    return struct.pack(">I", 8 + len(payload)) + t + payload


def full(t, payload, version=0, flags=0):
    return box(t, struct.pack(">I", (version << 24) | flags) + payload)


def esds_png():
    """esds of an 'mp4v' entry whose object type is PNG (0x6D), with FFmpeg's 4-byte descriptor lengths."""
    def descr(tag, body):
        return bytes([tag, 0x80, 0x80, 0x80, len(body)]) + body
    dcd = descr(4, bytes([0x6D, 0x11, 0, 0, 0]) + struct.pack(">II", 0, 0))
    return full(b"esds", descr(3, struct.pack(">HB", 1, 0) + dcd + descr(6, b"\x02")))


def sample_entry(fourcc, w, h, depth, children=b""):
    body = (b"\0" * 6 + struct.pack(">H", 1) + struct.pack(">HH", 0, 0) + b"FFMP" + struct.pack(">II", 0, 0x200) + struct.pack(">HH", w, h) +
            struct.pack(">II", 0x480000, 0x480000) + struct.pack(">IH", 0, 1) + b"\0" * 32 + struct.pack(">Hh", depth, -1) + children)
    return box(fourcc, body)


def mov(samples, fourcc, w, h, depth=24, children=b"", chunks=None, co64=False, moov_first=False, edit="identity", ctts=None, mp4=False,
        large_mdat=False, moof=False, delta=1001, timescale=30000, single_size=False):
    """A QuickTime (or MP4) file with one video track.  chunks: samples per chunk (default: all in one); edit: "identity",
    None (no edts) or a list of (segment duration in movie ticks, media time); ctts: composition offsets per sample."""
    n = len(samples)
    chunks = chunks or [n]
    assert sum(chunks) == n
    media_dur = n * delta
    movie_ts = 1000
    seg = -(-media_dur * movie_ts // timescale)

    def moov_box(mdat_data_at):
        offs, at, k = [], mdat_data_at, 0
        for c in chunks:
            offs.append(at)
            at += sum(len(s) for s in samples[k:k + c])
            k += c
        runs, prev = [], None
        for i, c in enumerate(chunks):
            if c != prev:
                runs.append((i + 1, c, 1))
                prev = c
        stbl = [full(b"stsd", struct.pack(">I", 1) + sample_entry(fourcc, w, h, depth, children)),
                full(b"stts", struct.pack(">III", 1, n, delta)),
                full(b"stsc", struct.pack(">I", len(runs)) + b"".join(struct.pack(">III", *r) for r in runs))]
        if single_size:
            assert len({len(s) for s in samples}) == 1
            stbl.append(full(b"stsz", struct.pack(">II", len(samples[0]), n)))
        else:
            stbl.append(full(b"stsz", struct.pack(">II", 0, n) + b"".join(struct.pack(">I", len(s)) for s in samples)))
        if co64:
            stbl.append(full(b"co64", struct.pack(">I", len(offs)) + b"".join(struct.pack(">Q", o) for o in offs)))
        else:
            stbl.append(full(b"stco", struct.pack(">I", len(offs)) + b"".join(struct.pack(">I", o) for o in offs)))
        if ctts is not None:
            stbl.append(full(b"ctts", struct.pack(">I", n) + b"".join(struct.pack(">II", 1, c) for c in ctts)))
        url = full(b"url ", b"", flags=1)
        minf = [full(b"vmhd", struct.pack(">HHHH", 0, 0, 0, 0), flags=1)]
        if not mp4:
            minf.append(full(b"hdlr", b"dhlr" + b"url " + b"\0" * 12 + b"\x0bDataHandler"))
        minf += [box(b"dinf", full(b"dref", struct.pack(">I", 1) + url)), box(b"stbl", b"".join(stbl))]
        mdia = box(b"mdia", full(b"mdhd", struct.pack(">IIIIHH", 0, 0, timescale, media_dur, 0x55C4 if mp4 else 0x7FFF, 0)) +
                   full(b"hdlr", (b"\0\0\0\0" if mp4 else b"mhlr") + b"vide" + b"\0" * 12 + (b"VideoHandler\0" if mp4 else b"\x0cVideoHandler")) +
                   box(b"minf", b"".join(minf)))
        matrix = struct.pack(">9I", 0x10000, 0, 0, 0, 0x10000, 0, 0, 0, 0x40000000)
        tkhd = full(b"tkhd", struct.pack(">IIIII", 0, 0, 1, 0, seg) + b"\0" * 8 + struct.pack(">HHHH", 0, 0, 0, 0) + matrix +
                    struct.pack(">II", w << 16, h << 16), flags=3)
        edts = b""
        if edit is not None:
            edits = [(seg, 0)] if edit == "identity" else edit
            edts = box(b"edts", full(b"elst", struct.pack(">I", len(edits)) + b"".join(struct.pack(">IiI", d, t, 0x10000) for d, t in edits)))
        trak = box(b"trak", tkhd + edts + mdia)
        mvhd = full(b"mvhd", struct.pack(">IIIII", 0, 0, movie_ts, seg, 0x10000) + struct.pack(">H", 0x100) + b"\0" * 10 + matrix +
                    b"\0" * 24 + struct.pack(">I", 2))
        return box(b"moov", mvhd + trak + (box(b"mvex", full(b"trex", b"\0" * 20)) if moof else b""))

    ftyp = box(b"ftyp", b"isom" + struct.pack(">I", 0x200) + b"isomiso2mp41") if mp4 else box(b"ftyp", b"qt  " + struct.pack(">I", 0x200) + b"qt  ")
    pre = ftyp + (box(b"free", b"") if mp4 else box(b"wide", b""))
    data = b"".join(samples)
    hl = 16 if large_mdat else 8
    tail = box(b"moof", full(b"mfhd", struct.pack(">I", 1))) if moof else b""
    if moov_first:
        m = moov_box(0)
        m = moov_box(len(pre) + len(m) + hl)
        return pre + m + box(b"mdat", data, large_mdat) + tail
    return pre + box(b"mdat", data, large_mdat) + moov_box(len(pre) + hl) + tail
