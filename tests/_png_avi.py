"""PNG-coded AVI test data: videos written by cv2.VideoWriter ('MPNG' / 'png '), hand-built AVIs around cv2.imencode PNGs
(widths the writer cannot produce), PNG files built from numpy filtering and Python's zlib, and the host reader
lmh_read_avi_png (host/lm_media.hpp)."""
import ctypes as C
import struct
import zlib

import numpy as np

from test_match2nd import _host


def read_avi_png(path):
    """(payload uint8[bytes], offsets int64[n + 1], (n, rows, cols)) of a PNG-coded AVI; RuntimeError with the reader's message."""
    H = _host()
    fn = H.lmh_read_avi_png
    fn.restype = C.c_int
    dims = np.zeros(4, np.int64)
    msg = C.create_string_buffer(512)
    if fn(str(path).encode(), C.c_void_p(dims.ctypes.data), None, None, msg, 512) != 0:
        raise RuntimeError(msg.value.decode())
    payload = np.zeros(int(dims[3]), np.uint8)
    offs = np.zeros(int(dims[0]) + 1, np.int64)
    assert fn(str(path).encode(), C.c_void_p(dims.ctypes.data), C.c_void_p(payload.ctypes.data), C.c_void_p(offs.ctypes.data), msg, 512) == 0
    return payload, offs, tuple(int(v) for v in dims[:3])


def write_cv2_avi(cv2, path, frames, fourcc="MPNG"):
    """frames: [n, h, w] grey or [n, h, w, 3] BGR; returns what cv2.VideoCapture + extractChannel(0) reads back."""
    n, h, w = frames.shape[:3]
    colour = frames.ndim == 4
    wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*fourcc), 30.0, (w, h), colour)
    assert wr.isOpened()
    for f in frames:
        wr.write(f)
    wr.release()
    return capture(cv2, path)


def capture(cv2, path):
    cap = cv2.VideoCapture(str(path))
    out = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        out.append(cv2.extractChannel(f, 0) if f.ndim == 3 else f)
    cap.release()
    return np.stack(out) if out else np.zeros((0,), np.uint8)


def _riff(tag, payload):
    return tag + struct.pack("<I", len(payload)) + payload + (b"\0" if len(payload) & 1 else b"")


def png_avi(pngs, w, h, fourcc=b"MPNG", empty_at=()):
    """An AVI whose stream 0 holds the given PNG files as '00dc' chunks (zero-size chunks inserted before indices in empty_at)."""
    bih = struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, struct.unpack("<I", fourcc)[0], w * h * 3, 0, 0, 0, 0)
    strh = b"vids" + fourcc + b"\0" * 48
    hdrl = b"hdrl" + _riff(b"avih", b"\0" * 56) + _riff(b"LIST", b"strl" + _riff(b"strh", strh) + _riff(b"strf", bih))
    movi = b"movi"
    for i, p in enumerate(pngs):
        if i in empty_at:
            movi += _riff(b"00dc", b"")
        movi += _riff(b"00dc", p)
    body = b"AVI " + _riff(b"LIST", hdrl) + _riff(b"JUNK", b"\0" * 11) + _riff(b"LIST", movi)
    return b"RIFF" + struct.pack("<I", len(body)) + body


def _chunk(tag, data):
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)


def png_from_zlib(zdata, w, h, ctype=0, depth=8, interlace=0, idat_split=None):
    """A PNG file around an already compressed zlib stream; IDAT split into pieces of idat_split bytes."""
    ihdr = struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, interlace)
    step = idat_split or max(len(zdata), 1)
    idats = b"".join(_chunk(b"IDAT", zdata[i:i + step]) for i in range(0, max(len(zdata), 1), step))
    return b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", ihdr) + idats + _chunk(b"IEND", b"")


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(img, filters):
    """The PNG filtered byte stream of img ([h, w] grey or [h, w, c]) with row r filtered by filters[r] (0..4)."""
    h = img.shape[0]
    rows = img.reshape(h, -1).astype(np.int32)
    bpp = 1 if img.ndim == 2 else img.shape[2]
    out = bytearray()
    prev = np.zeros_like(rows[0])
    for r in range(h):
        x = rows[r]
        a = np.concatenate([np.zeros(bpp, np.int32), x[:-bpp]])
        c = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]])
        pred = [np.zeros_like(x), a, prev, (a + prev) >> 1, _paeth(a, prev, c)][filters[r]]
        out.append(filters[r])
        out += ((x - pred) & 255).astype(np.uint8).tobytes()
        prev = x
    return bytes(out)


def make_png(img, filters=None, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, idat_split=None, raw=None):
    """PNG of img (grey [h, w], RGB [h, w, 3] or RGBA [h, w, 4], RGB byte order) built with numpy filtering and zlib."""
    h, w = img.shape[:2]
    ctype = 0 if img.ndim == 2 else {3: 2, 4: 6}[img.shape[2]]
    if filters is None:
        filters = [4] * h
    data = filter_rows(img, filters) if raw is None else raw
    co = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
    return png_from_zlib(co.compress(data) + co.flush(), w, h, ctype, idat_split=idat_split)


class BitWriter:
    """Deflate bit packing: fields LSB first, Huffman codes MSB first."""

    def __init__(self):
        self.bits = []

    def put(self, v, n):
        self.bits += [(v >> i) & 1 for i in range(n)]

    def code(self, c, n):
        self.bits += [(c >> (n - 1 - i)) & 1 for i in range(n)]

    def align(self):
        self.bits += [0] * (-len(self.bits) % 8)

    def raw(self, data):
        self.align()
        for b in data:
            self.put(b, 8)

    def bytes(self):
        self.align()
        a = np.array(self.bits, np.uint8).reshape(-1, 8)
        return bytes((a << np.arange(8, dtype=np.uint8)).sum(1).astype(np.uint8))

    def fixed_literal(self, v):
        if v < 144:
            self.code(0x30 + v, 8)
        elif v < 256:
            self.code(0x190 + v - 144, 9)
        elif v < 280:
            self.code(v - 256, 7)
        else:
            self.code(0xC0 + v - 280, 8)
