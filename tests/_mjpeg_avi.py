"""Motion-JPEG test data: a small baseline JPEG encoder in numpy (1 or 3 components, 4:2:0 / 4:2:2 / 4:4:4, restart
intervals, custom quantisation and Huffman tables, omitted DHT, fill bytes before markers), an AVI writer around its frames,
cv2.VideoWriter files, and the host entry points lmh_read_video_mjpeg / lmh_decode_mjpeg (host/lm_media.hpp with
decode_mjpeg on, csrc/mjpeg_format.h run on the CPU).

Every stream the encoder builds is decoded with cv2.VideoCapture by the tests that use it (mjpeg_file); a stream cv2
rejects fails the test, so the streams stay inside what libavcodec's decoder reads."""
import ctypes as C
import struct

import numpy as np

from _png_avi import _riff, capture
from test_match2nd import _host

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                   35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
                   62, 63])

# JPEG Annex K: the example quantisation tables (natural order) and Huffman tables (bits[1..16], values)
Q_LUMA = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80,
                   62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98,
                   112, 100, 103, 99])
Q_CHROMA = np.array([17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99,
                     99, 99] + [99] * 32)
DC_LUMA = ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12)))
DC_CHROMA = ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12)))
AC_LUMA = ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d], bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a434445464748494a"
    "535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7"
    "c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa"))
AC_CHROMA = ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77], bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738393a434445464748"
    "494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4"
    "c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa"))


def scaled_q(q, quality):
    """libjpeg's quality scaling of an example table."""
    s = 5000 // quality if quality < 50 else 200 - 2 * quality
    return np.clip((q * s + 50) // 100, 1, 255)


def _codes(bits, vals):
    code, k, out = 0, 0, {}
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            out[vals[k]] = (code, length)
            k += 1
            code += 1
        code <<= 1
    return out


class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, v, n):
        self.acc = (self.acc << n) | (v & ((1 << n) - 1))
        self.n += n
        while self.n >= 8:
            b = (self.acc >> (self.n - 8)) & 255
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)
            self.n -= 8

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)
        self.acc = 0


def _category(v):
    return int(abs(int(v))).bit_length()


def _put_value(bw, v, s):
    if s:
        bw.put(v if v > 0 else v + (1 << s) - 1, s)


def fdct_quant(plane, q):
    """[by, bx, 64] quantised coefficients (natural order) of a plane whose size is a multiple of 8."""
    h, w = plane.shape
    x = np.arange(8)
    c = np.where(x == 0, np.sqrt(1 / 8), np.sqrt(2 / 8))[:, None] * np.cos((2 * x[None, :] + 1) * x[:, None] * np.pi / 16)
    b = plane.astype(np.float64).reshape(h // 8, 8, w // 8, 8).transpose(0, 2, 1, 3) - 128
    d = np.einsum("ui,abij,vj->abuv", c, b, c)
    return np.round(d.reshape(h // 8, w // 8, 64) / q).astype(np.int64)


def _pad(plane, h, w):
    return np.pad(plane, ((0, h - plane.shape[0]), (0, w - plane.shape[1])), mode="edge")


class Jpeg:
    """One baseline JPEG frame.  comps: 1 (grey) or 3 (YCbCr); hv: Y's sampling (h, v), chroma 1 x 1."""

    def __init__(self, comps=1, hv=(2, 2), quality=75, dri=0, custom_huffman=False, omit_dht=False, fill=False, q=None, ids=(1, 2, 3),
                 extra_segments=b"", omit_dqt=False):
        self.comps, self.hv, self.dri, self.omit_dht, self.fill, self.ids, self.extra = comps, hv if comps == 3 else (1, 1), dri, omit_dht, fill, ids, extra_segments
        self.omit_dqt = omit_dqt
        self.q = q if q is not None else [scaled_q(Q_LUMA, quality), scaled_q(Q_CHROMA, quality)]
        tabs = [DC_LUMA, AC_LUMA, DC_CHROMA, AC_CHROMA]
        if custom_huffman:  # the same lengths with the values reversed: frequent symbols get the longest codes
            tabs = [(b, list(v)[::-1]) for b, v in tabs]
        self.tabs = [(list(b), list(v)) for b, v in tabs]

    def _marker(self, m, payload):
        return (b"\xff\xff\xff" if self.fill else b"\xff") + bytes([m]) + struct.pack(">H", len(payload) + 2) + payload

    def coefficients(self, y, cb=None, cr=None):
        """Quantised blocks of each component from planes: y [h, w]; cb / cr at chroma resolution."""
        h, w = y.shape
        hs, vs = self.hv
        mh, mw = -(-h // (8 * vs)), -(-w // (8 * hs))
        out = [fdct_quant(_pad(y, mh * 8 * vs, mw * 8 * hs), self.q[0].reshape(64))]
        if self.comps == 3:
            out += [fdct_quant(_pad(p, mh * 8, mw * 8), self.q[1].reshape(64)) for p in (cb, cr)]
        return out

    def encode(self, y, cb=None, cr=None):
        return self.encode_blocks(y.shape, self.coefficients(y, cb, cr))

    def encode_blocks(self, shape, blocks):
        """The file for quantised blocks [by, bx, 64] (natural order) of each component."""
        h, w = shape
        hs, vs = self.hv
        mh, mw = -(-h // (8 * vs)), -(-w // (8 * hs))
        out = bytearray(b"\xff\xd8")
        out += self._marker(0xE0, b"JFIF\0\x01\x01\0\0\x01\0\x01\0\0")
        out += self._marker(0xFE, b"test encoder")
        nq = 1 if self.comps == 1 else 2
        if not self.omit_dqt:
            out += self._marker(0xDB, b"".join(bytes([t]) + bytes(int(v) for v in self.q[t].reshape(64)[ZIGZAG]) for t in range(nq)))
        comp = [(self.ids[0], hs, vs, 0)] + ([(self.ids[1], 1, 1, 1), (self.ids[2], 1, 1, 1)] if self.comps == 3 else [])
        out += self._marker(0xC0, struct.pack(">BHHB", 8, h, w, self.comps) + b"".join(bytes([c, (a << 4) | b, t]) for c, a, b, t in comp))
        if not self.omit_dht:
            seg = b""
            for cls_id, (b, v) in zip([0x00, 0x10, 0x01, 0x11][:2 * nq], self.tabs):
                seg += bytes([cls_id]) + bytes(b) + bytes(v)
            out += self._marker(0xC4, seg)
        if self.dri:
            out += self._marker(0xDD, struct.pack(">H", self.dri))
        out += self.extra
        out += self._marker(0xDA, bytes([self.comps]) + b"".join(bytes([c[0], 0x00 if i == 0 else 0x11]) for i, c in enumerate(comp)) + b"\x00\x3f\x00")
        codes = [_codes(*t) for t in self.tabs]
        bw = _Bits()
        pred = [0] * self.comps
        for m in range(mh * mw):
            if self.dri and m and m % self.dri == 0:
                bw.flush()
                out += bw.out
                bw.out = bytearray()
                out += bytes([0xFF, 0xD0 + (m // self.dri - 1) % 8])
                pred = [0] * self.comps
            my, mx = divmod(m, mw)
            for ci in range(self.comps):
                dc_t, ac_t = codes[2 * min(ci, 1)], codes[2 * min(ci, 1) + 1]
                sh, sv = (hs, vs) if ci == 0 else (1, 1)
                for v in range(sv):
                    for u in range(sh):
                        blk = blocks[ci][my * sv + v, mx * sh + u][ZIGZAG]
                        d = int(blk[0]) - pred[ci]
                        pred[ci] = int(blk[0])
                        s = _category(d)
                        bw.put(*dc_t[s])
                        _put_value(bw, d, s)
                        run = 0
                        for k in range(1, 64):
                            a = int(blk[k])
                            if a == 0:
                                run += 1
                                continue
                            while run > 15:
                                bw.put(*ac_t[0xF0])
                                run -= 16
                            s = _category(a)
                            bw.put(*ac_t[(run << 4) | s])
                            _put_value(bw, a, s)
                            run = 0
                        if run:
                            bw.put(*ac_t[0x00])
        bw.flush()
        out += bw.out
        out += b"\xff\xd9"
        return bytes(out)


def mjpeg_avi(jpegs, w, h, fourcc=b"MJPG"):
    """An AVI whose stream 0 holds the given JPEG files as '00dc' chunks."""
    bih = struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, struct.unpack("<I", fourcc)[0], w * h * 3, 0, 0, 0, 0)
    strh = b"vids" + fourcc + b"\0" * 48
    hdrl = b"hdrl" + _riff(b"avih", b"\0" * 56) + _riff(b"LIST", b"strl" + _riff(b"strh", strh) + _riff(b"strf", bih))
    movi = b"movi" + b"".join(_riff(b"00dc", j) for j in jpegs)
    body = b"AVI " + _riff(b"LIST", hdrl) + _riff(b"LIST", movi)
    return b"RIFF" + struct.pack("<I", len(body)) + body


def mjpeg_file(cv2, path, jpegs, w, h, fourcc=b"MJPG"):
    """Writes the AVI and returns what cv2.VideoCapture + extractChannel(0) reads from it; fails when cv2 does not read
    every frame."""
    path.write_bytes(mjpeg_avi(jpegs, w, h, fourcc))
    want = capture(cv2, path)
    assert want.shape == (len(jpegs), h, w), f"cv2.VideoCapture read {want.shape} from {path.name}"
    return want


def write_cv2_mjpeg(cv2, path, frames, api=None, quality=None):
    """frames [n, h, w] grey or [n, h, w, 3] BGR through cv2.VideoWriter 'MJPG' (FFmpeg's encoder, or OpenCV's own with
    api = cv2.CAP_OPENCV_MJPEG); returns VideoCapture's channel 0."""
    n, h, w = frames.shape[:3]
    colour = frames.ndim == 4
    args = [str(path)] + ([api] if api is not None else []) + [cv2.VideoWriter_fourcc(*"MJPG"), 30.0, (w, h)]
    params = [cv2.VIDEOWRITER_PROP_IS_COLOR, int(colour)] + ([cv2.VIDEOWRITER_PROP_QUALITY, quality] if quality is not None else [])
    wr = cv2.VideoWriter(*args, params)
    assert wr.isOpened()
    for f in frames:
        wr.write(f)
    wr.release()
    return capture(cv2, path)


# ---- host reader / CPU decoder ---------------------------------------------------------------------------------------


def read_video_mjpeg(path):
    """(payload, offsets, (n, rows, cols)) of a Motion-JPEG video in any container, read with decode_mjpeg on;
    RuntimeError with the reader's message."""
    fn = _host().lmh_read_video_mjpeg
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p] + [C.c_void_p] * 3 + [C.c_char_p, C.c_int]
    dims = np.zeros(4, np.int64)
    msg = C.create_string_buffer(512)
    if fn(str(path).encode(), dims.ctypes.data, None, None, msg, 512) != 0:
        raise RuntimeError(msg.value.decode())
    payload = np.zeros(int(dims[3]), np.uint8)
    offs = np.zeros(int(dims[0]) + 1, np.int64)
    assert fn(str(path).encode(), dims.ctypes.data, payload.ctypes.data, offs.ctypes.data, msg, 512) == 0
    return payload, offs, tuple(int(v) for v in dims[:3])


def decode_cpu(payload, offsets, rows, cols):
    """mjpeg_format.h on the CPU: uint8 [n, rows, cols]; ValueError with the decoder's message."""
    fn = _host().lmh_decode_mjpeg
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_int]
    pay = np.ascontiguousarray(payload, np.uint8)
    offs = np.ascontiguousarray(offsets, np.int64)
    n = offs.size - 1
    out = np.zeros((n, rows, cols), np.uint8)
    msg = C.create_string_buffer(512)
    if fn(pay.ctypes.data, offs.ctypes.data, n, rows, cols, out.ctypes.data, msg, 512) != 0:
        raise ValueError(msg.value.decode())
    return out


def split(jpegs):
    """payload, offsets of a list of JPEG files"""
    offs = np.cumsum([0] + [len(j) for j in jpegs]).astype(np.int64)
    return np.frombuffer(b"".join(jpegs), np.uint8).copy(), offs
