"""FFV1-coded AVI test data: an AVI writer around FFV1 frames, a small FFV1 version 3 encoder (range and Golomb-Rice coders,
small and large context models, any slice grid and GOP, coded initial states, a custom state-transition table), and the
host entry points lmh_read_avi_ffv1 / lmh_decode_ffv1 (host/lm_media.hpp, csrc/ffv1_format.h run on the CPU).

The encoder follows libavcodec's ffv1enc.c.  Every stream it builds is decoded back with cv2.VideoCapture and must give
the encoder's input exactly (encode_avi checks it), which pins the encoder to libavcodec's decoder."""
import ctypes as C
import struct

import numpy as np

from _png_avi import _riff, capture
from test_match2nd import _host

# ---- host reader / CPU decoder ---------------------------------------------------------------------------------------


def read_avi_ffv1(path):
    """(extradata, payload, offsets, (n, rows, cols)) of an FFV1-coded AVI; RuntimeError with the reader's message."""
    fn = _host().lmh_read_avi_ffv1
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p] + [C.c_void_p] * 5 + [C.c_int]
    dims = np.zeros(5, np.int64)
    msg = C.create_string_buffer(512)
    if fn(str(path).encode(), dims.ctypes.data, None, None, None, msg, 512) != 0:
        raise RuntimeError(msg.value.decode())
    payload = np.zeros(int(dims[3]), np.uint8)
    offs = np.zeros(int(dims[0]) + 1, np.int64)
    ex = np.zeros(max(int(dims[4]), 1), np.uint8)
    assert fn(str(path).encode(), dims.ctypes.data, payload.ctypes.data, offs.ctypes.data, ex.ctypes.data, msg, 512) == 0
    return ex[:int(dims[4])], payload, offs, tuple(int(v) for v in dims[:3])


def decode_cpu(extradata, payload, offsets, rows, cols):
    """ffv1_format.h on the CPU: uint8 [n, rows, cols]; ValueError with the decoder's message."""
    fn = _host().lmh_decode_ffv1
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_int]
    ex = np.ascontiguousarray(extradata, np.uint8)
    pay = np.ascontiguousarray(payload, np.uint8)
    offs = np.ascontiguousarray(offsets, np.int64)
    n = offs.size - 1
    out = np.zeros((n, rows, cols), np.uint8)
    msg = C.create_string_buffer(512)
    if fn(ex.ctypes.data, ex.size, pay.ctypes.data, offs.ctypes.data, n, rows, cols, out.ctypes.data, msg, 512) != 0:
        raise ValueError(msg.value.decode())
    return out


# ---- AVI -----------------------------------------------------------------------------------------------------------


def ffv1_avi(frames, w, h, extradata, empty_at=()):
    """An AVI whose stream 0 is 'FFV1' with the given record in 'strf' and the given frames as '00dc' chunks."""
    bih = struct.pack("<IiiHHIIiiII", 40 + len(extradata), w, h, 1, 24, struct.unpack("<I", b"FFV1")[0], w * h * 3, 0, 0, 0, 0)
    strh = b"vids" + b"FFV1" + b"\0" * 48
    hdrl = b"hdrl" + _riff(b"avih", b"\0" * 56) + _riff(b"LIST", b"strl" + _riff(b"strh", strh) + _riff(b"strf", bih + bytes(extradata)))
    movi = b"movi"
    for i, f in enumerate(frames):
        if i in empty_at:
            movi += _riff(b"00dc", b"")
        movi += _riff(b"00dc", bytes(f))
    body = b"AVI " + _riff(b"LIST", hdrl) + _riff(b"LIST", movi)
    return b"RIFF" + struct.pack("<I", len(body)) + body


def strf_record(avi_bytes):
    """The FFV1 record (strf bytes after the BITMAPINFOHEADER) of an AVI file's bytes, and its offset in the file."""
    i = avi_bytes.find(b"strf")
    n = struct.unpack("<I", avi_bytes[i + 4:i + 8])[0]
    return avi_bytes[i + 48:i + 8 + n], i + 48


# ---- coders --------------------------------------------------------------------------------------------------------


def build_rac_states(factor=int(0.05 * (1 << 32)), max_p=256 - 8):
    """ff_build_rac_states: (one_state, zero_state)."""
    one = 1 << 32
    ones, zero = [0] * 256, [0] * 256
    last, p = 0, one // 2
    for _ in range(128):
        p8 = (256 * p + one // 2) >> 32
        if p8 <= last:
            p8 = last + 1
        if last and last < 256 and p8 <= max_p:
            ones[last] = p8
        p += ((one - p) * factor + one // 2) >> 32
        last = p8
    for i in range(256 - max_p, max_p + 1):
        if ones[i]:
            continue
        q = (i * one + 128) >> 8
        q += ((one - q) * factor + one // 2) >> 32
        p8 = (256 * q + one // 2) >> 32
        ones[i] = min(max(p8, i + 1), max_p)
    for i in range(1, 255):
        zero[i] = 256 - ones[256 - i]
    return ones, zero


DEFAULT_ONE, DEFAULT_ZERO = build_rac_states()


def tables_from_one(one):
    zero = [0] * 256
    zero[0] = DEFAULT_ZERO[0]
    for i in range(1, 256):
        zero[256 - i] = 256 - one[i]
    return one, zero


class RangeEnc:
    def __init__(self, one=DEFAULT_ONE, zero=DEFAULT_ZERO):
        self.low, self.range, self.outstanding_count, self.outstanding_byte = 0, 0xFF00, 0, -1
        self.out = bytearray()
        self.one, self.zero = one, zero

    def _renorm(self):
        while self.range < 0x100:
            if self.outstanding_byte < 0:
                self.outstanding_byte = self.low >> 8
            elif self.low <= 0xFF00:
                self.out.append(self.outstanding_byte)
                self.out += b"\xff" * self.outstanding_count
                self.outstanding_count = 0
                self.outstanding_byte = self.low >> 8
            elif self.low >= 0x10000:
                self.out.append(self.outstanding_byte + 1)
                self.out += b"\x00" * self.outstanding_count
                self.outstanding_count = 0
                self.outstanding_byte = (self.low >> 8) - 0x100
            else:
                self.outstanding_count += 1
            self.low = (self.low & 0xFF) << 8
            self.range <<= 8

    def put(self, st, k, bit):
        r1 = (self.range * st[k]) >> 8
        if not bit:
            self.range -= r1
            st[k] = self.zero[st[k]]
        else:
            self.low += self.range - r1
            self.range = r1
            st[k] = self.one[st[k]]
        self._renorm()

    def symbol(self, st, v, signed=False):
        if not v:
            self.put(st, 0, 1)
            return
        a = abs(v) if signed else v
        e = a.bit_length() - 1
        self.put(st, 0, 0)
        for i in range(e):
            self.put(st, 1 + min(i, 9), 1)
        self.put(st, 1 + min(e, 9), 0)
        for i in range(e - 1, -1, -1):
            self.put(st, 22 + min(i, 9), (a >> i) & 1)
        if signed:
            self.put(st, 11 + min(e, 10), int(v < 0))

    def terminate(self, version):
        """ff_rac_terminate: the bytes written."""
        if version == 1:
            self.put([129], 0, 0)
        self.range = 0xFF
        self.low += 0xFF
        self._renorm()
        self.range = 0xFF
        self._renorm()
        return bytes(self.out)


class BitWriter:
    def __init__(self):
        self.bits = []

    def put(self, n, v):
        self.bits += [(v >> (n - 1 - i)) & 1 for i in range(n)]

    def flush(self):
        b = self.bits + [0] * (-len(self.bits) % 8)
        return bytes(int("".join(map(str, b[i:i + 8])), 2) for i in range(0, len(b), 8))


_CRC = []
for _i in range(256):
    _c = _i << 24
    for _ in range(8):
        _c = ((_c << 1) ^ (0x04C11DB7 if _c & 0x80000000 else 0)) & 0xFFFFFFFF
    _CRC.append(_c)


def crc32_msb(data, crc=0):
    for b in data:
        crc = ((crc << 8) & 0xFFFFFFFF) ^ _CRC[(crc >> 24) ^ b]
    return crc


def with_crc(data):
    return bytes(data) + crc32_msb(data).to_bytes(4, "big")


# ---- encoder -------------------------------------------------------------------------------------------------------

# Quant tables as run lengths over 0..127 (value k on the k-th run, mirrored to negative differences).  SMALL is 11 x 11
# x 11 levels on L - LT, LT - T, T - RT (666 contexts); LARGE adds LL - L and TT - T (11 x 11 x 5 x 5 x 5: 7563 contexts).
_R11, _R5, _R1 = [1, 1, 3, 7, 16, 100], [1, 2, 125], [128]
SMALL = [_R11, _R11, _R11, _R1, _R1]
LARGE = [_R11, _R11, _R5, _R5, _R5]


def _quant(runs):
    tabs, scale = [], 1
    for r in runs:
        t = [0] * 256
        i = 0
        for v, n in enumerate(r):
            for _ in range(n):
                t[i] = scale * v
                i += 1
        for i in range(1, 128):
            t[256 - i] = -t[i]
        t[128] = -t[127]
        tabs.append(t)
        scale *= 2 * len(r) - 1
    return tabs, (scale + 1) // 2


def _log2_run(i):
    return i >> 2 if i < 16 else 4 + ((i - 16) >> 1) if i < 24 else i - 16


def _fold(v, bits):
    m = 1 << bits
    v &= m - 1
    return v - m if v >= m >> 1 else v


class _Vlc:
    __slots__ = ("drift", "error_sum", "bias", "count")

    def __init__(self):
        self.drift, self.error_sum, self.bias, self.count = 0, 4, 0, 1

    def update(self, v):
        drift, count = self.drift + v, self.count
        self.error_sum = (self.error_sum + abs(v)) & 0xFFFF
        if count == 128:
            count >>= 1
            drift >>= 1
            self.error_sum >>= 1
        count += 1
        if drift <= -count:
            self.bias = max(self.bias - 1, -128)
            drift = max(drift + count, -count + 1)
        elif drift > 0:
            self.bias = min(self.bias + 1, 127)
            drift = min(drift - count, 0)
        self.drift, self.count = drift, count


def _put_vlc(bw, s, v, bits):
    v = _fold(v - s.bias, bits)
    k, i = 0, s.count
    while i < s.error_sum:
        k += 1
        i += i
    code = ~v if 2 * s.drift + s.count < 0 else v
    u = 2 * code if code >= 0 else -2 * code - 1
    e = u >> k
    if e < 12:
        bw.put(e + k + 1, (1 << k) + (u & ((1 << k) - 1)))
    else:
        bw.put(12 + bits, u - 12 + 1)
    s.update(v)


class Encoder:
    """FFV1 version 3 (micro_version 4) with ec = 1.  coder: 0 Golomb-Rice, 1 range (default table), 2 range (custom table).
    model: SMALL or LARGE run lists for every plane; slices: (h, v); gop: keyframe interval (1 = intra-only)."""

    def __init__(self, colour, coder=0, model=SMALL, slices=(4, 2), gop=12, initial_states=False, custom_one=None):
        self.colour, self.coder, self.slices, self.gop = colour, coder, slices, gop
        self.quant, self.ctx_count = _quant(model)
        self.five = bool(self.quant[3][127] or self.quant[4][127])
        self.planes_ctx = 3 if colour else 1  # context planes in use (colour: with alpha)
        self.one, self.zero = DEFAULT_ONE, DEFAULT_ZERO
        if coder == 2:
            self.one, self.zero = tables_from_one(custom_one or build_rac_states(int(0.07 * (1 << 32)), 250)[0])
        rng = np.random.Generator(np.random.PCG64(7))
        self.initial = rng.integers(40, 220, (self.ctx_count, 32)).tolist() if initial_states else None
        self.state = {}
        self.head_bytes = {}  # Golomb-Rice streams: bytes of each slice's range-coded header in the last frame

    def record(self, colorspace=None, bits=8, chroma_planes=None, version=3):
        rc, st = RangeEnc(), [128] * 32
        rc.symbol(st, version)
        rc.symbol(st, 4)
        rc.symbol(st, self.coder)
        if self.coder == 2:
            for i in range(1, 256):
                rc.symbol(st, self.one[i] - DEFAULT_ONE[i], True)
        rc.symbol(st, int(self.colour) if colorspace is None else colorspace)
        rc.symbol(st, bits)
        rc.put(st, 0, int(self.colour) if chroma_planes is None else chroma_planes)
        rc.symbol(st, 0)
        rc.symbol(st, 0)
        rc.put(st, 0, int(self.colour))  # transparency: colour streams carry alpha, as OpenCV's BGRA input does
        rc.symbol(st, self.slices[0] - 1)
        rc.symbol(st, self.slices[1] - 1)
        rc.symbol(st, 1)
        for t in self.quant:
            qs, last = [128] * 32, 0
            for i in range(1, 128):
                if t[i] != t[i - 1]:
                    rc.symbol(qs, i - last - 1)
                    last = i
            rc.symbol(qs, 128 - last - 1)
        rc.put(st, 0, int(self.initial is not None))
        if self.initial is not None:
            st2 = [[128] * 32 for _ in range(32)]
            for j in range(self.ctx_count):
                for k in range(32):
                    pred = self.initial[j - 1][k] if j else 128
                    rc.symbol(st2[k], _fold(self.initial[j][k] - pred, 8), True)
        rc.symbol(st, 1)  # ec
        rc.symbol(st, int(self.gop == 1))  # intra
        return with_crc(rc.terminate(0))

    def _planes(self, img):
        """Sample planes: grey [Y], or colour [G, B, R, A] after the reversible colour transform."""
        if not self.colour:
            return [img.astype(np.int64)]
        b, g, r = (img[..., i].astype(np.int64) for i in range(3))
        b, r = b - g, r - g
        g = g + ((b + r) >> 2)
        return [g, b + 256, r + 256, np.full_like(g, 255)]

    def frame(self, img, key):
        nh, nv = self.slices
        h, w = img.shape[:2]
        planes = self._planes(img)
        out = bytearray()
        for s in range(nh * nv):
            sx, sy = s % nh, s // nh
            x0, x1, y0, y1 = w * sx // nh, w * (sx + 1) // nh, h * sy // nv, h * (sy + 1) // nv
            rc = RangeEnc()
            if s == 0:
                rc.put([128], 0, int(key))
            rc.one, rc.zero = self.one, self.zero
            hs = [128] * 32
            for v in (sx, sy, 0, 0):
                rc.symbol(hs, v)
            for _ in range(2 + int(self.colour)):
                rc.symbol(hs, 0)
            for v in (3, 0, 0):
                rc.symbol(hs, v)
            if key:
                self.state[s] = [[list(r) for r in self.initial] if self.coder and self.initial else
                                 [[128] * 32 for _ in range(self.ctx_count)] if self.coder else
                                 [_Vlc() for _ in range(self.ctx_count)] for _ in range(self.planes_ctx)]
            states = self.state[s]
            bw = BitWriter()
            if not self.coder:
                head = rc.terminate(1)
                self.head_bytes[s] = len(head)
            run_index = 0
            sl = [p[y0:y1, x0:x1] for p in planes]
            for y in range(y1 - y0):
                for p, P in enumerate(sl):  # colour: one line of each plane in turn
                    cp = (p + 1) // 2
                    run_index = _encode_row(self, rc, bw, P, y, states[cp], 9 if self.colour else 8, run_index)
            data = (head + bw.flush()) if not self.coder else rc.terminate(1)
            data = data + len(data).to_bytes(3, "big") + b"\0"
            out += with_crc(data)
        return bytes(out)

    def encode(self, frames):
        """frames: [n, h, w] grey or [n, h, w, 3] BGR uint8 -> (record, [frame bytes])."""
        self.state = {}
        return self.record(), [self.frame(f, i % self.gop == 0) for i, f in enumerate(frames)]


def _encode_row(enc, rc, bw, P, y, states, bits, run_index):
    """One line of one plane (the body of _encode_plane for row y), returning run_index."""
    h, w = P.shape
    q = enc.quant
    mask = (1 << bits) - 1

    def at(yy, x):
        return int(P[yy, x]) if yy >= 0 else 0
    run_mode = run_count = 0
    for x in range(w):
        T = at(y - 1, x)
        L = at(y, x - 1) if x else at(y - 1, 0)
        LT = at(y - 1, x - 1) if x else at(y - 2, 0)
        RT = at(y - 1, min(x + 1, w - 1))
        ctx = q[0][(L - LT) & 255] + q[1][(LT - T) & 255] + q[2][(T - RT) & 255]
        if enc.five:
            LL = at(y, x - 2) if x >= 2 else (at(y - 1, 0) if x == 1 else 0)
            ctx += q[3][(LL - L) & 255] + q[4][(at(y - 2, x) - T) & 255]
        pred = sorted((L, L + T - LT, T))[1]
        diff = int(P[y, x]) - pred
        if ctx < 0:
            ctx, diff = -ctx, -diff
        diff = _fold(diff & mask, bits)
        if enc.coder:
            rc.symbol(states[ctx], diff, True)
            continue
        if ctx == 0:
            run_mode = 1
        if run_mode:
            if diff:
                while run_count >= 1 << _log2_run(run_index):
                    run_count -= 1 << _log2_run(run_index)
                    run_index += 1
                    bw.put(1, 1)
                bw.put(1 + _log2_run(run_index), run_count)
                if run_index:
                    run_index -= 1
                run_count = run_mode = 0
                if diff > 0:
                    diff -= 1
            else:
                run_count += 1
        if run_mode == 0:
            _put_vlc(bw, states[ctx], diff, bits)
    if run_mode:
        while run_count >= 1 << _log2_run(run_index):
            run_count -= 1 << _log2_run(run_index)
            run_index += 1
            bw.put(1, 1)
        if run_count:
            bw.put(1, 1)
    return run_index


def encode_avi(cv2, path, frames, **kw):
    """Encodes frames with Encoder(**kw) into an AVI at path, checks that cv2.VideoCapture decodes it to channel 0 of the
    input exactly, and returns (record, frame bytes, channel 0 [n, h, w])."""
    frames = np.asarray(frames, np.uint8)
    enc = Encoder(frames.ndim == 4, **kw)
    rec, fr = enc.encode(frames)
    h, w = frames.shape[1:3]
    with open(path, "wb") as f:
        f.write(ffv1_avi(fr, w, h, rec))
    want = frames[..., 0] if frames.ndim == 4 else frames
    got = capture(cv2, path)
    assert got.shape == want.shape and np.array_equal(got, want), "cv2.VideoCapture does not decode the encoder's stream to its input"
    return rec, fr, want


def split_slices(frame, n_slices):
    """The slices of one FFV1 frame (ec = 1), footers included, found by walking the footers back from the end."""
    out, end = [], len(frame)
    for _ in range(n_slices):
        v = int.from_bytes(frame[end - 8:end - 5], "big") + 8
        out.append(frame[end - v:end])
        end -= v
    assert end == 0
    return out[::-1]


def make_slice(data):
    """A slice from its coded bytes: 24-bit size, error byte 0, CRC."""
    return with_crc(bytes(data) + len(data).to_bytes(3, "big") + b"\0")


def write_cv2_ffv1(cv2, path, frames):
    """frames: [n, h, w] grey or [n, h, w, 3] BGR, written by cv2.VideoWriter as 'FFV1'; returns what cv2.VideoCapture +
    extractChannel(0) reads back."""
    n, h, w = frames.shape[:3]
    wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"FFV1"), 30.0, (w, h), frames.ndim == 4)
    assert wr.isOpened()
    for f in frames:
        wr.write(f)
    wr.release()
    return capture(cv2, path)
