"""MPEG-4 Part 2 test data (csrc/mpeg4_format.h): videos written by cv2.VideoWriter ('mp4v' / 'XVID', libavcodec's mpeg4
encoder), the host reader and CPU decoder entry points, and a small bit writer that rebuilds a stream's VOL with chosen
fields or writes a VOP header, for the streams cv2 does not produce (refusals, not-coded VOPs)."""
import ctypes as C

import numpy as np

from _mjpeg_avi import mjpeg_avi
from _png_avi import capture
from test_match2nd import _host


def write_cv2_mpeg4(cv2, path, frames, fourcc):
    """frames [n, h, w] grey or [n, h, w, 3] BGR through cv2.VideoWriter; returns VideoCapture's channel 0."""
    n, h, w = frames.shape[:3]
    wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*fourcc), 30.0, (w, h), frames.ndim == 4)
    assert wr.isOpened(), (path, fourcc)
    for f in frames:
        wr.write(f)
    wr.release()
    return capture(cv2, path)


def mpeg4_avi(frames, w, h, fourcc=b"XVID"):
    """An AVI whose stream 0 holds the given MPEG-4 frames as '00dc' chunks."""
    return mjpeg_avi(frames, w, h, fourcc)


# ---- host reader / CPU decoder ---------------------------------------------------------------------------------------


def read_video_mpeg4(path):
    """(payload, offsets, extradata, ivop, (n, rows, cols)) of an MPEG-4 video in any container, read with decode_mpeg4 on;
    RuntimeError with the reader's message."""
    fn = _host().lmh_read_video_mpeg4
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p] + [C.c_void_p] * 5 + [C.c_char_p, C.c_int]
    dims = np.zeros(5, np.int64)
    msg = C.create_string_buffer(512)
    if fn(str(path).encode(), dims.ctypes.data, None, None, None, None, msg, 512) != 0:
        raise RuntimeError(msg.value.decode())
    payload = np.zeros(int(dims[3]), np.uint8)
    offs = np.zeros(int(dims[0]) + 1, np.int64)
    extra = np.zeros(max(int(dims[4]), 1), np.uint8)
    ivop = np.zeros(int(dims[0]), np.uint8)
    assert fn(str(path).encode(), dims.ctypes.data, payload.ctypes.data, offs.ctypes.data, extra.ctypes.data, ivop.ctypes.data, msg, 512) == 0
    return payload, offs, extra[:int(dims[4])].copy(), ivop, tuple(int(v) for v in dims[:3])


def decode_cpu(extradata, payload, offsets, rows, cols):
    """mpeg4_format.h on the CPU: uint8 [n, rows, cols]; ValueError with the decoder's message."""
    fn = _host().lmh_decode_mpeg4
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_int]
    ex = np.ascontiguousarray(np.frombuffer(bytes(extradata), np.uint8) if isinstance(extradata, bytes) else extradata, np.uint8)
    pay = np.ascontiguousarray(payload, np.uint8)
    offs = np.ascontiguousarray(offsets, np.int64)
    n = offs.size - 1
    out = np.zeros((n, rows, cols), np.uint8)
    msg = C.create_string_buffer(512)
    if fn(ex.ctypes.data if ex.size else None, ex.size, pay.ctypes.data, offs.ctypes.data, n, rows, cols, out.ctypes.data, msg, 512) != 0:
        raise ValueError(msg.value.decode())
    return out


def plan_mpeg4(path, max_bytes, batch_frames):
    fn = _host().lmh_plan_windows_mpeg4
    fn.restype = C.c_int
    fn.argtypes = [C.c_char_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int]
    starts = np.zeros(4096, np.int32)
    msg = C.create_string_buffer(512)
    k = fn(str(path).encode(), max_bytes, batch_frames, starts.ctypes.data, starts.size, msg, 512)
    if k < 0:
        raise RuntimeError(msg.value.decode())
    return list(starts[:k + 1])


def blue_table():
    """the restated colour rule, [Y, Cb]"""
    fn = _host().lmh_mpeg4_blue
    fn.argtypes = [C.c_void_p]
    t = np.zeros((256, 256), np.uint8)
    fn(t.ctypes.data)
    return t


def vlc_table(t):
    """[(code, length)] of VLC table t of mpeg4_format.h (T_MCBPC_I .. T_TCOEF_INTER)"""
    fn = _host().lmh_mpeg4_vlc
    fn.restype = C.c_int
    fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    codes, lens = np.zeros(256, np.int32), np.zeros(256, np.int32)
    k = fn(t, codes.ctypes.data, lens.ctypes.data)
    return list(zip(codes[:k].tolist(), lens[:k].tolist()))


def split(frames):
    """payload, offsets of a list of frames"""
    offs = np.cumsum([0] + [len(f) for f in frames]).astype(np.int64)
    return np.frombuffer(b"".join(frames), np.uint8).copy(), offs


def frames_of(payload, offs):
    return [bytes(payload[offs[i]:offs[i + 1]]) for i in range(offs.size - 1)]


# ---- start codes and the VOL writer ----------------------------------------------------------------------------------


def segments(data):
    """[(start code byte, start, end)] of the start-code segments of a frame (start: of the 00 00 01)"""
    at = []
    i = data.find(b"\0\0\1")
    while i >= 0 and i + 3 < len(data):
        at.append(i)
        i = data.find(b"\0\0\1", i + 3)
    return [(data[a + 3], a, at[k + 1] if k + 1 < len(at) else len(data)) for k, a in enumerate(at)]


def vop_type(frame):
    """coding type of a frame's VOP: 0 I, 1 P, 2 B, 3 S"""
    for c, a, e in segments(frame):
        if c == 0xB6:
            return frame[a + 4] >> 6
    raise ValueError("no VOP")


class Bits:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, value, bits):
        self.v = (self.v << bits) | (value & ((1 << bits) - 1))
        self.n += bits

    def stuffed(self):
        """the bits with MPEG-4 stuffing (0 then 1s) to a byte boundary"""
        self.put(0, 1)
        while self.n % 8:
            self.put(1, 1)
        return self.v.to_bytes(self.n // 8, "big")


def vol(w, h, res=30, vo_type=1, ver_id=None, shape=0, interlaced=0, sprite=0, not_8_bit=0, quant_type=0, qpel=0, complexity_disable=1,
        resync_disable=1, partitioned=0, newpred=0, reduced=0, scalability=0):
    """a video object layer with these fields (start code 00 00 01 20 included)"""
    b = Bits()
    b.put(0, 1)                  # random_accessible_vol
    b.put(vo_type, 8)
    if ver_id is None:
        b.put(0, 1)
        ver = 1
    else:
        b.put(1, 1), b.put(ver_id, 4), b.put(1, 3)
        ver = ver_id
    b.put(1, 4)                  # square pixels
    b.put(1, 1), b.put(1, 2), b.put(1, 1), b.put(0, 1)  # vol_control_parameters: 4:2:0, low_delay, no vbv
    b.put(shape, 2)
    b.put(1, 1)
    b.put(res, 16)
    b.put(1, 1)
    b.put(0, 1)                  # fixed_vop_rate
    b.put(1, 1), b.put(w, 13), b.put(1, 1), b.put(h, 13), b.put(1, 1)
    b.put(interlaced, 1)
    b.put(1, 1)                  # obmc_disable
    b.put(sprite, 1 if ver == 1 else 2)
    b.put(not_8_bit, 1)
    if not_8_bit:
        b.put(5, 4), b.put(8, 4)
    b.put(quant_type, 1)
    if quant_type:
        b.put(0, 1), b.put(0, 1)  # default matrices
    if ver != 1:
        b.put(qpel, 1)
    b.put(complexity_disable, 1)
    if not complexity_disable:
        b.put(0, 2), b.put(1, 1), b.put(0, 6), b.put(1, 1), b.put(0, 4), b.put(1, 1), b.put(0, 4), b.put(1, 1), b.put(0, 6), b.put(1, 1), b.put(0, 1)
    b.put(resync_disable, 1)
    b.put(partitioned, 1)
    if partitioned:
        b.put(0, 1)
    if ver != 1:
        b.put(newpred, 1)
        if newpred:
            b.put(0, 3)
        b.put(reduced, 1)
    b.put(scalability, 1)
    return b"\0\0\1\x20" + b.stuffed()


def with_vol(frame, new_vol):
    """the frame with every VOL segment replaced by new_vol"""
    out, last = b"", 0
    for c, a, e in segments(frame):
        if 0x20 <= c <= 0x2F:
            out += frame[last:a] + new_vol
            last = e
    return out + frame[last:]


def user_data(text):
    return b"\0\0\1\xb2" + text


def before_vop(frame, extra):
    """the frame with `extra` inserted in front of its VOP start code"""
    at = frame.index(b"\0\0\1\xb6")
    return frame[:at] + extra + frame[at:]


# ---- a test encoder of random, well-formed I- / P-VOP syntax ----------------------------------------------------------
# It writes the syntax elements the decoder reads, chosen at random inside their legal ranges, without modelling what
# they decode to: both decoders (VideoCapture's and this library's) then decode the same bits, so every tool that appears
# in the stream is compared, whatever pixels come out.  Macroblock and block syntax: ISO/IEC 14496-2 6.2.7 - 6.2.8.

T_MCBPC_I, T_MCBPC_P, T_CBPY, T_MVD, T_DC_LUM, T_DC_CHROM, T_TCOEF_INTRA, T_TCOEF_INTER = range(8)
DC_THRESHOLD = (99, 13, 15, 17, 19, 21, 23, 0)  # intra_dc_vlc_thr -> the quantiser below which DC has its own VLC


class Tcoef:
    """the (last, run, level) events of one TCOEF table with their codes, LMAX and RMAX"""

    def __init__(self, intra):
        fn = _host().lmh_mpeg4_tcoef_event
        fn.argtypes = [C.c_int, C.c_int, C.c_void_p]
        codes = vlc_table(T_TCOEF_INTRA if intra else T_TCOEF_INTER)
        self.esc = codes[102]
        self.code, self.lmax, self.rmax = {}, {}, {}
        e = np.zeros(3, np.int32)
        for s in range(102):
            fn(int(intra), s, e.ctypes.data)
            last, run, level = (int(v) for v in e)
            self.code[(last, run, level)] = codes[s]
            self.lmax[(last, run)] = max(self.lmax.get((last, run), 0), level)
            self.rmax[(last, level)] = max(self.rmax.get((last, level), 0), run)


class Mpeg4Fuzz:
    """I- and P-VOPs of random syntax for a w x h VOL (1MV, H.263 quantisation, no resync markers).  Every tool the
    decoder restates appears: stuffing, dquant (and the quantiser's clamp), ac_pred next to neighbours of other quantisers,
    intra DC by its VLC and in the TCOEF table (every intra_dc_vlc_thr), all three TCOEF escapes, not_coded and intra
    macroblocks in P-VOPs, every f_code with MVD residuals (vectors that wrap and point past the edges), both
    rounding_types.  `levels` bounds the coefficient levels (large ones saturate pixels to 0 and 255)."""

    def __init__(self, w, h, seed, levels=40):
        self.w, self.h = w, h
        self.rng = np.random.Generator(np.random.PCG64(seed))
        self.levels = levels
        self.tab = {t: vlc_table(t) for t in (T_MCBPC_I, T_MCBPC_P, T_CBPY, T_MVD, T_DC_LUM, T_DC_CHROM)}
        self.tcoef = {1: Tcoef(True), 0: Tcoef(False)}
        self.time = 0
        self.used = {"dquant": 0, "ac_pred": 0, "dc_in_tcoef": 0, "esc1": 0, "esc2": 0, "esc3": 0, "intra_in_p": 0, "not_coded": 0,
                     "stuffing": 0, "fcodes": set(), "rounding": set()}

    def headers(self):
        return b"\0\0\1\0" + vol(self.w, self.h) + user_data(b"Lavc62.11.100")

    def _put(self, b, t, s):
        c, l = self.tab[t][s]
        b.put(c, l)

    def _events(self, b, intra, first):
        """coefficients from scan position `first` to a random last position"""
        r = self.rng
        tab = self.tcoef[intra]
        pos = first - 1
        while True:
            run = int(min(r.geometric(0.5) - 1, 62 - pos - 1 if pos < 62 else 0))
            pos += run + 1
            last = int(pos >= 62 or r.random() < 0.3)
            level = int(r.integers(1, 4)) if r.random() < 0.8 else int(r.integers(1, self.levels + 1))
            sign = int(r.integers(0, 2))
            ways = []
            if (last, run, level) in tab.code:
                ways.append("plain")
            lm = tab.lmax.get((last, run), 0)
            if lm and (last, run, level - lm) in tab.code:
                ways.append("esc1")
            rm = tab.rmax.get((last, level))
            if rm is not None and (last, run - rm - 1, level) in tab.code:
                ways.append("esc2")
            ways.append("esc3")
            way = ways[int(r.integers(0, len(ways)))] if "plain" not in ways or r.random() < 0.3 else "plain"
            if way == "esc3":
                b.put(*tab.esc), b.put(3, 2), b.put(last, 1), b.put(run, 6), b.put(1, 1), b.put(-level if sign else level, 12), b.put(1, 1)
            else:
                if way == "esc1":
                    b.put(*tab.esc), b.put(0, 1)
                    b.put(*tab.code[(last, run, level - lm)])
                elif way == "esc2":
                    b.put(*tab.esc), b.put(2, 2)
                    b.put(*tab.code[(last, run - rm - 1, level)])
                else:
                    b.put(*tab.code[(last, run, level)])
                b.put(sign, 1)
            if way != "plain":
                self.used[way] += 1
            if last:
                return

    def _intra_mb(self, b, q, thr, cbp):
        """ac_pred, CBPY, dquant and six intra blocks after the MCBPC; returns the new quantiser"""
        r = self.rng
        ac = int(r.integers(0, 2))
        b.put(ac, 1)
        self.used["ac_pred"] += ac
        self._put(b, T_CBPY, cbp >> 2)
        dc_vlc = q < thr
        q = self._dquant(b, q)
        for k in range(6):
            if dc_vlc:  # small differences: a DC that predicts below 0 is an error (libavcodec and here alike)
                size = int(r.integers(0, 4))
                self._put(b, T_DC_LUM if k < 4 else T_DC_CHROM, size)
                if size:
                    v = int(r.integers(1 << (size - 1), 1 << size))
                    b.put(v if r.random() < 0.6 else v ^ ((1 << size) - 1), size)  # positive, or its negative
            else:
                self.used["dc_in_tcoef"] += 1
            if cbp & (32 >> k):
                self._events(b, 1, 1 if dc_vlc else 0)
            elif not dc_vlc:
                pass  # DC 0 + prediction
        return q

    def _dquant(self, b, q):
        if not self._dq:
            return q
        d = int(self.rng.integers(0, 4))
        b.put(d, 2)
        self.used["dquant"] += 1
        return min(31, max(1, q + (-1, -2, 1, 2)[d]))

    def vop(self, kind):
        """one VOP (0 I, 1 P) with its start code, stuffed to a byte boundary"""
        r = self.rng
        b = Bits()
        b.put(kind, 2), b.put(0, 1), b.put(1, 1), b.put(self.time % 30, 5), b.put(1, 1), b.put(1, 1)
        self.time += 1
        rounding = int(r.integers(0, 2))
        if kind:
            b.put(rounding, 1)
            self.used["rounding"].add(rounding)
        thr_code = int(r.integers(0, 8))
        thr = DC_THRESHOLD[thr_code]
        q = int(r.integers(1, 32))
        b.put(thr_code, 3), b.put(q, 5)
        fcode = int(r.integers(1, 8))
        if kind:
            b.put(fcode, 3)
            self.used["fcodes"].add(fcode)
        for _ in range(((self.w + 15) // 16) * ((self.h + 15) // 16)):
            if kind:
                if r.random() < 0.15:
                    b.put(1, 1)  # not_coded
                    self.used["not_coded"] += 1
                    continue
                b.put(0, 1)
                while r.random() < 0.05:
                    self._put(b, T_MCBPC_P, 20)
                    b.put(0, 1)
                    self.used["stuffing"] += 1
                mtype = int(r.choice([0, 1, 3, 4], p=[0.5, 0.2, 0.2, 0.1]))
            else:
                while r.random() < 0.05:
                    self._put(b, T_MCBPC_I, 8)
                    self.used["stuffing"] += 1
                mtype = int(r.choice([3, 4]))
            cbp = int(r.integers(0, 64))
            self._dq = mtype in (1, 4)
            if kind:
                self._put(b, T_MCBPC_P, mtype * 4 + (cbp & 3))
            else:
                self._put(b, T_MCBPC_I, (4 if mtype == 4 else 0) + (cbp & 3))
            if mtype >= 3:
                self.used["intra_in_p"] += kind
                q = self._intra_mb(b, q, thr, cbp)
                continue
            self._put(b, T_CBPY, (cbp >> 2) ^ 15)
            q = self._dquant(b, q)
            for _ in range(2):
                m = int(r.integers(0, 33)) if r.random() < 0.7 else int(r.integers(0, 3))
                self._put(b, T_MVD, m)
                if m:
                    b.put(int(r.integers(0, 2)), 1)
                    if fcode > 1:
                        b.put(int(r.integers(0, 1 << (fcode - 1))), fcode - 1)
            for k in range(6):
                if cbp & (32 >> k):
                    self._events(b, 0, 0)
        return b"\0\0\1\xb6" + b.stuffed()
