"""ctypes binding of liblocomouse_b200.so (the C ABI in include/locomouse_b200.h).

`Detector` is the Python-side handle on one `lm_ctx`: it mirrors, for a batch of frames, the part of
the reference's `LocoMouse` object that the hot loop of main.cpp:54-82 drives (readFrame,
cropBoundingBox, detectTail, detectBottomCandidates, detectSideCandidates,
matchBottomSideCandidates, storePreviousImage).  Errors keep the reference's convention:
LM_ERR_INVALID -> ValueError (std::invalid_argument), everything else -> RuntimeError
(std::runtime_error), main.cpp:94-101.

There is NO CPU fallback: if the CUDA library is missing or no sm_100 device is present, creating a
Detector raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .types import (LM_ERR_INVALID, LM_ERR_OVERFLOW, Config, Model, Results, lm_config, lm_results)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblocomouse_b200.so")
_lib = None

EXPORTS = ("lm_abi_version", "lm_create", "lm_destroy", "lm_last_error", "lm_configure", "lm_set_model",
           "lm_set_background", "lm_set_calibration", "lm_get_geometry", "lm_detect_batch", "lm_last_timing",
           "lm_debug_fetch", "lm_set_option", "lm_get_info", "lm_debug_nms", "lm_bounding_box_tm_de", "lm_moving_average",
           "lm_host_alloc", "lm_host_free", "lm_unary_costs", "lm_pairwise_costs", "lm_bounding_box_base", "lm_mouse_box_size", "lm_bounding_box_tm",
           "lm_decode_png", "lm_device_alloc", "lm_device_free", "lm_decode_ffv1",
           "lm_device_copy")


def _pinned_zeros(shape, dtype):
    """numpy array backed by page-locked memory (device -> host copies then run at the PCIe rate instead of through the
    driver's pageable staging).  tensor.numpy() keeps its tensor alive through the array's base chain."""
    import torch

    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    t = torch.zeros(max(nbytes, 1), dtype=torch.uint8, pin_memory=True)
    return t.numpy()[:nbytes].view(dtype).reshape(shape)


class OverflowError_(RuntimeError):
    """A fixed-capacity list overflowed (LM_ERR_OVERFLOW); results carry per-frame flags."""


def load_library():
    """dlopen the in-tree CUDA library.  Raises (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(make -C locomouse_cpp_b200/csrc). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    L.lm_abi_version.restype = C.c_int
    L.lm_create.restype = C.c_int
    L.lm_create.argtypes = [C.POINTER(vp), i32]
    L.lm_destroy.restype = C.c_int
    L.lm_destroy.argtypes = [vp]
    L.lm_last_error.restype = C.c_char_p
    L.lm_last_error.argtypes = [vp]
    L.lm_configure.restype = C.c_int
    L.lm_configure.argtypes = [vp, C.POINTER(lm_config)]
    L.lm_set_model.restype = C.c_int
    L.lm_set_model.argtypes = [vp, vp]
    L.lm_set_background.restype = C.c_int
    L.lm_set_background.argtypes = [vp, vp]
    L.lm_set_calibration.restype = C.c_int
    L.lm_set_calibration.argtypes = [vp, vp]
    L.lm_get_geometry.restype = C.c_int
    L.lm_get_geometry.argtypes = [vp, vp, vp]
    L.lm_detect_batch.restype = C.c_int
    L.lm_detect_batch.argtypes = [vp, vp, i32, vp, i64, i64, vp, vp, vp, C.POINTER(lm_results)]
    L.lm_last_timing.restype = C.c_int
    L.lm_last_timing.argtypes = [vp, vp, vp]
    L.lm_set_option.restype = C.c_int
    L.lm_set_option.argtypes = [vp, C.c_char_p, i64]
    L.lm_get_info.restype = C.c_int
    L.lm_get_info.argtypes = [vp, C.c_char_p, C.POINTER(C.c_double)]
    L.lm_bounding_box_tm_de.restype = C.c_int
    L.lm_bounding_box_tm_de.argtypes = [vp, vp, i32, i64, vp, vp, vp]
    L.lm_moving_average.restype = C.c_int
    L.lm_moving_average.argtypes = [vp, i64, i32, vp]
    L.lm_debug_nms.restype = C.c_int
    L.lm_debug_nms.argtypes = [vp, i32, i32, vp, vp]
    L.lm_debug_fetch.restype = i64
    L.lm_debug_fetch.argtypes = [vp, i32, i64, vp, i64, vp]
    L.lm_unary_costs.restype = C.c_int
    L.lm_unary_costs.argtypes = [vp, C.POINTER(lm_results), i64, i32, i32, i32, vp, i32, vp]
    L.lm_pairwise_costs.restype = C.c_int
    L.lm_pairwise_costs.argtypes = [vp, C.POINTER(lm_results), i64, i32, vp, vp, vp, vp, vp, i64, vp]
    L.lm_bounding_box_base.restype = C.c_int
    L.lm_bounding_box_base.argtypes = [vp, vp, i32, i64, vp, vp, vp]
    L.lm_bounding_box_tm.restype = C.c_int
    L.lm_bounding_box_tm.argtypes = [vp, vp, i32, i64, vp, vp, vp]
    L.lm_mouse_box_size.restype = C.c_int
    L.lm_mouse_box_size.argtypes = [vp, vp, vp, i64, vp]
    L.lm_host_alloc.restype = C.c_int
    L.lm_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.lm_host_free.restype = C.c_int
    L.lm_host_free.argtypes = [vp]
    L.lm_decode_png.restype = C.c_int
    L.lm_decode_png.argtypes = [vp, vp, i32, vp, i64, vp]
    L.lm_decode_ffv1.restype = C.c_int
    L.lm_decode_ffv1.argtypes = [vp, vp, i64, vp, i32, vp, i64, vp]
    L.lm_device_alloc.restype = C.c_int
    L.lm_device_alloc.argtypes = [vp, C.POINTER(vp), C.c_size_t]
    L.lm_device_free.restype = C.c_int
    L.lm_device_free.argtypes = [vp, vp]
    L.lm_device_copy.restype = C.c_int
    L.lm_device_copy.argtypes = [vp, vp, vp, C.c_size_t]
    _lib = L
    return L


class Detector:
    """One lm_ctx bound to one CUDA device and one video's static inputs."""

    STAGES = ("minmax", "prep", "corr", "tail", "nms", "pair", "total")

    def __init__(self, cfg: Config, model: Model, bkg, calib, device: int = 0):
        self._L = load_library()
        self._ctx = C.c_void_p()
        rc = self._L.lm_create(C.byref(self._ctx), int(device))
        if rc != 0:
            msg = self._L.lm_last_error(None).decode()
            self._ctx = C.c_void_p()
            raise RuntimeError(f"lm_create failed ({rc}): {msg}")
        self.device = int(device)
        self.configure(cfg, model, bkg, calib)

    def configure(self, cfg: Config, model: Model, bkg, calib):
        """Re-configures the context for another video (lm_configure + model, background and calibration); its device
        allocations are kept and reused wherever they are large enough."""
        self.cfg = cfg
        c = cfg.to_c()
        self._check(self._L.lm_configure(self._ctx, C.byref(c)))
        self.set_model(model)
        self.set_background(bkg)
        self.set_calibration(calib)

    # ---- error convention -----------------------------------------------------------------------------
    def _check(self, rc, allow_overflow=False):
        if rc == 0:
            return
        msg = self._L.lm_last_error(self._ctx).decode()
        if rc == LM_ERR_INVALID:
            raise ValueError(msg)
        if rc == LM_ERR_OVERFLOW:
            if allow_overflow:
                return
            raise OverflowError_(msg)
        raise RuntimeError(f"[{rc}] {msg}")

    # ---- per-video state ------------------------------------------------------------------------------
    def set_model(self, model: Model):
        self.model = model
        t = model.to_c()
        self._check(self._L.lm_set_model(self._ctx, C.cast(t, C.c_void_p)))

    def set_background(self, bkg):
        b = np.ascontiguousarray(bkg, dtype=np.uint8)
        if b.shape != (self.cfg.vid_rows, self.cfg.vid_cols):
            # validateImageVideoSize (LocoMouse_class.cpp:498-500) throws std::runtime_error
            raise RuntimeError(f"Background image does not match video size: {b.shape}")
        self._check(self._L.lm_set_background(self._ctx, b.ctypes.data))

    def set_calibration(self, calib):
        m = np.ascontiguousarray(calib, dtype=np.int32)
        if m.shape != (self.cfg.n_rows, self.cfg.n_cols):
            raise ValueError(f"calibration map must be {(self.cfg.n_rows, self.cfg.n_cols)}, got {m.shape}")
        self._check(self._L.lm_set_calibration(self._ctx, m.ctypes.data))

    def geometry(self):
        pads = np.zeros(8, np.int32)
        canvas = np.zeros(4, np.int32)
        self._check(self._L.lm_get_geometry(self._ctx, pads.ctypes.data, canvas.ctypes.data))
        return pads, canvas

    # ---- the hot path -----------------------------------------------------------------------------------
    def detect_batch(self, frames, bb_x, bb_y_side, bb_y_bottom, prev_frame=None, first_frame_index: int = 0,
                     results: Results | None = None, allow_overflow: bool = False) -> Results:
        """frames: uint8 [n, vid_rows, vid_cols] — a numpy array / CPU torch tensor (host path, copies
        happen inside the call) or a CUDA torch tensor on this detector's device (resident path).
        prev_frame: the raw frame preceding frames[0] (same kind of memory), needed iff first_frame_index > 0.
        """
        ptr, n, on_dev, keep = _frames_ptr(frames, self.cfg, self.device)
        pptr = None
        if prev_frame is not None:
            pptr, pn, p_dev, keep2 = _frames_ptr(prev_frame, self.cfg, self.device, single=True)
            if p_dev != on_dev:
                raise ValueError("prev_frame must live in the same memory space as frames")
        bx = np.ascontiguousarray(bb_x, dtype=np.uint32)
        bs = np.ascontiguousarray(bb_y_side, dtype=np.uint32)
        bb = np.ascontiguousarray(bb_y_bottom, dtype=np.uint32)
        if not (bx.size == bs.size == bb.size == n):
            raise ValueError("bounding-box arrays must have one entry per frame")
        res = results if results is not None else Results(n, self.cfg.cand_cap, self.cfg.match_cap, self.cfg.n_tail_points, pinned=True)
        r = res.to_c()
        rc = self._L.lm_detect_batch(self._ctx, ptr, int(on_dev), pptr, n, int(first_frame_index), bx.ctypes.data,
                                     bs.ctypes.data, bb.ctypes.data, C.byref(r))
        self._check(rc, allow_overflow)
        res.rc = rc
        return res

    def set_option(self, name: str, value: int):
        """'screen' (0/1) or 'subbatch'; never changes results."""
        self._check(self._L.lm_set_option(self._ctx, name.encode(), int(value)))

    def info(self, name: str) -> float:
        v = C.c_double(0.0)
        rc = self._L.lm_get_info(self._ctx, name.encode(), C.byref(v))
        if rc != 0:
            raise ValueError(f"unknown info item {name!r}")
        return float(v.value)

    def bounding_box_tm_de(self, frames, params=None, window: int = 5):
        """Pass 1 of LocoMouse_TM_DE (LocoMouse_TM_DE.cpp:8-113) for all frames: returns (BB_X_POS uint32[n] after the
        moving average, raw bb_x float64[n], lims int32[n, 2])."""
        from .types import bb_de_params

        ptr, n, on_dev, keep = _frames_ptr(frames, self.cfg, self.device)
        p = params if params is not None else bb_de_params(self.cfg)
        raw = np.zeros(n, np.float64)
        lims = np.zeros((n, 2), np.int32)
        self._check(self._L.lm_bounding_box_tm_de(self._ctx, ptr, int(on_dev), n, C.addressof(p), raw.ctypes.data, lims.ctypes.data))
        out = np.zeros(n, np.uint32)
        if n:
            self._check(self._L.lm_moving_average(raw.ctypes.data, n, int(window), out.ctypes.data))
        return out, raw, lims

    def bounding_box_base(self, frames, params=None):
        """Pass 1 of the base class, per frame (LocoMouse::computeMouseBox after the base readFrame, LocoMouse_class.cpp:579-631,
        921-997): (box float64[n, 6] = bb_x, bb_y_bottom, bb_y_side, width, height_bottom, height_side; lims int32[n, 4, 2])."""
        from .types import bb_base_params

        ptr, n, on_dev, keep = _frames_ptr(frames, self.cfg, self.device)
        p = params if params is not None else bb_base_params(self.cfg)
        box = np.zeros((n, 6), np.float64)
        lims = np.zeros((n, 4, 2), np.int32)
        self._check(self._L.lm_bounding_box_base(self._ctx, ptr, int(on_dev), n, C.addressof(p), box.ctypes.data, lims.ctypes.data))
        return box, lims

    def bounding_box_tm(self, frames, params):
        """Pass 1 of LocoMouse_TM, per frame (LocoMouse_TM::computeMouseBox_DD after the base readFrame, LocoMouse_TM.cpp:115-269):
        (raw bb_x float64[n], lims int32[n, 2]).  params: types.bb_tm_params(cfg, disk, ...)."""
        ptr, n, on_dev, keep = _frames_ptr(frames, self.cfg, self.device)
        raw = np.zeros(n, np.float64)
        lims = np.zeros((n, 2), np.int32)
        self._check(self._L.lm_bounding_box_tm(self._ctx, ptr, int(on_dev), n, C.addressof(params), raw.ctypes.data, lims.ctypes.data))
        return raw, lims

    def decode_png(self, payload, offsets, out=None):
        """PNG-coded video frames ('MPNG' / 'png ' AVI chunks) decoded on the device: frame i is payload[offsets[i]:offsets[i + 1]].
        payload: uint8 numpy array, CPU tensor (pinned or not) or CUDA tensor on this detector's device.  Returns (or fills
        `out`) a uint8 CUDA tensor [n, vid_rows, vid_cols], channel 0 of each decoded frame, ready for detect_batch and the
        bounding_box_* methods.  A malformed frame raises ValueError naming it."""
        return self._decode(lambda ptr, on_dev, offs, n, out_ptr: self._L.lm_decode_png(self._ctx, ptr, on_dev, offs, n, out_ptr),
                            payload, offsets, out)

    def decode_ffv1(self, extradata, payload, offsets, out=None):
        """FFV1-coded video frames ('FFV1' AVI chunks, version 3) decoded on the device, bit-exact with cv2.VideoCapture's
        channel 0.  extradata: the configuration record (the AVI 'strf' bytes after the BITMAPINFOHEADER); payload, offsets and
        out as for decode_png.  A refused record or a malformed frame raises ValueError naming the reason, frame and slice."""
        ex = np.ascontiguousarray(np.frombuffer(bytes(extradata), np.uint8) if isinstance(extradata, (bytes, bytearray)) else extradata,
                                  dtype=np.uint8).reshape(-1)
        return self._decode(lambda ptr, on_dev, offs, n, out_ptr: self._L.lm_decode_ffv1(self._ctx, ex.ctypes.data, ex.size, ptr, on_dev,
                                                                                          offs, n, out_ptr),
                            payload, offsets, out)

    def _decode(self, call, payload, offsets, out):
        import torch

        offs = np.ascontiguousarray(offsets, dtype=np.int64)
        if offs.ndim != 1 or offs.size < 1:
            raise ValueError("offsets must be a 1-D array of n + 1 entries")
        n = offs.size - 1
        if isinstance(payload, torch.Tensor):
            p = payload.reshape(-1)
            if p.dtype != torch.uint8:
                raise ValueError("payload must be uint8")
            p = p.contiguous()
            on_dev = p.is_cuda
            if on_dev:
                if p.device.index != self.device:
                    raise ValueError(f"payload lives on cuda:{p.device.index}, detector is on cuda:{self.device}")
                torch.cuda.current_stream(p.device).synchronize()
        else:
            p = np.ascontiguousarray(payload, dtype=np.uint8).reshape(-1)
            on_dev = False
        size = p.numel() if isinstance(p, torch.Tensor) else p.size
        if n and (offs[0] < 0 or offs[-1] > size):
            raise ValueError(f"offsets reach outside the payload ({size} bytes)")
        ptr = p.data_ptr() if isinstance(p, torch.Tensor) else p.ctypes.data
        shape = (n, self.cfg.vid_rows, self.cfg.vid_cols)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=f"cuda:{self.device}")
        elif out.dtype != torch.uint8 or tuple(out.shape) != shape or not out.is_cuda or out.device.index != self.device or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous uint8 tensor {shape} on cuda:{self.device}")
        else:
            torch.cuda.current_stream(out.device).synchronize()
        self._check(call(ptr, int(on_dev), offs.ctypes.data, n, out.data_ptr()))
        return out

    def mouse_box_size(self, w, hb, hs):
        """computeMouseBoxSize (LocoMouse_class.cpp:1481-1506) -> (width, bottom height, side height)."""
        a, b, c = (np.array(v, np.float64, copy=True) for v in (w, hb, hs))
        size = np.zeros(3, np.int32)
        self._check(self._L.lm_mouse_box_size(a.ctypes.data, b.ctypes.data, c.ctypes.data, a.size, size.ctypes.data))
        return tuple(int(v) for v in size)

    # ---- cost builders of the host tracker (SURVEY 8f-2) ----------------------------------------------------------------
    def unary_costs(self, res: Results, feat: int, bb_w: int, bb_h: int, priors):
        """UNARY_BOTTOM_{PAW,SNOUT} for every frame of `res` (LocoMouse::unaryCostBox, LocoMouse_class.cpp:1909-1952):
        float64 [n, n_priors, cand_cap]; [f, j, i] = MyMat(i, j) of frame f.  priors: types.location_priors(...)."""
        out = _pinned_zeros((res.n, len(priors), res.cand_cap), np.float64)
        r = res.to_c()
        self._L.lm_unary_costs.restype = C.c_int
        self._check(self._L.lm_unary_costs(self._ctx, C.byref(r), C.c_int64(res.n), int(feat), int(bb_w), int(bb_h), priors, len(priors),
                                           C.c_void_p(out.ctypes.data)))
        return out

    def pairwise_costs(self, res: Results, feat: int, params, cap: int | None = None):
        """PAIRWISE_BOTTOM_{PAW,SNOUT} for every frame >= 1 of `res` (LocoMouse::pairwisePotential + MATSPARSE,
        LocoMouse_class.cpp:1954-2070, MyMat.cpp:141-178) as packed CSC: (offs int64[n + 1], jc int32[n, cand_cap + Nong + 1],
        ir int32[total], pr float64[total]); frame f's matrix has n_bottom[f] + Nong rows, n_bottom[f - 1] + Nong columns."""
        nong = params.ong_w * params.ong_h
        offs = np.zeros(res.n + 1, np.int64)
        jc = _pinned_zeros((max(res.n, 1), res.cand_cap + nong + 1), np.int32)
        total = C.c_int64(0)
        r = res.to_c()
        self._L.lm_pairwise_costs.restype = C.c_int
        if cap is None:   # generous first guess; the library reports the exact need on overflow
            cap = int(res.n) * (2 * nong + 64) + 1024
        for _ in range(2):
            ir = _pinned_zeros((max(cap, 1),), np.int32)
            pr = _pinned_zeros((max(cap, 1),), np.float64)
            rc = self._L.lm_pairwise_costs(self._ctx, C.byref(r), C.c_int64(res.n), int(feat), C.byref(params), C.c_void_p(offs.ctypes.data),
                                           C.c_void_p(jc.ctypes.data), C.c_void_p(ir.ctypes.data), C.c_void_p(pr.ctypes.data), C.c_int64(cap),
                                           C.byref(total))
            if rc == LM_ERR_OVERFLOW and total.value > cap:
                cap = int(total.value)
                continue
            self._check(rc)
            break
        return offs, jc[:res.n], ir[:total.value], pr[:total.value]

    def debug_nms(self, view: int, feat: int, scores):
        """nmsMax (view 0) / peakClustering (view 1) kernels on a given score map -> list of (x, y, score)."""
        from .types import CAND_DTYPE

        h = self.cfg.bb_h_bottom if view == 0 else self.cfg.bb_h_side
        s = np.ascontiguousarray(scores, dtype=np.float32)
        if s.shape != (h, self.cfg.bb_w):
            raise ValueError(f"score map must be {(h, self.cfg.bb_w)}, got {s.shape}")
        out = np.zeros(self.cfg.cand_cap, CAND_DTYPE)
        n = self._L.lm_debug_nms(self._ctx, int(view), int(feat), s.ctypes.data, out.ctypes.data)
        if n < 0:
            self._check(n)
        return out[:n]

    def last_timing(self):
        ms = np.zeros(7, np.float32)
        n = C.c_int64(0)
        self._check(self._L.lm_last_timing(self._ctx, ms.ctypes.data, C.addressof(n)))
        return dict(zip(self.STAGES, map(float, ms))), int(n.value)

    def debug_fetch(self, what: int, frame: int):
        dims = np.zeros(4, np.int32)
        need = self._L.lm_debug_fetch(self._ctx, what, frame, None, 0, dims.ctypes.data)
        nbytes = {0: int(dims[0]) * int(dims[1]), 1: int(dims[0]) * int(dims[1]), 2: int(dims[0]) * int(dims[1]), 3: 8}[what]
        del need
        buf = np.zeros(nbytes, np.uint8)
        got = self._L.lm_debug_fetch(self._ctx, what, frame, buf.ctypes.data, nbytes, dims.ctypes.data)
        if got < 0:
            self._check(int(got))
        if what == 3:
            mm = buf.view(np.int32)
            return np.array([255 - mm[0], mm[1]], np.int32), dims
        return buf.reshape(int(dims[0]), int(dims[1])), dims

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._L.lm_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _frames_ptr(frames, cfg: Config, device: int, single: bool = False):
    """(pointer, n, on_device, keepalive) for numpy arrays and torch tensors."""
    fshape = (cfg.vid_rows, cfg.vid_cols)
    try:
        import torch
    except Exception:  # pragma: no cover
        torch = None
    if torch is not None and isinstance(frames, torch.Tensor):
        t = frames
        if t.dtype != torch.uint8:
            raise ValueError("frames must be uint8")
        if single and t.dim() == 2:
            t = t.unsqueeze(0)
        if t.dim() != 3 or tuple(t.shape[1:]) != fshape:
            raise ValueError(f"frames must be [n, {fshape[0]}, {fshape[1]}], got {tuple(t.shape)}")
        t = t.contiguous()
        if t.is_cuda:
            if t.device.index != device:
                raise ValueError(f"frames live on cuda:{t.device.index}, detector is on cuda:{device}")
            torch.cuda.current_stream(t.device).synchronize()  # producer stream -> library stream hand-over
            return t.data_ptr(), t.shape[0], True, t
        return t.data_ptr(), t.shape[0], False, t
    a = np.ascontiguousarray(frames, dtype=np.uint8)
    if single and a.ndim == 2:
        a = a[None]
    if a.ndim != 3 or a.shape[1:] != fshape:
        raise ValueError(f"frames must be [n, {fshape[0]}, {fshape[1]}], got {a.shape}")
    return a.ctypes.data, a.shape[0], False, a
