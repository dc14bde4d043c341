"""ctypes wrapper of oracle/_ref/libref_nms.so: the REFERENCE's own nmsMax / peakClustering / Candidate / P22D code
(LocoMouse_class.cpp:1610-1905, Candidates/Candidates.cpp) compiled by `make -C oracle ref` against the value-type
shim in oracle/ref_shim.  TEST INFRASTRUCTURE ONLY (tests/ and the golden-vector generator)."""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libref_nms.so")


def _ref_root() -> str:
    """The careylab/LocoMouse_cpp checkout: LOCOMOUSE_CPP_REFERENCE if set, else BASELINE.json's reference_path.  Where
    there is none, the checks against the reference's own code skip and the committed golden vectors under tests/golden/
    stand in for it."""
    env = os.environ.get("LOCOMOUSE_CPP_REFERENCE")
    if env:
        return env
    with open(os.path.join(_HERE, "..", "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


REF_ROOT = _ref_root()
CAND = np.dtype([("x", "<i4"), ("y", "<i4"), ("s", "<f8")])
_lib = None


def make_ref() -> None:
    """Builds oracle/_ref/ from the checkout at REF_ROOT (`make -C oracle ref REF=...`); raises with make's output if
    that fails."""
    p = subprocess.run(["make", "-C", _HERE, "ref", f"REF={REF_ROOT}"], capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"building oracle/_ref/ from {REF_ROOT} failed:\n{p.stdout[-2000:]}\n{p.stderr[-2000:]}")


def available(build: bool = True) -> bool:
    """True when the library exists (built from REF_ROOT on demand)."""
    if not os.path.exists(LIB_PATH) and build and os.path.isdir(os.path.join(REF_ROOT, "LocoMouse_Core")):
        make_ref()
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError(f"oracle/_ref/libref_nms.so is missing and there is no LocoMouse_cpp checkout at {REF_ROOT}")
        L = C.CDLL(LIB_PATH)
        f32p = C.POINTER(C.c_float)
        L.ref_nms_max.restype = C.c_int
        L.ref_nms_max.argtypes = [f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int]
        L.ref_peak_clustering.restype = C.c_int
        L.ref_peak_clustering.argtypes = [f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int]
        L.ref_p22d.restype = C.c_int
        L.ref_p22d.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.ref_vecmovingaverage.restype = None
        L.ref_vecmovingaverage.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.ref_first_last_over_t.restype = None
        L.ref_first_last_over_t.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_void_p]
        L.ref_imadjust_lut.restype = None
        L.ref_imadjust_lut.argtypes = [C.c_double] * 4 + [C.c_void_p]
        L.ref_default_candidate.restype = C.c_int
        L.ref_default_candidate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _run(fn, scores, box_w, box_h, *extra, cap=4096):
    s = np.ascontiguousarray(scores, np.float32)
    out = np.zeros(cap, CAND)
    n = fn(s.ctypes.data_as(C.POINTER(C.c_float)), s.shape[0], s.shape[1], box_w, box_h, *extra, out.ctypes.data, cap)
    assert 0 <= n <= cap
    return out[:n]


def nms_max(scores, box_w, box_h, overlap=0.5):
    return _run(lib().ref_nms_max, scores, box_w, box_h, C.c_double(overlap))


def peak_clustering(scores, box_w, box_h, overlap=0.5, method=3):
    return _run(lib().ref_peak_clustering, scores, box_w, box_h, method, C.c_double(overlap))


def p22d(xb, yb, sb, side):
    """side: list of (y, score).  Returns (number_of_candidates, [(y, s), ...]) of the reference's P22D."""
    ys = np.array([y for y, _ in side], np.int32)
    ss = np.array([s for _, s in side], np.float64)
    oy = np.zeros(max(len(side), 1), np.int32)
    os_ = np.zeros(max(len(side), 1), np.float64)
    n = lib().ref_p22d(xb, yb, float(sb), len(side), ys.ctypes.data, ss.ctypes.data, oy.ctypes.data, os_.ctypes.data, len(oy))
    return n, list(zip(oy[:n].tolist(), os_[:n].tolist()))


def vecmovingaverage(v, window: int):
    """The reference's vecmovingaverage (LocoMouse_class.cpp:1559-1608)."""
    a = np.ascontiguousarray(v, np.float64)
    out = np.zeros(a.size, np.uint32)
    lib().ref_vecmovingaverage(a.ctypes.data, a.size, int(window), out.ctypes.data)
    return out


def first_last_over_t(values, th: int):
    """The reference's firstLastOverT<int> (LocoMouse_class.hpp:411-442)."""
    a = np.ascontiguousarray(values, np.float32)
    fl = np.zeros(2, np.int32)
    lib().ref_first_last_over_t(a.ctypes.data, a.size, int(th), fl.ctypes.data)
    return int(fl[0]), int(fl[1])


def imadjust_lut(low_in=0.0, high_in=0.6, low_out=0.0, high_out=1.0):
    """The 256-entry mapping the reference's LocoMouse::imadjust applies (LocoMouse_class.cpp:3204-3242)."""
    lut = np.zeros(256, np.uint8)
    lib().ref_imadjust_lut(float(low_in), float(high_in), float(low_out), float(high_out), lut.ctypes.data)
    return lut


def match_views(cb, cs, vel_check, tsize_b, tsize_s, T, I, Iprev, x0, y0b, y0s, hb, hs, width, spre_b, spre_s, spost=None,
                cap=4096):
    """The reference's matchingWithVelocityConstraint / xDist / matchViews / checkVelCriterion (LocoMouse_class.cpp:1023-1267)
    on the arguments matchBottomSideCandidates passes (999-1021): the PADDED crops of the current and the previous calibrated
    image (cut here from the zero-extended canvas, class.cpp:672-697) and the pre-pads as offsets.
    cb / cs: lists of (x, y, s) in unpadded-crop coordinates; tsize_* = (cols, rows); crops are `width` x hb / hs at
    (x0, y0b) / (x0, y0s) of I; spre_* = (x, y) pre-pads.  Returns, per bottom candidate, the list of (y_side, score)."""
    L = lib()
    L.ref_match_views.restype = C.c_int
    spost = spost or (spre_b, spre_s)
    I, Iprev = np.ascontiguousarray(I, np.uint8), np.ascontiguousarray(Iprev, np.uint8)
    big = 4 * max(width, hb, hs) + 64

    def crop(img, y0, h, pre, post):
        canvas = np.zeros((img.shape[0] + 2 * big, img.shape[1] + 2 * big), np.uint8)
        canvas[big:big + img.shape[0], big:big + img.shape[1]] = img
        return np.ascontiguousarray(canvas[big + y0 - pre[1]: big + y0 + h + post[1], big + x0 - pre[0]: big + x0 + width + post[0]])

    a = np.array([tuple(c) for c in cb], CAND) if len(cb) else np.zeros(0, CAND)
    b = np.array([tuple(c) for c in cs], CAND) if len(cs) else np.zeros(0, CAND)
    Ib, Ibp = crop(I, y0b, hb, spre_b, spost[0]), crop(Iprev, y0b, hb, spre_b, spost[0])
    It, Itp = crop(I, y0s, hs, spre_s, spost[1]), crop(Iprev, y0s, hs, spre_s, spost[1])
    mn = np.zeros(max(len(cb), 1), np.int32)
    my = np.zeros(cap, np.int32)
    ms = np.zeros(cap, np.float64)
    rc = L.ref_match_views(C.c_void_p(a.ctypes.data), len(cb), C.c_void_p(b.ctypes.data), len(cs), int(bool(vel_check)),
                           int(tsize_b[0]), int(tsize_b[1]), int(tsize_s[0]), int(tsize_s[1]), C.c_double(T),
                           C.c_void_p(Ib.ctypes.data), C.c_void_p(Ibp.ctypes.data), Ib.shape[1], Ib.shape[0],
                           C.c_void_p(It.ctypes.data), C.c_void_p(Itp.ctypes.data), It.shape[1], It.shape[0],
                           int(spre_b[0]), int(spre_b[1]), int(spre_s[0]), int(spre_s[1]),
                           C.c_void_p(mn.ctypes.data), C.c_void_p(my.ctypes.data), C.c_void_p(ms.ctypes.data), cap)
    if rc < 0:
        raise RuntimeError("the reference's pairing code threw (CV_Assert / ROI out of range)")
    n_p22d, total = divmod(rc, 100000)
    assert n_p22d == len(cb) and total <= cap
    out, o = [], 0
    for i in range(len(cb)):
        m = int(mn[i])
        out.append([(int(my[o + j]), float(ms[o + j])) for j in range(m)])
        o += m
    return out


def unary_cost_box(cands, bb_w, bb_h, prior_rows):
    """The reference's LocoMouse::unaryCostBox (LocoMouse_class.cpp:1909-1952) returning its own MyMat.
    prior_rows: (x, y, max_distance, min_x, max_x, min_y, max_y) per prior -> (n, n_priors) array."""
    L = lib()
    L.ref_unary_cost_box.restype = None
    c = np.array([tuple(k) for k in cands], CAND) if len(cands) else np.zeros(0, CAND)
    pr = np.ascontiguousarray(prior_rows, np.float64).reshape(-1, 7)
    out = np.zeros(max(len(c) * len(pr), 1), np.float64)
    L.ref_unary_cost_box(C.c_void_p(c.ctypes.data), len(c), int(bb_w), int(bb_h), C.c_void_p(pr.ctypes.data), len(pr), C.c_void_p(out.ctypes.data))
    return out[:len(c) * len(pr)].reshape(len(pr), len(c)).T.copy()


def pairwise_potential(ci, cip1, grid_x, grid_y, spacing, ong_w, ong_h, max_disp, alpha_vel, occluded_cost, cap=1 << 16):
    """The reference's LocoMouse::pairwisePotential (LocoMouse_class.cpp:1954-2070) and its own MATSPARSE (MyMat.cpp:141-178)
    -> (n_rows, n_cols, jc, ir, pr)."""
    L = lib()
    L.ref_pairwise_potential.restype = C.c_int
    a = np.array([tuple(k) for k in ci], CAND) if len(ci) else np.zeros(0, CAND)
    b = np.array([tuple(k) for k in cip1], CAND) if len(cip1) else np.zeros(0, CAND)
    jc = np.zeros(len(a) + ong_w * ong_h + 1, np.int32)
    ir = np.zeros(cap, np.int32)
    pr = np.zeros(cap, np.float64)
    dims = np.zeros(3, np.int32)
    rc = L.ref_pairwise_potential(C.c_void_p(a.ctypes.data), len(a), C.c_void_p(b.ctypes.data), len(b), C.c_double(grid_x), C.c_double(grid_y),
                                  C.c_double(spacing), int(ong_w), int(ong_h), C.c_double(max_disp), C.c_double(alpha_vel),
                                  C.c_double(occluded_cost), C.c_void_p(jc.ctypes.data), C.c_void_p(ir.ctypes.data), C.c_void_p(pr.ctypes.data),
                                  cap, C.c_void_p(dims.ctypes.data))
    assert rc == 0
    return int(dims[0]), int(dims[1]), jc, ir[:dims[2]].copy(), pr[:dims[2]].copy()


_CC_FN = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_ushort), C.POINTER(C.c_int), C.c_int)


def detect_tail(score_bottom, score_side, conn=8, n_points=15):
    """The reference's detectTail / detectLineCandidates / selectLargestRegion (LocoMouse_class.cpp:2541-2767) on given tail
    score maps (what its two filter2D calls return on the unpadded tail boxes).  connectedComponentsWithStats runs in the
    REAL OpenCV (cv2) through a callback.  Returns (tracks int32[3, n_points], tail_mask uint8[hb, tw] with 0 / 255)."""
    import cv2

    L = lib()
    sb = np.ascontiguousarray(score_bottom, np.float32)
    ss = np.ascontiguousarray(score_side, np.float32)
    assert sb.shape[1] == ss.shape[1]

    def cc(img, rows, cols, connectivity, labels, areas, cap):
        a = np.ctypeslib.as_array(img, shape=(rows, cols))
        n, lab, stats, _ = cv2.connectedComponentsWithStats(a, connectivity=connectivity, ltype=cv2.CV_16U)
        assert n <= cap
        np.ctypeslib.as_array(labels, shape=(rows, cols))[:] = lab
        np.ctypeslib.as_array(areas, shape=(cap,))[:n] = stats[:, cv2.CC_STAT_AREA]
        return int(n)

    cb = _CC_FN(cc)
    tracks = np.zeros((3, n_points), np.int32)
    mask = np.zeros(sb.shape, np.uint8)
    L.ref_detect_tail.restype = C.c_int
    rc = L.ref_detect_tail(C.c_void_p(sb.ctypes.data), C.c_void_p(ss.ctypes.data), sb.shape[0], ss.shape[0], sb.shape[1], int(conn),
                           int(n_points), cb, C.c_void_p(tracks.ctypes.data), C.c_void_p(mask.ctypes.data))
    if rc != 0:
        raise RuntimeError("the reference's tail code threw")
    return tracks, mask


def detect_candidates(crop_b, crop_s, tail_mask, maps, pad_b, pad_s, unpad_b, unpad_s, tsz, cap=256):
    """The reference's detectBottomCandidates + detectSideCandidates (+ detectPointCandidates*, nmsMax, peakClustering;
    LocoMouse_class.cpp:771-870, 1610-1905) for one frame.  crop_b / crop_s: unpadded crops; tail_mask: TAIL_MASK (0 / 255);
    maps: the four filter2D outputs over the padded crops [bottom paw, bottom snout, side paw, side snout] (injected);
    pad_* = (cols, rows) of the padded crops, unpad_* = (x, y) of the unpadded window inside them;
    tsz = (paw_b w, h, paw_s w, h, snout_b w, h, snout_s w, h).  Returns 4 lists of (x, y, score)."""
    L = lib()
    L.ref_detect_candidates.restype = C.c_int
    cb, cs = np.ascontiguousarray(crop_b, np.uint8), np.ascontiguousarray(crop_s, np.uint8)
    tm = np.ascontiguousarray(tail_mask, np.uint8)
    ms = [np.ascontiguousarray(m, np.float32) for m in maps]
    assert ms[0].shape == ms[1].shape == (pad_b[1], pad_b[0]) and ms[2].shape == ms[3].shape == (pad_s[1], pad_s[0])
    ptrs = (C.c_void_p * 4)(*[m.ctypes.data for m in ms])
    i4 = lambda v: (C.c_int * len(v))(*[int(x) for x in v])
    out = np.zeros((4, cap), CAND)
    n = np.zeros(4, np.int32)
    rc = L.ref_detect_candidates(C.c_void_p(cb.ctypes.data), C.c_void_p(cs.ctypes.data), cb.shape[0], cs.shape[0], cb.shape[1],
                                 C.c_void_p(tm.ctypes.data), tm.shape[1], ptrs, i4(pad_b), i4(pad_s), i4(unpad_b), i4(unpad_s), i4(tsz),
                                 C.c_void_p(out.ctypes.data), cap, C.c_void_p(n.ctypes.data))
    if rc != 0:
        raise RuntimeError("the reference's candidate detection threw")
    assert (n <= cap).all()
    return [[(int(c["x"]), int(c["y"]), float(c["s"])) for c in out[k, :n[k]]] for k in range(4)]


_U8OP_FN = C.CFUNCTYPE(None, C.c_int, C.POINTER(C.c_ubyte), C.POINTER(C.c_ubyte), C.c_int, C.c_int)


def read_frame(frame, bkg, calib, flip=False):
    """The reference's LocoMouse::readFrame(cv::Mat&) + correctImage (LocoMouse_class.cpp:1273-1406) on an injected raw frame.
    cv::normalize(F, F, 0, 255, NORM_MINMAX, CV_8UC1) and cv::flip run in the REAL OpenCV (cv2) through a callback;
    cv::subtract is the shim's saturating loop; the calibration gather is the reference's own loop.
    Returns the calibrated image (uint8 [n_rows, n_cols])."""
    import cv2

    L = lib()
    fr, bk = np.ascontiguousarray(frame, np.uint8), np.ascontiguousarray(bkg, np.uint8)
    cal = np.ascontiguousarray(calib, np.int32)

    def op(code, src, dst, rows, cols):
        a = np.ctypeslib.as_array(src, shape=(rows, cols))
        r = cv2.normalize(a, None, 0, 255, cv2.NORM_MINMAX, cv2.CV_8U) if code == 0 else cv2.flip(a, 1)
        np.ctypeslib.as_array(dst, shape=(rows, cols))[:] = r

    cb = _U8OP_FN(op)
    out = np.zeros(cal.shape, np.uint8)
    L.ref_read_frame.restype = C.c_int
    rc = L.ref_read_frame(C.c_void_p(fr.ctypes.data), C.c_void_p(bk.ctypes.data), fr.shape[0], fr.shape[1], C.c_void_p(cal.ctypes.data),
                          cal.shape[0], cal.shape[1], int(bool(flip)), cb, C.c_void_p(out.ctypes.data))
    if rc != 0:
        raise RuntimeError("the reference's readFrame threw")
    return out


_SCALE_FN = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.c_double, C.c_double)


def mouse_box_de(side_view, threshold=255 * 0.05, min_count=10, margin=1.1):
    """The reference's LocoMouse_TM_DE::computeMouseBox_DE + LocoMouse::imadjust_default (LocoMouse_TM_DE.cpp:56-113,
    LocoMouse_class.cpp:3244-3311) on a calibrated side view (its zeroed bands 46 / 760 / 100 / 149 are hard-coded there).
    The scaled 8-bit conversion of imadjust_default runs in the real OpenCV (cv2.convertScaleAbs).  Returns bb_x (double)."""
    import cv2

    L = lib()
    img = np.array(side_view, dtype=np.uint8, order="C", copy=True)   # modified in place by the reference

    def scale(src, dst, rows, cols, alpha, beta):
        a = np.ctypeslib.as_array(src, shape=(rows, cols))
        np.ctypeslib.as_array(dst, shape=(rows, cols))[:] = cv2.convertScaleAbs(a, alpha=alpha, beta=beta)

    cb = _SCALE_FN(scale)
    bbx = C.c_double(0.0)
    L.ref_mouse_box_de.restype = C.c_int
    rc = L.ref_mouse_box_de(C.c_void_p(img.ctypes.data), img.shape[0], img.shape[1], C.c_double(threshold), int(min_count), C.c_double(margin),
                            cb, C.byref(bbx))
    if rc != 0:
        raise RuntimeError("the reference's computeMouseBox_DE threw")
    return float(bbx.value)


_FILT8_FN = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int)
_FLOOD_FN = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int)


def mouse_box_dd(side_view, disk, threshold=3, min_pixel_count=10, min_pixel_visible=1, conn=8, zero=(0, None, 0, None)):
    """The reference's LocoMouse_TM::computeMouseBox_DD + bwAreaOpen + imfill (LocoMouse_TM.cpp:158-269) on a calibrated side
    view, with LocoMouse::imadjust_default (LocoMouse_class.cpp:3244-3311).  zero = (ZERO_COL_PRE, ZERO_COL_POST,
    ZERO_ROW_PRE, ZERO_ROW_POST), None = the image size (an empty band).  connectedComponentsWithStats, filter2D (8-bit,
    BORDER_REPLICATE), floodFill and the scaled 8-bit conversions run in the REAL OpenCV (cv2).  Returns (bb_x, stages):
    stages holds what the reference's code handed to OpenCV on the way -- "adjusted" (I_SIDE after imadjust_default and the
    zeroed bands), "binary" (the labelling's input), "opened" (the filter's input, after bwAreaOpen), "filtered" (the flood
    fill's input) -- and "row_sums" (the CV_32S column sums firstLastOverT reads)."""
    import cv2

    L = lib()
    img = np.array(side_view, dtype=np.uint8, order="C", copy=True)   # modified in place by the reference
    rows, cols = img.shape
    z = [int(zero[0]), cols if zero[1] is None else int(zero[1]), int(zero[2]), rows if zero[3] is None else int(zero[3])]
    dk = np.ascontiguousarray(disk, np.float32)
    assert dk.ndim == 2 and dk.shape[0] == dk.shape[1]

    def scale(src, dst, r, c, alpha, beta):
        a = np.ctypeslib.as_array(src, shape=(r, c))
        np.ctypeslib.as_array(dst, shape=(r, c))[:] = cv2.convertScaleAbs(a, alpha=alpha, beta=beta)

    stages = {}

    def cc(im, r, c, connectivity, labels, areas, cap):
        a = np.ctypeslib.as_array(im, shape=(r, c))
        stages["binary"] = np.array(a, copy=True)
        k, lab, stats, _ = cv2.connectedComponentsWithStats(a, connectivity=connectivity, ltype=cv2.CV_16U)
        assert k <= cap
        np.ctypeslib.as_array(labels, shape=(r, c))[:] = lab
        np.ctypeslib.as_array(areas, shape=(cap,))[:k] = stats[:, cv2.CC_STAT_AREA]
        return int(k)

    def filt(src, dst, r, c, kern, kr, kc):
        a = np.ascontiguousarray(np.ctypeslib.as_array(src, shape=(r, c)))
        stages["opened"] = np.array(a, copy=True)
        kk = np.ascontiguousarray(np.ctypeslib.as_array(kern, shape=(kr, kc)))
        np.ctypeslib.as_array(dst, shape=(r, c))[:] = cv2.filter2D(a, cv2.CV_8U, kk, anchor=(-1, -1), delta=0, borderType=cv2.BORDER_REPLICATE)

    def flood(im, r, c, x, y, value):
        a = np.ascontiguousarray(np.ctypeslib.as_array(im, shape=(r, c)))
        stages["filtered"] = np.array(a, copy=True)
        cv2.floodFill(a, None, (x, y), value)
        np.ctypeslib.as_array(im, shape=(r, c))[:] = a

    cbs = (_SCALE_FN(scale), _CC_FN(cc), _FILT8_FN(filt), _FLOOD_FN(flood))
    bbx = C.c_double(0.0)
    sums = np.zeros(cols, np.int32)
    L.ref_mouse_box_dd.restype = C.c_int
    rc = L.ref_mouse_box_dd(C.c_void_p(img.ctypes.data), rows, cols, int(threshold), int(min_pixel_count), int(min_pixel_visible), int(conn),
                            (C.c_int * 4)(*z), C.c_void_p(dk.ctypes.data), dk.shape[0], *cbs, C.byref(bbx), C.c_void_p(sums.ctypes.data))
    if rc != 0:
        raise RuntimeError("the reference's computeMouseBox_DD threw")
    stages["adjusted"] = img
    stages["row_sums"] = sums
    return float(bbx.value), stages


_MEDIAN_FN = C.CFUNCTYPE(None, C.POINTER(C.c_ubyte), C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.c_int)


def compute_mouse_box(images, side, bottom, median_size=11, min_pixel_visible=1, conn=8):
    """The reference's LocoMouse::computeMouseBox + largestBWAreaObject (LocoMouse_class.cpp:921-997) for a sequence of
    calibrated images (what the base readFrame writes into I_center), set up as computeBoundingBox does (579-631): one
    zero-padded I_median kept across frames.  cv::medianBlur and cv::connectedComponentsWithStats run in the REAL OpenCV
    (cv2) through callbacks.  side / bottom = (x, y, w, h).  Returns box float64[n, 6]."""
    import cv2

    L = lib()
    imgs = np.ascontiguousarray(images, np.uint8)
    n, rows, cols = imgs.shape

    def med(src, dst, r, c, k):
        a = np.ctypeslib.as_array(src, shape=(r, c))
        np.ctypeslib.as_array(dst, shape=(r, c))[:] = cv2.medianBlur(np.ascontiguousarray(a), k)

    def cc(img, r, c, connectivity, labels, areas, cap):
        a = np.ctypeslib.as_array(img, shape=(r, c))
        k, lab, stats, _ = cv2.connectedComponentsWithStats(a, connectivity=connectivity, ltype=cv2.CV_16U)
        assert k <= cap
        np.ctypeslib.as_array(labels, shape=(r, c))[:] = lab
        np.ctypeslib.as_array(areas, shape=(cap,))[:k] = stats[:, cv2.CC_STAT_AREA]
        return int(k)

    m_cb, c_cb = _MEDIAN_FN(med), _CC_FN(cc)
    box = np.zeros((n, 6), np.float64)
    sv = (C.c_int * 4)(*[int(v) for v in side])
    bv = (C.c_int * 4)(*[int(v) for v in bottom])
    L.ref_compute_mouse_box.restype = C.c_int
    rc = L.ref_compute_mouse_box(C.c_void_p(imgs.ctypes.data), n, rows, cols, sv, bv, int(median_size), int(min_pixel_visible), int(conn),
                                 m_cb, c_cb, C.c_void_p(box.ctypes.data))
    if rc != 0:
        raise RuntimeError("the reference's computeMouseBox threw")
    return box


def mouse_box_size(w, hb, hs):
    """The reference's computeMouseBoxSize + medianvec + stdvec (LocoMouse_class.cpp:1481-1556) -> (width, bottom h, side h)."""
    L = lib()
    a, b, c = (np.array(v, np.float64, copy=True) for v in (w, hb, hs))
    size = np.zeros(3, np.int32)
    L.ref_mouse_box_size.restype = C.c_int
    L.ref_mouse_box_size(C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), C.c_void_p(c.ctypes.data), int(a.size), C.c_void_p(size.ctypes.data))
    return tuple(int(v) for v in size)
