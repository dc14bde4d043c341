"""Pass 1 of LocoMouse_TM (LocoMouse_TM::computeMouseBox_DD / bwAreaOpen / imfill, LocoMouse_TM.cpp:158-269): the oracle's
restatement against the REFERENCE'S OWN compiled lines (oracle/_ref, every OpenCV algorithm executed by the real cv2), stage by
stage, on fresh inputs where /root/reference is mounted and on the committed vectors everywhere."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle, reference_nms

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_pass1_tm.npz")


def disk(r):
    """A normalised disk like MATLAB's fspecial('disk', r) (the reference ships no diskfilter.yml)."""
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    h = ((x * x + y * y) <= (r + 0.5) ** 2).astype(np.float64)
    return (h / h.sum()).astype(np.float32)


def make_side(rng, rows, cols, kind):
    img = np.zeros((rows, cols), np.uint8)
    if kind != "empty":
        x0 = int(rng.integers(cols // 8, cols // 2))
        w = int(rng.integers(cols // 6, cols // 3))
        y0 = int(rng.integers(rows // 6, rows // 2))
        h = int(rng.integers(rows // 4, rows // 2))
        img[y0:y0 + h, x0:x0 + w] = rng.integers(30, 220, (h, w))
        # holes (imfill), a ring that encloses background, specks (bwAreaOpen)
        img[y0 + h // 3:y0 + h // 2, x0 + w // 3:x0 + w // 2] = 0
        for _ in range(int(rng.integers(3, 12))):
            yy, xx = int(rng.integers(0, rows - 4)), int(rng.integers(0, cols - 4))
            img[yy:yy + int(rng.integers(1, 4)), xx:xx + int(rng.integers(1, 4))] = int(rng.integers(60, 255))
        if kind == "noisy":
            img[rng.random(img.shape) < 0.02] = 180
        if kind == "touching":   # foreground on pixel (0, 0): the flood fill starts on the object
            img[0:rows // 3, 0:cols // 5] = 200
    return img


CASES = [("plain", 8, 10, 1, 1), ("noisy", 4, 25, 1, 1), ("noisy", 8, 3, 0, 0), ("touching", 8, 10, 1, 0), ("empty", 8, 10, 1, 1),
         ("plain", 4, 1, 5, 0), ("plain", 8, 40, 300, 0), ("noisy", 8, 12, 2000, 0)]


def run_oracle(img, dk, threshold, min_count, min_vis, conn, zero, as_float):
    return oracle.mouse_box_tm(img, dk, threshold=threshold, min_pixel_count=min_count, min_pixel_visible=min_vis, conn=conn, zero=zero,
                               sums_as_float=as_float)


def check(got, bbx_ref, st_ref):
    bbx, lims, st = got
    for k in ("adjusted", "binary", "opened", "filtered", "row_sums"):
        assert np.array_equal(st[k], st_ref[k]), k
    assert bbx == bbx_ref


@pytest.mark.skipif(not reference_nms.available(), reason="no LocoMouse_cpp checkout (see oracle/reference_nms.py): committed vectors only")
def test_oracle_equals_reference_compiled_code_stage_by_stage():
    rng = np.random.default_rng(77)
    for i, (kind, conn, min_count, min_vis, as_float) in enumerate(CASES * 2):
        rows, cols = int(rng.integers(40, 120)), int(rng.integers(90, 260))
        img = make_side(rng, rows, cols, kind)
        zero = (int(rng.integers(0, 6)), cols - int(rng.integers(0, 6)), int(rng.integers(0, 5)), rows - int(rng.integers(0, 5)))
        dk = disk(int(rng.integers(1, 6)))     # up to 11 x 11 = 121 taps: OpenCV's direct path
        thr = int(rng.integers(0, 12))
        bbx_ref, st_ref = reference_nms.mouse_box_dd(img, dk, threshold=thr, min_pixel_count=min_count, min_pixel_visible=min_vis, conn=conn, zero=zero)
        # the reference always reads the sums through a float pointer: sums_as_float = 1 is its result
        check(run_oracle(img, dk, thr, min_count, min_vis, conn, zero, 1), bbx_ref, st_ref)
        # the integer reading: same stages, limits from the integer sums
        bbx_i, lims_i, st_i = run_oracle(img, dk, thr, min_count, min_vis, conn, zero, 0)
        ok = np.nonzero(st_ref["row_sums"] >= min_vis)[0]
        want = (-1, -1) if ok.size == 0 else (int(ok[0]), int(ok[-1]) if ok.size > 1 else 0)
        assert tuple(lims_i) == want and bbx_i == float(want[1])


def test_reference_float_read_of_integer_sums():
    """firstLastOverT reads CV_32S sums as floats (LocoMouse_class.hpp:417): with min_pixel_visible >= 1 nothing qualifies."""
    rng = np.random.default_rng(5)
    img = make_side(rng, 60, 150, "plain")
    bbx, lims, _ = run_oracle(img, disk(3), 3, 5, 1, 8, (0, 150, 0, 60), 1)
    assert bbx == -1.0 and tuple(lims) == (-1, -1)
    bbx, lims, _ = run_oracle(img, disk(3), 3, 5, 0, 8, (0, 150, 0, 60), 1)
    assert bbx == 149.0 and tuple(lims) == (0, 149)
    bbx, lims, st = run_oracle(img, disk(3), 3, 5, 1, 8, (0, 150, 0, 60), 0)
    cols = np.nonzero(st["row_sums"] >= 1)[0]
    assert bbx == float(cols[-1]) and lims[0] == cols[0]


def test_oracle_equals_committed_reference_vectors():
    z = np.load(GOLD)
    n = int(z["n"])
    assert n >= 8
    for i in range(n):
        img, dk = z[f"img{i}"], z[f"disk{i}"]
        thr, min_count, min_vis, conn = (int(v) for v in z[f"par{i}"][:4])
        zero = tuple(int(v) for v in z[f"par{i}"][4:8])
        st_ref = {k: z[f"{k}{i}"] for k in ("adjusted", "binary", "opened", "filtered", "row_sums")}
        check(run_oracle(img, dk, thr, min_count, min_vis, conn, zero, 1), float(z[f"bbx{i}"]), st_ref)


def test_larger_disks_agree_with_opencv_away_from_ties():
    """Kernels of >= 130 taps take OpenCV's DFT path, whose float noise can flip results only where the exact sum is within
    ~1e-5 of a .5 tie: everywhere else the row-major float sum is what cv2 returns."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(9)
    img = (rng.random((70, 160)) < 0.45).astype(np.uint8)
    dk = disk(7)  # 15 x 15
    got = cv2.filter2D(img, cv2.CV_8U, dk, anchor=(-1, -1), delta=0, borderType=cv2.BORDER_REPLICATE)
    exact = cv2.filter2D(img.astype(np.float64), cv2.CV_64F, dk.astype(np.float64), anchor=(-1, -1), delta=0, borderType=cv2.BORDER_REPLICATE)
    mine = oracle.filter2d_u8(img, dk)
    away = np.abs(exact - np.floor(exact) - 0.5) > 1e-4
    assert np.array_equal(mine[away], got[away])
    assert away.mean() > 0.99


def make_golden():
    """Writes tests/golden/reference_pass1_tm.npz from the reference's own compiled code (needs /root/reference + cv2):
    python -c "import sys; sys.path.insert(0, 'tests'); import test_oracle_pass1_tm as t; t.make_golden()" """
    rng = np.random.default_rng(2024)
    out = {}
    i = 0
    for kind, conn, min_count, min_vis, _as_float in CASES + [("plain", 8, 6, 0, 0), ("noisy", 4, 9, 1, 0)]:
        rows, cols = int(rng.integers(30, 70)), int(rng.integers(70, 150))
        img = make_side(rng, rows, cols, kind)
        zero = (int(rng.integers(0, 6)), cols - int(rng.integers(0, 6)), int(rng.integers(0, 5)), rows - int(rng.integers(0, 5)))
        dk = disk(int(rng.integers(1, 6)))
        thr = int(rng.integers(0, 12))
        bbx, st = reference_nms.mouse_box_dd(img, dk, threshold=thr, min_pixel_count=min_count, min_pixel_visible=min_vis, conn=conn, zero=zero)
        out[f"img{i}"], out[f"disk{i}"], out[f"bbx{i}"] = img, dk, np.float64(bbx)
        out[f"par{i}"] = np.array([thr, min_count, min_vis, conn, *zero], np.int32)
        for k in ("adjusted", "binary", "opened", "filtered", "row_sums"):
            out[f"{k}{i}"] = st[k]
        i += 1
    out["n"] = np.int32(i)
    np.savez_compressed(GOLD, **out)
