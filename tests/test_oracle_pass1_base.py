"""Pass 1 of the base class (SURVEY 8f-1): LocoMouse::computeBoundingBox / computeMouseBox / largestBWAreaObject /
computeMouseBoxSize (LocoMouse_class.cpp:579-653, 921-997, 1481-1556).

* The oracle's restatement equals the REFERENCE'S OWN compiled lines (medianBlur and connectedComponentsWithStats executed
  by the real OpenCV through callbacks) on committed vectors and on fresh images -- including the property those lines
  really have: firstLastOverT reads the CV_32S sums through a float pointer, so for min_pixel_visible >= 1 every limit is
  -1 and for 0 every limit spans the whole range, whatever the image shows.
* The pipeline in front of that comparison (median, threshold, largest component, sums), which the float read hides, is
  pinned against the real OpenCV directly (sums_as_float = 0).
"""
import copy
import os

import numpy as np
import pytest

from locomouse_cpp_b200 import synth
from locomouse_cpp_b200.types import bb_base_params
from oracle import oracle
from oracle import reference_nms as ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pass1_base.npz")


def _images(n=5, seed=1000, flip=False):
    spec = synth.SynthSpec(method="base", flip=flip)
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=seed)
    frames = frames.numpy()
    c0 = copy.copy(cfg)
    c0.imadjust = 0
    imgs = np.stack([oracle.preprocess(c0, bkg, calib, frames[f])[0] for f in range(n)])
    return spec, cfg, bkg, calib, frames, imgs


def _views(cfg, spec):
    return (0, 0, cfg.n_cols, spec.side_h), (0, spec.side_h, cfg.n_cols, cfg.n_rows - spec.side_h)


def make_golden():
    spec, cfg, bkg, calib, frames, imgs = _images()
    side, bottom = _views(cfg, spec)
    out = {}
    for th in (0, 1, 7):
        out[f"box_th{th}"] = ref.compute_mouse_box(imgs, side, bottom, 11, th, 8)
    rng = np.random.Generator(np.random.PCG64(11))
    for i in range(12):
        n = int(rng.integers(1, 30))
        w, hb, hs = (np.floor(rng.uniform(50, 400, n)) for _ in range(3))
        out[f"size_in_{i}"] = np.stack([w, hb, hs])
        out[f"size_out_{i}"] = np.array(ref.mouse_box_size(w, hb, hs))
    np.savez_compressed(GOLD, **out)


def test_oracle_equals_reference_golden():
    spec, cfg, bkg, calib, frames, imgs = _images()
    G = np.load(GOLD)
    for th in (0, 1, 7):
        P = bb_base_params(cfg, side_h=spec.side_h, min_pixel_visible=th)
        box, lims = oracle.bounding_box_base(cfg, bkg, calib, frames, P)
        assert np.array_equal(box, G[f"box_th{th}"]), th
    # what the reference's float read of integer sums amounts to
    assert (G["box_th1"][:, [0, 2]] == -1).all() and (G["box_th1"][:, 3:] == 0).all()
    assert (G["box_th0"][:, 0] == cfg.n_cols - 1).all()
    for i in range(12):
        w, hb, hs = G[f"size_in_{i}"]
        assert oracle.mouse_box_size(w, hb, hs) == tuple(int(v) for v in G[f"size_out_{i}"]), i


def test_oracle_equals_reference_fresh():
    if not ref.available():
        pytest.skip("reference library not built (no LocoMouse_cpp checkout, see oracle/reference_nms.py); golden vectors cover it")
    spec, cfg, bkg, calib, frames, imgs = _images(n=3, seed=1003, flip=True)
    side, bottom = _views(cfg, spec)
    for th, k, conn in ((1, 11, 8), (0, 5, 4), (3, 11, 4)):
        want = ref.compute_mouse_box(imgs, side, bottom, k, th, conn)
        c2 = copy.copy(cfg)
        c2.conn = conn
        P = bb_base_params(cfg, side_h=spec.side_h, min_pixel_visible=th, median_filter_size=k)
        got, _ = oracle.bounding_box_base(c2, bkg, calib, frames, P)
        assert np.array_equal(got, want), (th, k, conn)
    rng = np.random.Generator(np.random.PCG64(12))
    for _ in range(60):
        n = int(rng.integers(1, 40))
        w, hb, hs = (np.floor(rng.uniform(0, 500, n)) for _ in range(3))
        assert oracle.mouse_box_size(w, hb, hs) == ref.mouse_box_size(w, hb, hs)


def test_pipeline_behind_the_float_read_matches_opencv():
    """sums_as_float = 0: median (zero-extended window) -> threshold -> largest component -> CV_32S sums -> first / last index
    >= threshold, every step executed by the real OpenCV."""
    cv2 = pytest.importorskip("cv2")
    spec, cfg, bkg, calib, frames, imgs = _images(n=4, seed=1001)
    side, bottom = _views(cfg, spec)
    rng = np.random.Generator(np.random.PCG64(2))
    for f, (k, conn, th) in enumerate(((11, 8, 1), (11, 4, 300), (5, 8, 1), (3, 8, 2000))):
        img = imgs[f].copy()
        speck = rng.uniform(size=img.shape) < 0.02          # isolated specks the median removes / keeps depending on k
        img[speck] = 200
        h = k // 2
        pad = np.zeros((img.shape[0] + 2 * h, img.shape[1] + 2 * h), np.uint8)
        pad[h:h + img.shape[0], h:h + img.shape[1]] = img
        med = cv2.medianBlur(pad, k)[h:h + img.shape[0], h:h + img.shape[1]]
        _, b = cv2.threshold(med, 2.55, 1, cv2.THRESH_BINARY)
        want = []
        for (x, y, w, hh) in (side, bottom):
            v = np.ascontiguousarray(b[y:y + hh, x:x + w])
            n, lab, stats, _ = cv2.connectedComponentsWithStats(v, connectivity=conn, ltype=cv2.CV_32S)
            big = np.zeros_like(v)
            if n > 1:
                best = 1 + int(np.argmax(stats[1:, cv2.CC_STAT_AREA]))   # first maximum = lowest label
                big = ((lab == best) * 255).astype(np.uint8)
            row = cv2.reduce(big, 0, cv2.REDUCE_SUM, dtype=cv2.CV_32S).reshape(-1)
            col = cv2.reduce(big, 1, cv2.REDUCE_SUM, dtype=cv2.CV_32S).reshape(-1)
            want.append((row, col))

        def fl(s):
            q = np.nonzero(s >= th)[0]
            return (-1, -1) if len(q) == 0 else (int(q[0]), int(q[-1]) if len(q) > 1 else 0)

        P = bb_base_params(cfg, side_h=spec.side_h, min_pixel_visible=th, median_filter_size=k, sums_as_float=0)
        box, lims = oracle.mouse_box_base(img, conn, P)
        assert tuple(lims[0]) == fl(want[0][0]) and tuple(lims[1]) == fl(want[1][0]), f
        assert tuple(lims[2]) == fl(want[0][1]) and tuple(lims[3]) == fl(want[1][1]), f
        assert lims.max() > 0


if __name__ == "__main__":
    make_golden()
    print("wrote", GOLD)
