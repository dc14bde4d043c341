"""Pre-processing on the CPU: the oracle's normalisation table against cv2.normalize for every (min, max) pair, the size of
the difference a multiply-then-add table would make, and the validity and reach of the designed calibration maps that
tests/test_gpu_preprocess.py feeds to the kernels."""
import numpy as np
import pytest

from locomouse_cpp_b200.types import Config

import _preprocess_designs as D

ROW = 4096 + 7          # one row: cv2's vectorised body covers the first 4 096 pixels, the scalar tail the last few
BODY = 4032


def _pairs():
    return [(a, b) for a in range(256) for b in range(a, 256)]


def _muladd_table(a, b):
    rng = float(b - a)
    scale = 255.0 * (1.0 / rng if rng > 2.220446049250313e-16 else 0.0)
    A, S = np.float32(scale), np.float32(0.0 - a * scale)
    v = np.arange(256, dtype=np.float32)
    return np.clip(np.rint((v * A).astype(np.float32) + S), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("imadjust", [False, True])
def test_normalisation_table_equals_cv2_for_every_pair(oracle, imadjust):
    """For every 0 <= min <= max <= 255: a frame holding min .. max (zero background, identity map) normalised by the
    oracle equals cv2.normalize(NORM_MINMAX, CV_8U) read from its vectorised body, with imadjust(0, 0.6) applied to cv2's
    result when the configuration asks for it."""
    cv2 = pytest.importorskip("cv2")
    cfg = Config(vid_rows=1, vid_cols=ROW, n_rows=1, n_cols=ROW, imadjust=imadjust)
    bkg = np.zeros((1, ROW), np.uint8)
    calib = np.arange(ROW, dtype=np.int32).reshape(1, ROW)
    adj = oracle.imadjust_lut() if imadjust else np.arange(256, dtype=np.uint8)
    bad = []
    for a, b in _pairs():
        row = (a + np.arange(ROW) % (b - a + 1)).astype(np.uint8).reshape(1, ROW)
        I, mm = oracle.preprocess(cfg, bkg, calib, row)
        assert mm.tolist() == [a, b]
        want = adj[cv2.normalize(row, None, 0, 255, cv2.NORM_MINMAX, cv2.CV_8UC1)]
        if not np.array_equal(I[0, :BODY], want[0, :BODY]):
            bad.append((a, b))
    assert bad == [], f"{len(bad)} pairs differ from cv2, first {bad[:5]}"


def test_multiply_then_add_table_differs_on_many_pairs(oracle):
    """The fused table is not an accident of rounding that any formula reproduces: dropping the FMA changes the table for
    thousands of (min, max) pairs, each of which the GPU sweep puts into a frame of its own."""
    cfg = Config(vid_rows=1, vid_cols=256, n_rows=1, n_cols=256, imadjust=False)
    bkg = np.zeros((1, 256), np.uint8)
    calib = np.arange(256, dtype=np.int32).reshape(1, 256)
    n = 0
    for a, b in _pairs():
        if b > a:
            row = np.full((1, 256), a, np.uint8)
            row[0, a:b + 1] = np.arange(a, b + 1)
            I, _ = oracle.preprocess(cfg, bkg, calib, row)
            table = I[0, a:b + 1]
        else:
            table = np.zeros(1, np.uint8)
        n += not np.array_equal(_muladd_table(a, b)[a:b + 1], table)
    print(f"multiply-then-add normalisation differs from the fused one on {n} of 32896 (min, max) pairs")
    assert n > 4000


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("flip", [False, True])
def test_designed_maps_are_valid_and_reach_every_tier(oracle, odd, flip):
    cfg, model = D.small_geometry(odd, flip=flip)
    fbytes = cfg.vid_rows * cfg.vid_cols
    places = D.placements(cfg, model)
    assert len(places) > 100
    for t in places:
        assert oracle.check_roi(cfg, model, *t) == 0
    boxes = D.boxes_of(cfg, model, places)
    tiers = dict.fromkeys(D.TIERS, 0)
    hist = dict.fromkeys(D.HIST16, 0)
    for name, m in D.design_maps(cfg).items():
        assert m.dtype == np.int32 and m.shape == (cfg.n_rows, cfg.n_cols), name
        assert 0 <= m.min() and m.max() < fbytes, name
        for k, v in D.tier_counts(cfg, m, boxes, fbytes).items():
            tiers[k] += v
        for k, v in D.hist16_counts(cfg, m, 3, 0, cfg.n_cols - 3, cfg.n_rows - cfg.bb_h_bottom, fbytes).items():
            hist[k] += v
    print(f"odd={odd} flip={flip} k_prep paths {tiers}\n  k_bb_hist16 paths {hist}")
    assert all(v > 0 for v in tiers.values()), tiers
    assert all(v > 0 for v in hist.values()), hist


def test_run_mode_restatement_on_known_maps():
    """run_mode: a 16-pixel run is flagged where it starts, a 15-pixel run is not; a mirrored reversed row is ascending."""
    cfg = Config(vid_rows=4, vid_cols=40, n_rows=1, n_cols=40)
    m = np.zeros((1, 40), np.int64)
    m[0, :16] = 100 + np.arange(16)          # run of 16
    m[0, 16:31] = 10 + np.arange(15)         # run of 15
    m[0, 31:] = 150 - np.arange(9)           # descending run of 9
    _, mode = D.run_mode(m, False)
    assert mode[0, 0] == 5 and mode[0, 1] == 1 and mode[0, 16] == 1 and mode[0, 31] == 2
    _, mode = D.run_mode(D.map_reversed(Config(vid_rows=2, vid_cols=20, n_rows=2, n_cols=20)), True)
    assert mode[0, 0] == 5 and mode[1, 4] == 5 and mode[1, 5] == 1


@pytest.mark.parametrize("name", list(D.IMADJUST_DESIGNS))
def test_imadjust_designs_hit_their_boundary(oracle, name):
    """Each side-view histogram of the imadjust_default designs gives the (i0, i1) it was built for, and where the design
    sits on a boundary, moving one pixel across it changes the first difference the stretched table passes."""
    W, H, band, filler, alt, want = D.IMADJUST_DESIGNS[name]
    frame, hist = D.imadjust_frame(name, *D.imadjust_shape(name))
    assert int(hist.sum()) == W * H < (1 << 24)
    assert oracle.imadjust_default_lut(hist)[1] == want
    th, first = D.imadjust_threshold(oracle, name)
    assert (th is None) == (alt is None)
    if alt is not None:
        assert 0 <= first < 256


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("flip", [False, True])
def test_de_frames_see_the_calibration_map(oracle, odd, flip):
    """The LocoMouse_TM_DE pass-1 frames of the GPU test give limits that move with the body and change with every
    designed map, so a gather or a kept difference through the wrong pixels would show."""
    cfg, _ = D.small_geometry(odd, flip=flip)
    bkg = D.background(cfg)
    D.assert_de_input_sees_the_map(oracle, cfg, bkg, D.de_frames(cfg, bkg), D.de_params(cfg))
