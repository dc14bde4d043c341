"""CPU side of the designed-frame tests (tests/_designed_frames.py): the harness maps every designed pixel to itself, the
restated screen bound holds on every output of windows built to sit on its edges (and they really sit there), and the
oracle's largest-region choice on the designed tail maps is OpenCV's."""
import numpy as np
import pytest

import _designed_frames as D

# An output whose exact score is > 0 must come this close (as a fraction of t_hi - t_lo) to t_lo, and a tail output with
# score <= 0 this close to t_hi, for the small templates.  Both fractions reached are about 0.02 - 0.03; a bound shrunk by
# the 255 * E_q term moves t_lo and t_hi by nearly half the band.
EDGE_FRACTION_SMALL = 0.05
# Templates with hundreds of taps: the fp32 term alone is a third of the band, so the edge is reached only to within it.
EDGE_FRACTION_LARGE = 0.45


def test_lround_rounds_halfway_cases_away_from_zero():
    assert [D.lround(x) for x in (0.5, 1.5, 2.5, -0.5, -2.5, 0.49999999999999994, 3.2, -3.7)] == [1, 2, 3, -1, -3, 0, 3, -4]


def test_screen_quantize_restatement_degenerate_and_clamped():
    qz = D.screen_quantize(np.zeros((2, 3), np.float32), 0.0)
    assert qz["scale"] == 1.0 and qz["eq"] == 0.0 and not qz["vq"].any()
    assert qz["t_lo"] == -2 and qz["t_hi"] == 2 and qz["q_need"] == -1 and qz["q_sign"] == 0
    w = np.array([[1.0, -1.0, 0.5 / 32000.0 * 2.5]], np.float32)     # 2.5 units (to float32): lround, not half-even
    qz = D.screen_quantize(w, 1.0)
    assert list(qz["vq"][0]) == [32000, -32000, D.lround(float(w[0, 2]) / qz["scale"])]


def test_tight_templates_have_one_residual_sign():
    for shape in ((2, 2), (3, 5), (40, 40)):
        for d in (1, -1):
            w = D.tight_template(shape, D.tap_layout(shape), d)
            qz = D.screen_quantize(w, 0.0)
            res = w.astype(np.float64) - qz["scale"] * qz["vq"]
            nz = (w != 0) & (qz["vq"] != 32000)
            assert np.all(res[nz] * d > 0)
            assert 255 * qz["eq"] > 0.9 * 255 * qz["scale"] * 0.48 * (nz.sum() - 1)   # every k-tap near half a unit


@pytest.mark.parametrize("shapes,fma_mode", [(D.SMALL_SHAPES, True), (D.SMALL_SHAPES, False), (D.MIXED_SHAPES, True),
                                             (D.LARGE_SHAPES, True)], ids=["small", "small-nofma", "mixed", "large40"])
def test_threshold_designs_obey_the_bound_and_sit_on_its_edges(oracle, shapes, fma_mode):
    cfg, model, bkg, calib, frames, bx, bs, bb = D.threshold_problem(shapes, fma_mode)   # also checks the harness
    tight = shapes is D.SMALL_SHAPES
    frac = EDGE_FRACTION_SMALL if tight else EDGE_FRACTION_LARGE
    near_lo, near_hi, at_q_need = {}, {}, 0
    for v in (0, 1):
        for k in (0, 1, 2):
            for f in range(len(frames)):
                V, _, _, qz = D.view_outputs(cfg, model, frames[f], v, k, fma_mode)
                span = qz["t_hi"] - qz["t_lo"]
                H = np.floor_divide(V, 256)
                for mode in (True, False):
                    sc = D.view_outputs(cfg, model, frames[f], v, k, mode)[1]
                    pos = sc > 0
                    # the bound: V <= t_lo proves score <= 0, V > t_hi proves score > 0 (both accumulation orders)
                    assert not np.any(pos & (V <= qz["t_lo"])), (v, k, f, mode)
                    assert np.all(pos[V > qz["t_hi"]]), (v, k, f, mode)
                    # the 32-bit forms: H >= q_need whenever V > t_lo; H > q_sign only when V > t_hi
                    assert np.all(H[V > qz["t_lo"]] >= qz["q_need"])
                    assert np.all(V[H > qz["q_sign"]] > qz["t_hi"])
                sc = D.view_outputs(cfg, model, frames[f], v, k, fma_mode)[1]
                pos = sc > 0
                if k < 2 and pos.any():
                    near_lo[(v, k)] = min(near_lo.get((v, k), 1.0), float((V[pos] - qz["t_lo"]).min()) / span)
                    at_q_need += int((pos & (H == qz["q_need"])).sum())
                if k == 2 and (~pos).any():
                    near_hi[v] = min(near_hi.get(v, 1.0), float((qz["t_hi"] - V[~pos]).min()) / span)
    assert set(near_lo) == {(0, 0), (0, 1), (1, 0), (1, 1)} and set(near_hi) == {0, 1}
    print(f"edge fractions: paw / snout {sorted(near_lo.values())}, tail {sorted(near_hi.values())}")
    assert max(near_lo.values()) < frac and max(near_hi.values()) < frac
    if tight:
        assert at_q_need > 0        # positives in the block H = q_need: k_screen2 must keep them with H >= q_need


def test_threshold_problem_tail_frame_is_empty_in_the_oracle(oracle):
    """Frame 1 carries only tail windows with score <= 0 in the bottom view: the oracle's tracks are all -1 there, so one
    output wrongly declared positive by the screen changes the result."""
    cfg, model, bkg, calib, frames, bx, bs, bb = D.threshold_problem(D.SMALL_SHAPES)
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb)
    assert np.all(ref.tail[1] == -1)
    assert np.any(ref.tail[2] >= 0)
    assert ref.n_bottom[0].sum() > 0 and ref.n_side[0].sum() > 0


def _cv2_winner(binary, conn):
    cv2 = pytest.importorskip("cv2")
    n, labels, stats, _ = cv2.connectedComponentsWithStats(np.ascontiguousarray(binary, np.uint8), connectivity=conn)
    if n <= 1:
        return np.zeros_like(binary, np.uint8), 0
    areas = stats[1:, cv2.CC_STAT_AREA]
    best = 1 + int(np.argmax(areas))             # largest area, ties -> lowest label
    return (labels == best).astype(np.uint8), int((areas == areas.max()).sum())


@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("name", sorted(D.TAIL_MAPS))
def test_tail_maps_oracle_agrees_with_cv2(oracle, name, conn):
    b, s = D.TAIL_MAPS[name]
    want_b, ties = _cv2_winner(b, conn)
    got_b = oracle.largest_region(b, conn) != 0
    assert np.array_equal(got_b, want_b != 0)
    gate = want_b.max(axis=0) != 0
    side_in = ((s != 0) & gate[None, :]).astype(np.uint8)
    want_s, _ = _cv2_winner(side_in, conn)
    assert np.array_equal(oracle.largest_region(side_in, conn) != 0, want_s != 0)
    tracks, mask = oracle.tail_from_binary(b, s, conn, 15)
    assert np.array_equal(mask != 0, want_b != 0)
    if (name.startswith("tie_") and name != "tie_diagonal") or (name in ("checkerboard", "tie_diagonal") and conn == 4):
        assert ties >= 2, "the map was meant to hold a tie"


def test_tail_map_ties_pick_different_regions_per_connectivity():
    """The block-vs-raster map is the one where 8- and 4-connectivity orders disagree (OpenCV's 8-connectivity labels by
    2x2 blocks)."""
    b, _ = D.TAIL_MAPS["tie_block_vs_raster"]
    w8, _ = _cv2_winner(b, 8)
    w4, _ = _cv2_winner(b, 4)
    assert w8[1, 10] == 1 and w4[0, 12] == 1


def test_unit_model_maps_pixels_to_the_binary_map(oracle):
    b, s = D.TAIL_MAPS["word_crossing_runs"]
    bottom, side = D.maps_to_boxes(b[None], s[None])
    bottom[0, 0, 0] = 26
    bottom[0, 1, 0] = 25
    cfg, model, bkg, calib, frames, *_ = D.make_problem(bottom, side, D.unit_model())
    _, sc, _, _ = D.view_outputs(cfg, model, frames[0], 0, 2, True)
    want = b.copy()
    want[0, 0], want[1, 0] = 1, 0
    assert np.array_equal(sc > 0, want != 0)


@pytest.mark.parametrize("fma_mode", [True, False])
def test_zero_score_designs_hit_zero_exactly(oracle, fma_mode):
    """The designed output scores exactly +0.0, the smallest positive value the rho search reaches, and -0.0."""
    for name, (problem, (v, x, y)) in D.zero_score_problems(fma_mode).items():
        cfg, model, bkg, calib, frames, *_ = problem
        x0, y0 = D.box_origin(cfg, v)
        f = 1 if name == "negzero" else 0
        sc = D.output_score(frames[f], model.w[v][0], model.rho[v][0], x0 + x, y0 + y, fma_mode)
        assert frames[f][y0 + y, x0 + x] > 25
        if name == "zero":
            assert sc == 0.0 and not np.signbit(sc)
        elif name == "negzero":
            assert sc == 0.0 and np.signbit(sc)
        else:   # the smallest positive score that float32 values of float(-rho) give this output: a few ulps of rho
            assert 0 < sc <= 4 * np.spacing(np.float32(model.rho[v][0]))


@pytest.mark.parametrize("conn", [4, 8])
def test_tail_mask_problem_keeps_its_tie(oracle, conn):
    """The paw pixels of the TAIL_MASK test lie on tail pixels: frame 0's bottom map still holds the equal-area tie, and the
    winner (which decides whether the paw pixel in A or the one in B is masked) differs between the connectivities."""
    cv2 = pytest.importorskip("cv2")
    problem, maps = D.tail_mask_problem(conn)
    cfg, model, bkg, calib, frames, *_ = problem
    _, sc, _, _ = D.view_outputs(cfg, model, frames[0], 0, 2, True)
    assert np.array_equal(sc > 0, maps[0] != 0)
    n, _, stats, _ = cv2.connectedComponentsWithStats(maps[0], connectivity=conn)
    assert list(stats[1:, cv2.CC_STAT_AREA]) == [4, 4]
    winner, _ = _cv2_winner(maps[0], conn)
    assert winner[2, 10] == (1 if conn == 8 else 0) and winner[0, 13] == (0 if conn == 8 else 1)


def test_bbox_tie_problem_keeps_its_ties(oracle):
    """After the 3 x 3 median the thickened maps still hold their ties, and the oracle's pass-1 limits depend on the
    connectivity on some frame (a wrong winner changes the result)."""
    import dataclasses

    (cfg, model, bkg, calib, frames, params), med_b, med_s = D.bbox_tie_problem()
    for f, name in enumerate(D.BBOX_TIE_MAPS):
        for conn in (4, 8):
            if conn == 8 and name in ("tie_diagonal", "checkerboard"):
                continue
            for m in (med_b[f], med_s[f]):
                assert _cv2_winner(m.astype(np.uint8), conn)[1] >= 2, (name, conn)
    lims = [oracle.bounding_box_base(dataclasses.replace(cfg, conn=c), bkg, calib, frames, params)[1] for c in (4, 8)]
    assert not np.array_equal(lims[0], lims[1])
