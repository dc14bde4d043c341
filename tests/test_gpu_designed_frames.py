"""Designed frames on the device (tests/_designed_frames.py): outputs placed on the screen's decision thresholds, tail maps
with ties, spirals and edge cases on the fast and the slow labelling path, and TAIL_MASK / Q6 in the pipeline.  Every result
must equal the oracle bit for bit.  Needs a B200:  pytest -m gpu."""
import numpy as np
import pytest

import _designed_frames as D
from locomouse_cpp_b200.types import BOTTOM, PAW, diff_results

pytestmark = pytest.mark.gpu


def _detect(problem, screen, layout=3, **opts):
    from locomouse_cpp_b200.api import Detector

    cfg, model, bkg, calib, frames, bx, bs, bb = problem
    det = Detector(cfg, model, bkg, calib, device=0)
    try:
        det.set_option("screen", screen)
        det.set_option("screen_layout", layout)
        det.set_option("subbatch", len(frames))
        for k, v in opts.items():
            det.set_option(k, v)
        got = det.detect_batch(frames, bx, bs, bb)
        info = {k: det.info(k) for k in ("screen_active", "positives")}
        info.update({f"{q}_{v}{f}": det.info(f"screen_{q}_{v}{f}") for q in ("eps", "scale") for v in (0, 1) for f in (0, 1, 2)})
    finally:
        det.close()
    return got, info


@pytest.mark.parametrize("shapes,fma_mode", [(D.SMALL_SHAPES, True), (D.SMALL_SHAPES, False), (D.MIXED_SHAPES, True),
                                             (D.LARGE_SHAPES, True)], ids=["small", "small-nofma", "mixed", "large40"])
def test_threshold_designs_equal_oracle_in_every_screen_mode(oracle, shapes, fma_mode):
    """Outputs in the blocks H = q_need - 1, q_need, q_need + 1 and next to t_lo / t_hi, at x = 0 / 31 (mod 32), the last
    column, y = 127 / 128 / 255 / 256 and in side-view tiles that straddle frames: the CTA-pair screen in all four layouts,
    the single-CTA screen and the dense kernel give the oracle's results, keep every positive output, and use the restated
    quantisation scale and error bound."""
    problem = D.threshold_problem(shapes, fma_mode)
    cfg, model, bkg, calib, frames, bx, bs, bb = problem
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=4)
    n_pos = D.count_positives(cfg, model, frames)
    assert n_pos > 0
    large = shapes is D.LARGE_SHAPES
    runs = [(2, layout, 2.0) for layout in (3, 2, 1, 0)] + [(1, 3, 0.0 if large else 1.0), (0, 3, 0.0)]
    for screen, layout, active in runs:
        got, info = _detect(problem, screen, layout)
        assert info["screen_active"] == active, (screen, layout)
        assert diff_results(got, ref) == [], (screen, layout)
        assert info["positives"] == n_pos, (screen, layout)
        if screen == 2:
            for v in (0, 1):
                for f in (0, 1, 2):
                    qz = D.screen_quantize(model.w[v][f], model.rho[v][f])
                    assert info[f"eps_{v}{f}"] == qz["eps"] and info[f"scale_{v}{f}"] == qz["scale"], (v, f)


@pytest.mark.parametrize("fma_mode", [True, False])
def test_subnormal_and_zero_scores(oracle, fma_mode):
    """1 x 1 templates with w = 2^-149 and rho = 25 * 2^-149: pixel 26 scores the smallest subnormal, pixel 25 exactly 0
    (not a detection).  No flush-to-zero anywhere, so the lists equal the oracle bit for bit."""
    tiny = np.float32(np.ldexp(1.0, -149))
    rng = np.random.Generator(np.random.PCG64(5))
    b = rng.choice(np.array([0, 24, 25, 26, 27, 255], np.uint8), size=(2, D.MAP_BOX[1], D.MAP_BOX[0]), p=[.9, .02, .02, .02, .02, .02])
    s = rng.choice(np.array([0, 25, 26], np.uint8), size=(2, D.MAP_BOX[2], D.MAP_BOX[0]), p=[.96, .02, .02])
    model = D.unit_model()
    w = np.full((1, 1), tiny, np.float32)
    model.w = [[w, w, model.w[0][2]], [w, w, model.w[1][2]]]
    model.rho = [[25 * float(tiny), 25 * float(tiny), 25.5], [25 * float(tiny), 25 * float(tiny), 25.5]]
    problem = D.make_problem(b, s, model, fma_mode=fma_mode, cand_cap=1024, match_cap=8192)
    cfg, model, bkg, calib, frames, bx, bs, bb = problem
    sc = D.view_outputs(cfg, model, frames[0], BOTTOM, PAW, fma_mode)[1]
    px = frames[0][cfg.bb_h_side:, D.MARGIN:D.MARGIN + cfg.bb_w]
    assert np.all(sc[px == 26] == tiny) and np.all(sc[px == 25] == 0.0)
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb)
    assert ref.n_bottom[:, PAW].sum() > 0 and not ref.flags.any()
    for screen in (2, 0):
        got, info = _detect(problem, screen)
        assert info["screen_active"] == float(screen)
        assert diff_results(got, ref) == [], screen
        assert info["positives"] == D.count_positives(cfg, model, frames)


def _map_problem(name, conn):
    b, s = D.TAIL_MAPS[name]
    bottom, side = D.maps_to_boxes(b[None], s[None])
    return D.make_problem(bottom, side, D.unit_model(), conn=conn), b, s


@pytest.mark.parametrize("conn", [4, 8])
def test_tail_maps_fast_and_slow_path_equal_oracle(oracle, conn, monkeypatch):
    """Every designed tail map on the shared-memory path with the run capacity exactly at the map's run count, and on the
    global-memory path with one run less: tracks equal oracle.detect and oracle.tail_from_binary bit for bit."""
    from locomouse_cpp_b200.api import Detector

    det = None
    try:
        for name in sorted(D.TAIL_MAPS):
            problem, b, s = _map_problem(name, conn)
            cfg, model, bkg, calib, frames, bx, bs, bb = problem
            ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb)
            tracks, mask = oracle.tail_from_binary(b, s, conn, cfg.n_tail_points)
            assert np.array_equal(ref.tail[0], tracks), name
            gate = mask.max(axis=0) != 0
            runs = max(D.run_count(b), D.run_count((s != 0) & gate[None, :]))
            if det is None:
                det = Detector(cfg, model, bkg, calib, device=0)
            for cap in (runs, runs - 1):
                if cap < 0:
                    continue
                monkeypatch.setenv("LM_TAIL_RUNCAP", str(cap))
                got = det.detect_batch(frames, bx, bs, bb)
                assert det.info("screen_active") == 2.0
                assert diff_results(got, ref) == [], (name, cap)
                assert np.array_equal(got.tail[0], tracks), (name, cap)
    finally:
        if det is not None:
            det.close()


@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("screen", [2, 0])
def test_tail_mask_and_q6_in_the_pipeline(oracle, conn, screen):
    """Bottom paw positives inside the tie winner and inside the region that lost the tie (the winner differs between 4- and
    8-connectivity), inside a clear winner, on its border, diagonally next to it and beyond tail_w: the candidate lists
    equal the oracle's (a wrong winner or a mask off by one changes which survive).  A frame without bottom paw positives
    keeps the side paw list empty (Q6) although its side view has positives."""
    problem, _ = D.tail_mask_problem(conn)
    cfg, model, bkg, calib, frames, bx, bs, bb = problem
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb)
    assert ref.n_bottom[2, PAW] == 0 and ref.n_side[2, PAW] == 0 and ref.n_side[0, PAW] > 0
    got, info = _detect(problem, screen)
    assert info["screen_active"] == float(screen)
    assert diff_results(got, ref) == []
    assert got.n_side[2, PAW] == 0


@pytest.mark.parametrize("fma_mode", [True, False])
def test_scores_exactly_zero_smallest_positive_and_negative_zero(oracle, fma_mode):
    """A designed output scoring exactly +0.0 (not a detection), the smallest positive value it can reach (a detection), and
    -0.0 (not a detection): every screen mode equals the oracle and counts the same positive outputs."""
    for name, (problem, _) in D.zero_score_problems(fma_mode).items():
        cfg, model, bkg, calib, frames, bx, bs, bb = problem
        ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb)
        n_pos = D.count_positives(cfg, model, frames)
        for screen in (2, 1, 0):
            got, info = _detect(problem, screen)
            assert info["screen_active"] == float(screen), (name, screen)
            assert diff_results(got, ref) == [], (name, screen)
            assert info["positives"] == n_pos, (name, screen)


def test_bounding_box_base_on_thickened_tie_maps(oracle, monkeypatch):
    """Pass 1 of the base class labels with the same run-based component code (cc_runs.cuh): the tie maps, three pixels
    thick, through a 3 x 3 median, on the shared-memory path with the run capacity at the larger view's run count and on
    the global-memory path with one run less, under both connectivities.  Box and limits equal the oracle."""
    import dataclasses

    from locomouse_cpp_b200.api import Detector

    (cfg, model, bkg, calib, frames, params), med_b, med_s = D.bbox_tie_problem()
    runs = max(max(D.run_count(m) for m in med_b), max(D.run_count(m) for m in med_s))
    for conn in (4, 8):
        c = dataclasses.replace(cfg, conn=conn)
        want, wl = oracle.bounding_box_base(c, bkg, calib, frames, params)
        det = Detector(c, model, bkg, calib, device=0)
        try:
            for cap in (runs, runs - 1):
                monkeypatch.setenv("LM_BBOX_RUNCAP", str(cap))
                got, gl = det.bounding_box_base(frames, params)
                assert np.array_equal(gl, wl) and np.array_equal(got, want), (conn, cap)
        finally:
            det.close()
