"""Pre-processing stage by stage on the device against the oracle, bit for bit: k_minmax's per-frame min / max, k_lut's
normalisation table for every (min, max) pair, k_prep's windows through designed calibration maps that reach every gather
tier, the folded per-video arrays after the map, background or mirror change, detection and pairing on maps with defects,
and the pass-1 front ends (k_bb_hist16 / k_bb_hist / k_bb_pred, k_bbtm_bin, k_bbb_bin) on the same maps.  The designs and
the window check live in tests/_preprocess_designs.py.  Needs a B200: pytest -m gpu."""
import dataclasses

import numpy as np
import pytest

from locomouse_cpp_b200.types import Config, bb_base_params, bb_de_params, bb_tm_params, diff_results

import _preprocess_designs as D

pytestmark = pytest.mark.gpu


def _detector(cfg, model, bkg, calib):
    from locomouse_cpp_b200.api import Detector

    return Detector(cfg, model, bkg, calib, device=0)


def _disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    h = ((x * x + y * y) <= (r + 0.5) ** 2).astype(np.float64)
    return (h / h.sum()).astype(np.float32)


# ---- 1. every normalisation table ----------------------------------------------------------------------------------
@pytest.mark.parametrize("imadjust", [False, True])
def test_every_normalisation_table(oracle, imadjust):
    """One frame per (min, max) pair, 0 <= min <= max <= 255, zero background, identity map: the frame holds every value
    min .. max in a pattern whose window shows them all, so every entry of every table reaches a window pixel."""
    import torch

    cfg, model = D.small_geometry(False, vid_pad=1, imadjust=imadjust)
    bkg = np.zeros((cfg.vid_rows, cfg.vid_cols), np.uint8)
    calib = D.map_identity(cfg)
    det = _detector(cfg, model, bkg, calib)
    pairs = np.array([(a, b) for a in range(256) for b in range(a, 256)], np.int32)
    x0, y0, win_w, _ = D.window_origin(cfg, model, 0, 150, cfg.n_rows - 1)
    r, c = np.mgrid[0:cfg.vid_rows, 0:cfg.vid_cols]
    pos = r * win_w + c - x0                               # consecutive along the window's rows, row after row
    bx, bs, bb = np.full(D.CHUNK, 150), np.full(D.CHUNK, cfg.bb_h_side + 2), np.full(D.CHUNK, cfg.n_rows - 1)
    nmm = set()
    for k in range(0, len(pairs), D.CHUNK):
        p = pairs[k:k + D.CHUNK]
        m = (p[:, 1] - p[:, 0] + 1)[:, None, None]
        frames = (p[:, 0][:, None, None] + pos[None] % m).astype(np.uint8)
        dev = torch.from_numpy(frames).cuda()
        n = len(p)
        D.stage_check(det, cfg, bkg, calib, dev, bx[:n], bs[:n], bb[:n])
        nmm.update(map(tuple, p.tolist()))
    assert len(nmm) == 32896
    det.close()


# ---- 2. k_minmax seams ---------------------------------------------------------------------------------------------
def _seam_frames(cfg, bkg, seed=21):
    """(prev frame, frames, names): each frame has its extreme difference at one seam of k_minmax."""
    rng = np.random.Generator(np.random.PCG64(seed))
    fb = cfg.vid_rows * cfg.vid_cols
    B = bkg.reshape(-1).astype(np.int32)

    def base():
        return np.clip(B + rng.integers(10, 51, fb), 0, 255)            # d in 10 .. 50 (the background is at most 200)

    seams = {"first_byte": 0, "last_byte": fb - 1, "cta_end": 16383, "cta_start": 16384, "last_vector": fb - (fb % 16) - 1,
             "tail": fb - (fb % 16) if fb % 16 else fb - 2, "tail_end": fb - 1 - (fb % 16) // 2,
             "border_top": 1, "border_left": cfg.vid_cols, "border_bottom": fb - 3}
    frames, names = [], []
    for name, p in seams.items():
        for kind in ("max", "min", "zero"):
            f = base()
            f[p] = B[p] + 55 if kind == "max" else (B[p] + 3 if kind == "min" else max(B[p] - 7, 0))
            frames.append(f)
            names.append(f"{name}/{kind}")
    frames.append(np.clip(B - rng.integers(0, 40, fb), 0, 255))                         # F <= BKG everywhere
    names.append("all_below")
    frames.append(base())                                                               # the halo frame's extremes are its own
    names.append("after_halo")
    prev = base()
    prev[0], prev[fb - 1], prev[fb // 2] = 255, max(B[fb - 1] - 9, 0), B[fb // 2] + 2
    shape = (cfg.vid_rows, cfg.vid_cols)
    return prev.astype(np.uint8).reshape(shape), np.stack(frames).astype(np.uint8).reshape((-1,) + shape), names


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("offset", [0, 1, 4, 15])
def test_minmax_seams(oracle, odd, offset):
    """The extreme pixel at the first / last byte, at both sides of a CTA's 16 kB range, behind the last 16-byte vector,
    in the raw border outside the calibrated image, only in the halo frame, and no pixel above the background; frames
    read from a device buffer at byte offsets 0, 1, 4 and 15 (the byte-wise path unless all is 16-byte aligned)."""
    import torch

    cfg, model = D.small_geometry(odd)
    bkg = D.background(cfg)
    calib = D.map_identity(cfg)
    prev, frames, names = _seam_frames(cfg, bkg)
    fb = cfg.vid_rows * cfg.vid_cols
    n = frames.shape[0]
    buf = torch.zeros(offset + (n + 1) * fb + 16, dtype=torch.uint8, device="cuda")
    buf[offset:offset + fb] = torch.from_numpy(prev.reshape(-1)).cuda()
    buf[offset + fb:offset + (n + 1) * fb] = torch.from_numpy(frames.reshape(-1)).cuda()
    dprev = buf[offset:offset + fb].view(cfg.vid_rows, cfg.vid_cols)
    dframes = buf[offset + fb:offset + (n + 1) * fb].view(n, cfg.vid_rows, cfg.vid_cols)
    places = D.placements(cfg, model)
    sel = places[np.linspace(0, len(places) - 1, n).astype(int)]
    det = _detector(cfg, model, bkg, calib)
    D.stage_check(det, cfg, bkg, calib, dframes, sel[:, 0], sel[:, 1], sel[:, 2], prev=dprev, first_frame_index=7)
    mm = [oracle.preprocess(cfg, bkg, calib, f)[1].tolist() for f in frames]
    assert mm[names.index("first_byte/max")][1] == 55 and mm[names.index("cta_start/min")][0] == 3
    assert mm[names.index("all_below")] == [0, 0] and mm[names.index("tail/zero")][0] == 0
    det.close()


# ---- 3. gather tiers -----------------------------------------------------------------------------------------------
def _tier_run(oracle, odd, flip, maps=None, n_distinct=4):
    cfg, model = D.small_geometry(odd, flip=flip)
    bkg = D.background(cfg)
    distinct = D.frames_around(bkg, n_distinct)
    places = D.placements(cfg, model)
    n = len(places)
    frames = distinct[np.arange(n) % n_distinct]
    det = None
    for name, calib in (maps or D.design_maps(cfg)).items():
        imgs = [oracle.preprocess(cfg, bkg, calib, f) for f in distinct]
        if det is None:
            det = _detector(cfg, model, bkg, calib)
        else:
            det.set_calibration(calib)
        D.stage_check(det, cfg, bkg, calib, frames, places[:, 0], places[:, 1], places[:, 2],
                      oracle_images=[imgs[i % n_distinct] for i in range(n)])
    return det


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("flip", [False, True])
def test_gather_tiers(oracle, odd, flip):
    """Every designed map (tests/test_preprocess_designs.py proves that together they reach every tier of k_prep) with
    windows inside the image, straddling each border and in the top-left / bottom-right corners."""
    _tier_run(oracle, odd, flip).close()


def test_gather_tiers_guard_mode(oracle, monkeypatch):
    """The same under LM_GUARD=1: no kernel writes outside its buffers."""
    monkeypatch.setenv("LM_GUARD", "1")
    det = _tier_run(oracle, True, True)
    assert det.info("guard_violations") == 0
    det.close()


# ---- 4. the folded arrays follow changes ------------------------------------------------------------------------------
def test_folded_arrays_follow_changes(oracle):
    """calib_flip, bkg_warp and run_mode are rebuilt after set_calibration, set_background and a configure that toggles the
    mirror: each second call's windows equal the oracle for the new inputs."""
    cfg, model = D.small_geometry(True)
    bkg = D.background(cfg)
    frames = D.frames_around(bkg, 12, seed=31)
    places = D.placements(cfg, model)
    sel = places[np.linspace(0, len(places) - 1, 12).astype(int)]
    args = (frames, sel[:, 0], sel[:, 1], sel[:, 2])
    a, b = D.map_runs(cfg, False), D.map_runs(cfg, True, seed=99)
    det = _detector(cfg, model, bkg, a)
    D.stage_check(det, cfg, bkg, a, *args)
    det.set_calibration(b)
    D.stage_check(det, cfg, bkg, b, *args)
    bkg2 = D.background(cfg, seed=77)
    det.set_background(bkg2)
    D.stage_check(det, cfg, bkg2, b, *args)
    cfg2 = dataclasses.replace(cfg, flip=True)
    det.configure(cfg2, model, bkg2, b)
    D.stage_check(det, cfg2, bkg2, b, *args)
    det.close()


# ---- 5. detection and pairing on designed maps ------------------------------------------------------------------------
def test_detection_and_pairing_on_designed_maps(oracle):
    """The pairing clip of test_gpu_pairing_coverage.py calibrated with identity-with-defects maps, and with the reversed
    map under the mirror: whole results bit-exact for screen 2 and 0 with sub-batches of 16 (k_pair re-derives the previous
    frame through calib_flip / bkg_warp and that frame's table), and the velocity branches reached."""
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.types import Model

    total, start, n = 600, 200, 40
    spec = synth.SynthSpec()
    cfg, model, bkg, _, _, _, _, _ = synth.make_problem(spec, 8, seed=1000)
    frames, bx, bs, bb = synth.make_video(spec, n, 1000, "cpu", bkg, start_frame=start, total=total)
    prev = synth.make_video(spec, 1, 1000, "cpu", bkg, start_frame=start - 1, total=total)[0][0].numpy()
    frames = frames.numpy()
    model = Model(w=model.w, rho=list(model.rho))
    cases = [(k, cfg, D.map_defects(cfg, k)) for k in ("shift", "dup", "rev", "all")]
    cases.append(("reversed_flip", dataclasses.replace(cfg, flip=True), D.map_reversed(cfg)))
    oracle.coverage(reset=True)
    for name, c, calib in cases:
        ref = oracle.detect(c, model, bkg, calib, frames, bx, bs, bb, prev_frame=prev, first_frame_index=start, n_threads=8)
        assert ref.n_bottom.sum() > 0 and ref.n_side.sum() > 0, name
        for screen in (2, 0):
            det = _detector(c, model, bkg, calib)
            det.set_option("screen", screen)
            det.set_option("subbatch", 16)
            got = det.detect_batch(frames, bx, bs, bb, prev_frame=prev, first_frame_index=start)
            det.close()
            assert diff_results(got, ref) == [], (name, screen)
    cov = oracle.coverage()
    print(f"pairing coverage over the designed maps: {cov}")
    assert cov["velocity_rejections"] > 0 and cov["velocity_accepts"] > 0, cov


# ---- 6. pass 1 on the same maps ---------------------------------------------------------------------------------------
def _pass1_frames(cfg, bkg, n=6, seed=41):
    """Frames around the background with a bright body moving along the side and bottom views."""
    fr = D.frames_around(bkg, n, seed=seed).astype(np.int32)
    for f in range(n):
        x = 20 + f * (cfg.vid_cols - 80) // n
        fr[f, 8:22, x:x + 45] += 90
        fr[f, 36:52, x + 5:x + 50] += 80
    return np.clip(fr, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("flip", [False, True])
def test_pass1_on_designed_maps(oracle, odd, flip):
    """bounding_box_tm_de (k_bb_hist16's tiers and its word / byte stores of the kept differences: the side view is inset
    by 3 columns, so its width is odd in one geometry), bounding_box_tm (k_bbtm_bin) and bounding_box_base (k_bbb_bin) on
    every designed map, from host and device frames: raw positions and limits equal the oracle's."""
    import torch

    side_h = 28
    for imadjust in (True, False):
        cfg, model = D.small_geometry(odd, flip=flip, side_h=side_h, imadjust=imadjust)
        bkg = D.background(cfg)
        frames = _pass1_frames(cfg, bkg)
        dframes = torch.from_numpy(frames).cuda()
        de_frames = D.de_frames(cfg, bkg)
        de_dframes = torch.from_numpy(de_frames).cuda()
        de = D.de_params(cfg)
        tm = bb_tm_params(cfg, _disk(2), side_h=side_h, sums_as_float=0, min_pixel_count=5, zero_col_pre=4,
                          zero_col_post=cfg.n_cols - 9, zero_row_pre=1, zero_row_post=26)
        base = bb_base_params(cfg, side_h=side_h, sums_as_float=0, median_filter_size=5)
        if imadjust:
            D.assert_de_input_sees_the_map(oracle, cfg, bkg, de_frames, de)
        det = None
        for name, calib in D.design_maps(cfg).items():
            if det is None:
                det = _detector(cfg, model, bkg, calib)
            else:
                det.set_calibration(calib)
            if imadjust:
                want = oracle.bounding_box_tm_de(cfg, bkg, calib, de_frames, de)
                for src in (de_frames, de_dframes):
                    got = det.bounding_box_tm_de(src, de)
                    for x, y in zip(got, want):
                        assert np.array_equal(x, y), (name, "tm_de")
                want_tm = oracle.bounding_box_tm(cfg, bkg, calib, frames, tm)
                for src in (frames, dframes):
                    got = det.bounding_box_tm(src, tm)
                    for x, y in zip(got, want_tm):
                        assert np.array_equal(x, y), (name, "tm")
            else:
                want = oracle.bounding_box_base(cfg, bkg, calib, frames, base)
                for src in (frames, dframes):
                    got = det.bounding_box_base(src, base)
                    for x, y in zip(got, want):
                        assert np.array_equal(x, y), (name, "base")
        det.close()


# ---- 7. imadjust_default boundaries -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(D.IMADJUST_DESIGNS) + ["empty_view"])
def test_imadjust_default_boundaries(oracle, name):
    """Side views whose histogram puts cumsum / sum exactly on 0.01f or 0.99f or on the floats next to them, makes
    i0 == i1, alpha == 1, fills one bin, or leaves nothing after the bands are zeroed.  Only row 0 survives the bands and
    its column x holds difference x: the first qualifying column is the first difference k_bb_pred's table passes."""
    import torch

    design = "min_at_0.01f" if name == "empty_view" else name
    W, H = D.IMADJUST_DESIGNS[design][:2]
    rows_, cols_ = D.imadjust_shape(design)
    cfg = Config(vid_rows=rows_, vid_cols=cols_, n_rows=rows_, n_cols=cols_, bb_w=100, bb_h_bottom=30, bb_h_side=24, imadjust=True)
    _, model = D.small_geometry(False)
    frame, hist = D.imadjust_frame(design, cfg.vid_rows, cfg.vid_cols)
    assert oracle.imadjust_default_lut(hist)[1] == D.IMADJUST_DESIGNS[design][5]
    th, first = D.imadjust_threshold(oracle, design)
    bkg = np.zeros_like(frame)
    calib = D.map_identity(cfg)
    rows = (1, 1) if name == "empty_view" else (0, 1)
    p = bb_de_params(cfg, side_h=H, side_w=W, zero_col_pre=0, zero_col_post=W, zero_row_pre=rows[0], zero_row_post=rows[1],
                     threshold=th if th is not None else 255 * 0.05, min_count=1)
    frames = np.stack([frame, frame])
    want = oracle.bounding_box_tm_de(cfg, bkg, calib, frames, p)
    det = _detector(cfg, model, bkg, calib)
    for src in (frames, torch.from_numpy(frames).cuda()):
        got = det.bounding_box_tm_de(src, p)
        for x, y in zip(got, want):
            assert np.array_equal(x, y)
    if name == "empty_view":
        assert want[2][0].tolist() == [-1, -1]
    elif first is not None:
        assert want[2][0][0] == first
    det.close()
