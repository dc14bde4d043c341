"""Designed inputs for the pre-processing stage (k_minmax -> k_lut -> k_fold_calib -> k_prep, csrc/k_pre.cu) and the pass-1
front ends that share its table and gather (k_bb_hist16 / k_bb_hist / k_bb_pred, csrc/k_bbox.cu): calibration maps that reach
every gather tier, a Python restatement of the tier choice to prove it, and a window check against the oracle.

Synthetic videos only ever use the identity map or a smooth sine warp, and a wrong window pixel is seen through the final
candidates only when it lies under a positive, unmasked score.  The checks here compare the pre-processed windows and the
per-frame min / max themselves, bit for bit.  Test infrastructure: imported by tests/ and tests/dev_gpu_check.py."""
from __future__ import annotations

import numpy as np

from locomouse_cpp_b200 import synth
from locomouse_cpp_b200.types import Config, Model

CHUNK = 64          # frames per detect_batch call in stage_check: a call of <= 64 frames stays one sub-batch
BIG_RHO = 1.0e4     # no score of a designed frame gets near it: the back phase has nothing to do


# ---- geometry -------------------------------------------------------------------------------------------------------
# Template shapes per view [paw, snout, tail] of mixed sizes: the halos of a window come from different templates.
TSHAPES = (((7, 9), (5, 11), (9, 5)), ((5, 7), (7, 5), (3, 13)))


def small_geometry(odd: bool, vid_pad: int = 1, side_h: int = 28, flip: bool = False, imadjust: bool = True):
    """(cfg, model) of a small problem: 62 x 298 calibrated in a 64 x 300 raw frame (19 200 bytes, a multiple of 16) or
    61 x 301 in 63 x 303 (19 089 bytes: odd rows and columns, a tail behind the last 16-byte vector)."""
    n_rows, n_cols = (61, 301) if odd else (62, 298)
    cfg = Config(vid_rows=n_rows + 2 * vid_pad, vid_cols=n_cols + 2 * vid_pad, n_rows=n_rows, n_cols=n_cols, bb_w=100,
                 bb_h_bottom=n_rows - side_h, bb_h_side=24, flip=flip, imadjust=imadjust, cand_cap=64, det_cap=8192, match_cap=256)
    spec = synth.SynthSpec(tshapes=TSHAPES)
    model = synth.make_model(spec, rho=[[BIG_RHO] * 3 for _ in range(2)])
    return cfg, model


def window_dims(model: Model, view: int):
    """(halo_x, halo_y, extra_x, extra_y) of a view's window: the largest template half-widths before and after the anchor
    over all three templates of the view, as the correlation stages read them."""
    hx = hy = px = py = 0
    for w in model.w[view]:
        kh, kw = w.shape
        hx, hy = max(hx, kw // 2), max(hy, kh // 2)
        px, py = max(px, kw - 1 - kw // 2), max(py, kh - 1 - kh // 2)
    return hx, hy, px, py


def window_origin(cfg: Config, model: Model, view: int, bb_x: int, ypos: int):
    hx, hy, px, py = window_dims(model, view)
    box_h = cfg.bb_h_bottom if view == 0 else cfg.bb_h_side
    return int(bb_x) - cfg.bb_w + 1 - hx, int(ypos) - box_h + 1 - hy, cfg.bb_w + hx + px, box_h + hy + py


def expected_window(I, x0, y0, H, P, win_w):
    """The oracle image cropped at (x0, y0), H x P, zero outside the image and right of win_w (the pitch padding)."""
    n_rows, n_cols = I.shape
    exp = np.zeros((H, P), np.uint8)
    ys, xs = np.arange(y0, y0 + H), np.arange(x0, x0 + P)
    yv, xv = (ys >= 0) & (ys < n_rows), (xs >= 0) & (xs < n_cols)
    exp[np.ix_(yv, xv)] = I[np.ix_(ys[yv], xs[xv])]
    exp[:, win_w:] = 0
    return exp


def stage_check(det, cfg: Config, bkg, calib, frames, bx, bs, bb, prev=None, first_frame_index=None, oracle_images=None):
    """Runs det.detect_batch on device-resident frames in chunks of at most CHUNK frames and asserts, for every frame, that
    the min / max of max(F - BKG, 0) and both pre-processed windows (pitch padding included) equal the oracle's.
    frames: uint8 numpy [n, vid_rows, vid_cols] or a CUDA tensor.  prev: the raw frame before frames[0] (the halo frame)
    or None.  oracle_images: optional list of (I, mm) per frame, computed here otherwise.  Returns the number of frames."""
    import torch

    from oracle import oracle

    if isinstance(frames, torch.Tensor):
        dev_frames = frames
        host = frames.cpu().numpy()
    else:
        host = np.ascontiguousarray(frames)
        dev_frames = torch.from_numpy(host).cuda(det.device)
    n = host.shape[0]
    bx, bs, bb = (np.ascontiguousarray(a, np.uint32) for a in (bx, bs, bb))
    model = det.model
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        if c0 == 0:
            pf = prev
            ffi = first_frame_index if first_frame_index is not None else (1 if prev is not None else 0)
        else:
            pf, ffi = dev_frames[c0 - 1], c0 + (first_frame_index or 0)
        if pf is not None and not isinstance(pf, torch.Tensor):
            pf = torch.from_numpy(np.ascontiguousarray(pf)).cuda(det.device)
        det.detect_batch(dev_frames[c0:c1], bx[c0:c1], bs[c0:c1], bb[c0:c1], prev_frame=pf, first_frame_index=ffi,
                         allow_overflow=True)
        for f in range(c0, c1):
            I, mm = oracle_images[f] if oracle_images is not None else oracle.preprocess(cfg, bkg, calib, host[f])
            gmm, _ = det.debug_fetch(3, f - c0)
            assert np.array_equal(gmm, mm), f"frame {f}: min/max {gmm.tolist()} != oracle {mm.tolist()}"
            for v, ypos in ((0, bb[f]), (1, bs[f])):
                win, dims = det.debug_fetch(v, f - c0)
                x0, y0, win_w, _ = window_origin(cfg, model, v, bx[f], ypos)
                hx, hy = window_dims(model, v)[:2]
                assert (int(dims[2]), int(dims[3])) == (hy, hx), f"halo {dims[2:].tolist()} != {(hy, hx)}"
                exp = expected_window(I, x0, y0, win.shape[0], win.shape[1], win_w)
                if not np.array_equal(win, exp):
                    bad = np.argwhere(win != exp)
                    r, c = bad[0]
                    raise AssertionError(f"frame {f} view {v} (x0={x0}, y0={y0}): {len(bad)} window pixels differ, first at "
                                         f"({r}, {c}): device {win[r, c]} oracle {exp[r, c]}")
    return n


# ---- inputs ---------------------------------------------------------------------------------------------------------
def background(cfg: Config, seed: int = 5):
    """Random background in 40 .. 200: frames drawn around it are above it in some bytes of a word and below in others."""
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(40, 201, (cfg.vid_rows, cfg.vid_cols), dtype=np.uint8)


def frames_around(bkg, n: int, seed: int = 6):
    """n frames = background + noise of a per-frame spread (some bytes below the background, some far above)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = np.empty((n,) + bkg.shape, np.uint8)
    for f in range(n):
        lo, hi = int(rng.integers(-60, -1)), int(rng.integers(20, 120))
        out[f] = np.clip(bkg.astype(np.int32) + rng.integers(lo, hi, bkg.shape), 0, 255).astype(np.uint8)
    return out


# ---- designed calibration maps --------------------------------------------------------------------------------------
def _raw_index(cfg: Config, r, c, pad: int):
    return ((np.asarray(r) + pad) * cfg.vid_cols + np.asarray(c) + pad).astype(np.int64)


def map_identity(cfg: Config, pad: int | None = None):
    pad = (cfg.vid_rows - cfg.n_rows) // 2 if pad is None else pad
    r, c = np.mgrid[0:cfg.n_rows, 0:cfg.n_cols]
    return _raw_index(cfg, r, c, pad).astype(np.int32)


def map_reversed(cfg: Config):
    """The identity reversed in every row: descending runs (ascending again once a mirror is folded in)."""
    return np.ascontiguousarray(map_identity(cfg)[:, ::-1])


def map_runs(cfg: Config, descending: bool, seed: int = 11):
    """Rows cut into runs of 1 .. 20 consecutive raw bytes at random starts, so that run breaks fall at every column
    offset mod 16; descending runs read their raw bytes backwards."""
    rng = np.random.Generator(np.random.PCG64(seed))
    nraw = cfg.vid_rows * cfg.vid_cols
    out = np.empty((cfg.n_rows, cfg.n_cols), np.int64)
    for r in range(cfg.n_rows):
        c = 0
        while c < cfg.n_cols:
            L = min(int(rng.integers(1, 21)), cfg.n_cols - c)
            start = int(rng.integers(L, nraw - L))
            q = np.arange(L)
            out[r, c:c + L] = start - q if descending else start + q
            c += L
    return out.astype(np.int32)


def map_resample(cfg: Config, up: bool):
    """Repeated indices (up-sampling: each raw column twice) or skipped ones (down-sampling: every other raw column)."""
    pad = (cfg.vid_rows - cfg.n_rows) // 2
    r, c = np.mgrid[0:cfg.n_rows, 0:cfg.n_cols]
    src = c // 2 if up else np.minimum(2 * c, cfg.vid_cols - 1 - pad)
    return _raw_index(cfg, r, src, pad).astype(np.int32)


def map_row_wrap(cfg: Config):
    """Every calibrated row is the continuation of the raw bytes of the row before: runs cross each calibrated row end."""
    n = cfg.n_rows * cfg.n_cols
    off = (cfg.vid_rows * cfg.vid_cols - n) // 2
    return (off + np.arange(n)).reshape(cfg.n_rows, cfg.n_cols).astype(np.int32)


def map_frame_ends(cfg: Config, seed: int = 12):
    """Runs of 3 .. 20 routed to the first 24 and the last 24 raw bytes of the frame (the bounds tests of the word loads)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    nraw = cfg.vid_rows * cfg.vid_cols
    out = np.empty((cfg.n_rows, cfg.n_cols), np.int64)
    for r in range(cfg.n_rows):
        c = 0
        while c < cfg.n_cols:
            L = min(int(rng.integers(3, 21)), cfg.n_cols - c)
            desc = bool(rng.integers(0, 2))
            if rng.integers(0, 2):
                start = int(rng.integers(0, 24 - L + 1)) if L <= 24 else 0
            else:
                start = nraw - L - int(rng.integers(0, max(1, 24 - L + 1)))
            q = np.arange(L)
            out[r, c:c + L] = start + (L - 1 - q if desc else q)
            c += L
    return out.astype(np.int32)


def map_permutation(cfg: Config, seed: int = 13):
    """A random injection into the raw frame: no two neighbours are consecutive, every word is a gather."""
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.permutation(cfg.vid_rows * cfg.vid_cols)[:cfg.n_rows * cfg.n_cols].reshape(cfg.n_rows, cfg.n_cols).astype(np.int32)


def map_defects(cfg: Config, kind: str, seed: int = 14):
    """The identity with defects a real calibration shows; the picture survives, so a mouse still yields candidates.
    kind: 'shift' (periodic +-1 row shifts of 37-column stretches), 'dup' (a duplicated column every 23), 'drop' (a dropped
    column every 19), 'rev' (reversed 5-pixel segments every 29 columns), 'all' (all four)."""
    pad = (cfg.vid_rows - cfg.n_rows) // 2
    r, c = np.mgrid[0:cfg.n_rows, 0:cfg.n_cols]
    rr, cc = r.copy(), c.copy()
    if kind in ("shift", "all"):
        rr = rr + ((c // 37) % 3 - 1)
    if kind in ("dup", "all"):
        cc = cc - (cc // 23)
    if kind in ("drop", "all"):
        cc = cc + (cc // 19)
    if kind in ("rev", "all"):
        seg = (c % 29) < 5
        cc = np.where(seg, cc - (c % 29) + (4 - (c % 29)), cc)
    rr = np.clip(rr + pad, 0, cfg.vid_rows - 1)
    cc = np.clip(cc + pad, 0, cfg.vid_cols - 1)
    return (rr * cfg.vid_cols + cc).astype(np.int32)


def design_maps(cfg: Config):
    """name -> map for the whole design set (every map indexes inside the raw frame)."""
    return {
        "identity": map_identity(cfg),
        "identity_pad0": map_identity(cfg, pad=0),
        "reversed": map_reversed(cfg),
        "runs_asc": map_runs(cfg, False),
        "runs_desc": map_runs(cfg, True),
        "upsample": map_resample(cfg, True),
        "downsample": map_resample(cfg, False),
        "row_wrap": map_row_wrap(cfg),
        "frame_ends": map_frame_ends(cfg),
        "permutation": map_permutation(cfg),
        "defects_all": map_defects(cfg, "all"),
    }


# ---- the tier choice of k_fold_calib / k_prep / k_bb_hist16, restated --------------------------------------------------
def run_mode(calib, flip: bool):
    """(calib_flip, run_mode) as k_fold_calib builds them: bit 0 / 1 = the 4 pixels from column c on come from consecutive
    ascending / descending raw bytes, bit 2 / 3 = the same for 16 pixels (runs stop at the calibrated row end)."""
    cf = np.ascontiguousarray(np.asarray(calib, np.int64)[:, ::-1] if flip else np.asarray(calib, np.int64))
    rows, cols = cf.shape
    up_ok = np.ones((rows, cols), bool)
    dn_ok = np.ones((rows, cols), bool)
    mode = np.zeros((rows, cols), np.uint8)
    for q in range(1, 16):
        nxt = np.full((rows, cols), -(1 << 40), np.int64)
        nxt[:, :cols - q] = cf[:, q:]
        up_ok &= nxt == cf + q
        dn_ok &= nxt == cf - q
        if q == 3:
            mode |= up_ok.astype(np.uint8) | (dn_ok.astype(np.uint8) << 1)
    mode |= (up_ok.astype(np.uint8) << 2) | (dn_ok.astype(np.uint8) << 3)
    return cf, mode


TIERS = ("t1_asc", "t1_desc", "t1_lo_fallback", "t1_hi_fallback", "t2_run_asc", "t2_run_desc", "t2_run_fallback", "t2_gather",
         "t3_border")


def tier_counts(cfg: Config, calib, boxes, fbytes: int):
    """Counts of the paths k_prep takes for the given windows.  boxes: iterable of (x0, y0, win_w, win_h) in calibrated image
    coordinates.  Tier 1 and its bounds fall-backs count 16-pixel segments (t1_lo_fallback: lo_i < 4, t1_hi_fallback:
    lo_i + 24 > fbytes); tiers 2 and 3 count 4-pixel words."""
    cf, mode = run_mode(calib, cfg.flip)
    n = dict.fromkeys(TIERS, 0)
    for x0, y0, win_w, win_h in boxes:
        for r in range(win_h):
            yy = y0 + r
            if yy < 0 or yy >= cfg.n_rows:
                continue
            for c16 in range(0, win_w, 16):
                xx0 = x0 + c16
                if xx0 + 16 <= 0 or xx0 >= cfg.n_cols:
                    continue
                if xx0 >= 0 and xx0 + 16 <= cfg.n_cols and mode[yy, xx0] & 12:
                    lo_i = int(cf[yy, xx0]) if mode[yy, xx0] & 4 else int(cf[yy, xx0]) - 15
                    if lo_i < 4:
                        n["t1_lo_fallback"] += 1
                    elif lo_i + 24 > fbytes:
                        n["t1_hi_fallback"] += 1
                    else:
                        n["t1_asc" if mode[yy, xx0] & 4 else "t1_desc"] += 1
                        continue
                for w in range(4):
                    c4, xw = c16 + 4 * w, xx0 + 4 * w
                    if c4 >= win_w:
                        break
                    if xw >= 0 and xw + 4 <= cfg.n_cols:
                        m = int(mode[yy, xw]) & 3
                        lo_i = int(cf[yy, xw]) - 3 if m == 2 else int(cf[yy, xw])
                        if m and 4 <= lo_i and lo_i + 8 <= fbytes:
                            n["t2_run_asc" if m == 1 else "t2_run_desc"] += 1
                        else:
                            n["t2_run_fallback" if m else "t2_gather"] += 1
                    else:
                        n["t3_border"] += 1
    return n


HIST16 = ("h_asc", "h_desc", "h_lo_fallback", "h_hi_fallback", "h_gather_full", "h_gather_partial")


def hist16_counts(cfg: Config, calib, side_x: int, side_y: int, side_w: int, side_h: int, fbytes: int):
    """Counts of the 16-pixel items of k_bb_hist16 over a side view, per path (h_gather_partial: the item at the row end
    holds fewer than 16 pixels)."""
    cf, mode = run_mode(calib, cfg.flip)
    n = dict.fromkeys(HIST16, 0)
    for r in range(side_h):
        for c16 in range(0, side_w, 16):
            if side_w - c16 < 16:
                n["h_gather_partial"] += 1
                continue
            yy, xx = side_y + r, side_x + c16
            m = int(mode[yy, xx])
            if m & 12:
                lo_i = int(cf[yy, xx]) if m & 4 else int(cf[yy, xx]) - 15
                if lo_i < 4:
                    n["h_lo_fallback"] += 1
                elif lo_i + 24 > fbytes:
                    n["h_hi_fallback"] += 1
                else:
                    n["h_asc" if m & 4 else "h_desc"] += 1
            else:
                n["h_gather_full"] += 1
    return n


# ---- box placement ------------------------------------------------------------------------------------------------
def placements(cfg: Config, model: Model, sweep: int = 18):
    """(bb_x, bb_y_side, bb_y_bottom) triples whose windows sit inside the image, straddle each of its four borders
    (the window edge swept over `sweep` columns / rows around the border) and sit in the top-left and bottom-right
    corners.  Every triple passes the oracle's ROI check."""
    from oracle import oracle

    hxb, hyb, pxb, pyb = window_dims(model, 0)
    hxs, hys, pxs, pys = window_dims(model, 1)
    hx, px = max(hxb, hxs), max(pxb, pxs)
    win_w = cfg.bb_w + hx + px
    # bb_x for a window whose left edge is at x0: x0 = bb_x - bb_w + 1 - hx
    xs_left = [cfg.bb_w - 1 + hx + x0 for x0 in range(-sweep // 2, sweep // 2 + 1)]
    xs_right = [cfg.bb_w - 1 + hx + x0 for x0 in range(cfg.n_cols - win_w - sweep // 2, cfg.n_cols - win_w + sweep // 2 + 1)]
    xs_mid = [(cfg.n_cols + cfg.bb_w) // 2 + k for k in range(4)]

    def ys(hy, py, box_h):
        top = [box_h - 1 + hy + y0 for y0 in range(-3, 4)]                   # window top edge around row 0
        h = box_h + hy + py
        bot = [box_h - 1 + hy + y0 for y0 in range(cfg.n_rows - h - 3, cfg.n_rows - h + 4)]
        return top, bot

    tops, bots = ys(hys, pys, cfg.bb_h_side)
    topb, botb = ys(hyb, pyb, cfg.bb_h_bottom)
    mid_s, mid_b = cfg.bb_h_side + 2, cfg.n_rows - 3
    out = []
    for i, x in enumerate(xs_left + xs_mid + xs_right):
        out.append((x, mid_s, mid_b))
        out.append((x, tops[i % len(tops)], botb[i % len(botb)]))
        out.append((x, bots[i % len(bots)], topb[i % len(topb)]))
    for i, x in enumerate(xs_left):                                           # top-left corner
        out.append((x, tops[i % len(tops)], topb[i % len(topb)]))
    for i, x in enumerate(xs_right):                                          # bottom-right corner
        out.append((x, bots[i % len(bots)], botb[i % len(botb)]))
    ok = [t for t in out if t[0] >= 0 and t[1] >= 0 and t[2] >= 0 and oracle.check_roi(cfg, model, *t) == 0]
    return np.array(ok, np.int64)


def boxes_of(cfg: Config, model: Model, places):
    """The (x0, y0, win_w, win_h) windows of both views for each placement (what tier_counts takes)."""
    out = []
    for bx, bs, bb in places:
        for v, ypos in ((0, bb), (1, bs)):
            x0, y0, win_w, h = window_origin(cfg, model, v, bx, ypos)
            out.append((x0, y0, win_w, (h + 3) & ~3))
    return out


# ---- pass 1 of LocoMouse_TM_DE on the designed maps --------------------------------------------------------------------
def de_frames(cfg: Config, bkg, n: int = 6, seed: int = 43):
    """Frames for LocoMouse_TM_DE's pass 1: at or just above the background (differences 0 .. 3, counted in k_bb_hist16's
    registers) with a sparse bright body of varying size moving along the side view, so that imadjust_default stretches the
    body, not the noise, and the first / last qualifying columns follow the body through the calibration map."""
    rng = np.random.Generator(np.random.PCG64(seed))
    B = bkg.astype(np.int32)
    fr = np.empty((n,) + bkg.shape, np.int32)
    for f in range(n):
        fr[f] = B + rng.integers(-20, 4, bkg.shape)
        x, h, w = 25 + f * (cfg.vid_cols - 90) // n, 6 + 2 * (f % 3), 30 + 4 * f
        fr[f, 12:12 + h, x:x + w] = B[12:12 + h, x:x + w] + rng.integers(60, 120, (h, w))
    return np.clip(fr, 0, 255).astype(np.uint8)


def de_params(cfg: Config, side_h: int = 28):
    """The side view inset by 3 columns (its width is odd in one of the two geometries: k_bb_hist16 then stores the kept
    differences of alternate rows byte by byte), bands inside it."""
    from locomouse_cpp_b200.types import bb_de_params

    return bb_de_params(cfg, side_h=side_h, side_x=3, side_w=cfg.n_cols - 3, zero_col_pre=5, zero_col_post=cfg.n_cols - 12,
                        zero_row_pre=2, zero_row_post=25, threshold=255 * 0.05, min_count=3)


def assert_de_input_sees_the_map(oracle, cfg: Config, bkg, frames, p):
    """The oracle's pass-1 limits on `frames` follow the body (a different first column in every frame, both limits inside
    the bands) and change when the identity map is replaced by every other designed map: a gather through the wrong pixels
    cannot give the same answer."""
    maps = design_maps(cfg)
    lims = oracle.bounding_box_tm_de(cfg, bkg, maps["identity"], frames, p)[2]
    assert np.unique(lims[:, 0]).size == len(frames), lims
    assert (lims[:, 0] > p.zero_col_pre).all() and (lims[:, 1] < p.zero_col_post - 1).all(), lims
    for name, m in maps.items():
        if name != "identity":
            assert not np.array_equal(oracle.bounding_box_tm_de(cfg, bkg, m, frames, p)[2], lims), name


# ---- imadjust_default boundaries (k_bb_pred) --------------------------------------------------------------------------
# A side view W wide, H high at the top of a zero-background, identity-calibrated image.  Row 0 is the only row that survives
# the zeroed bands; its column x holds the difference x mod 256, so with min_count 1 the first qualifying column is the first
# difference d whose stretched value passes the threshold.  Rows 1 .. H - 1 lie in the zeroed band: they shape the histogram
# (k_bb_hist16 counts every side-view pixel) without reaching the column sums.  Row 0 holds 0 and 255, so the normalisation
# is the identity and the histogram bins are the differences themselves.
#   name -> (W, H, {bin: count} in the band, filler bin for the rest of the band, alternative: (from_bin, to_bin) moving one
#   count that shifts the boundary index by one, the (i0, i1) imadjust_default must find)
# The floats next to 0.01f need large side views: with sum s and cumsum c both exact below 2^24, c / s rounds to a
# neighbour of 0.01f only when s is in the millions (about 6.2e6 for the lower one); the two views below are 6.2 M and 8.5 M.
def _row0_cum(W: int, b: int) -> int:
    """Pixels of row 0 (column x holds x mod 256) in bins 0 .. b."""
    return int(((np.arange(W) % 256) <= b).sum())


IMADJUST_DESIGNS = {
    "min_at_0.01f": (256, 25, {20: 43}, 200, (21, 20), (21, 200)),               # cumsum / sum == 0.01f at bin 20: not > 0.01f
    "min_below_0.01f": (1971, 3131, {20: 61712 - _row0_cum(1971, 20)}, 200, (21, 20), (21, 200)),   # the float below 0.01f
    "min_above_0.01f": (2591, 3289, {20: 85218 - _row0_cum(2591, 20)}, 200, (20, 21), (20, 200)),   # the float above 0.01f
    "max_at_0.99f": (256, 25, {10: 6105}, 250, (10, 231), (10, 230)),            # == 0.99f at bin 230: >= 0.99f
    "max_below_0.99f": (257, 507, {10: 128996 - 232}, 250, (250, 230), (10, 231)),   # the float below 0.99f at bin 230
    "max_above_0.99f": (257, 493, {10: 125434 - 232}, 250, (10, 231), (10, 230)),   # the float above 0.99f at bin 230
    "i0_eq_i1": (256, 100, {}, 128, None, (128, 256)),                          # one bin jumps from < 1 % to > 99 %
    "alpha_one": (256, 25, {0: 3000}, 255, None, (0, 255)),                      # i0 = 0, i1 = 255: the identity copy
    "one_bin": (256, 25, {}, 90, None, (90, 256)),                               # every side-view pixel in bin 90
}


def imadjust_shape(name: str):
    """(vid_rows, vid_cols) of the identity-calibrated frame that holds a design's side view."""
    W, H = IMADJUST_DESIGNS[name][:2]
    return H + 2, max(W, 300)


def imadjust_frame(name: str, vid_rows: int, vid_cols: int):
    """(frame uint8 [vid_rows, vid_cols], histogram uint32[256] of the side view) of a design."""
    W, H, band, filler, _, _ = IMADJUST_DESIGNS[name]
    fr = np.zeros((vid_rows, vid_cols), np.uint8)
    if name == "one_bin":
        fr[:H, :W] = filler
        fr[H + 1, 0], fr[H + 1, 1] = 0, 255            # min and max outside the side view
    else:
        fr[0, :W] = np.arange(W) % 256
        vals = np.concatenate([np.full(c, b, np.uint8) for b, c in band.items()] +
                              [np.full((H - 1) * W - sum(band.values()), filler, np.uint8)])
        fr[1:H, :W] = vals.reshape(H - 1, W)
    hist = np.bincount(fr[:H, :W].reshape(-1), minlength=256).astype(np.uint32)
    return fr, hist


def imadjust_threshold(oracle, name: str):
    """A threshold at which the first passing difference of the design's stretched table differs from that of the table
    with the boundary index moved by one (None for designs without an alternative), and that first difference."""
    _, hist = imadjust_frame(name, *imadjust_shape(name))
    alt = IMADJUST_DESIGNS[name][4]
    lut, _ = oracle.imadjust_default_lut(hist)
    if alt is None:
        return None, None
    h2 = hist.copy()
    h2[alt[0]] -= 1
    h2[alt[1]] += 1
    lut2, _ = oracle.imadjust_default_lut(h2)
    d = int(np.argmax(lut != lut2))
    assert lut[d] != lut2[d]
    th = min(int(lut[d]), int(lut2[d])) + 0.5
    first = lambda t: int(np.argmax(t > th)) if (t > th).any() else -1  # noqa: E731
    assert first(lut) != first(lut2)
    return th, first(lut)
