"""Frames whose detector windows are exactly the pixels a test chooses (CPU only).

With method "base" (no imadjust), an all-zero background, the identity calibration and one 0 and one 255 pixel in every
frame, readFrame's min/max normalisation is the identity (scale = float(255 * (1/255)) = 1, shift = 0): every window pixel
equals the frame pixel written here.  `make_problem` checks that with the oracle for every frame it builds.

Layout of the calibrated image (= the raw frame): the side box in rows [0, Hs), the bottom box in rows [Hs, Hs + Hb), both
in columns [MARGIN, MARGIN + W).  Everything outside the boxes is 0 except the 255 marker in the top-right corner, which is
MARGIN columns right of the boxes and so out of reach of every template (cols <= 64).

Also here: a restatement of the screen's quantisation and thresholds (csrc/k_screen.cu screen_quantize, csrc/k_screen2.cu
q_need / q_sign), exact integer scores V and an fp32 emulation of the oracle's tap loop used to pick designs.
"""
from __future__ import annotations

import math

import numpy as np

from locomouse_cpp_b200.types import Config, Model

MARGIN = 48


# ---- the harness --------------------------------------------------------------------------------------------------------
def make_problem(bottom, side, model: Model, conn=8, fma_mode=True, cand_cap=256, det_cap=8192, match_cap=2048,
                 n_tail_points=15, check=True):
    """bottom: uint8 [n, Hb, W] and side: uint8 [n, Hs, W] box images -> (cfg, model, bkg, calib, frames, bb_x, bb_y_side,
    bb_y_bottom) with frames uint8 [n, Hs + Hb, W + 2 MARGIN] holding the boxes where the box positions point."""
    bottom = np.asarray(bottom, np.uint8)
    side = np.asarray(side, np.uint8)
    n, Hb, W = bottom.shape
    assert side.shape[0] == n and side.shape[2] == W
    Hs = side.shape[1]
    rows, cols = Hs + Hb, W + 2 * MARGIN
    cfg = Config(vid_rows=rows, vid_cols=cols, n_rows=rows, n_cols=cols, bb_w=W, bb_h_bottom=Hb, bb_h_side=Hs,
                 tail_sub_bounding_box=0.6, flip=False, imadjust=False, conn=conn, n_tail_points=n_tail_points,
                 min_overlap=0.7, fma_mode=fma_mode, cand_cap=cand_cap, det_cap=det_cap, match_cap=match_cap)
    frames = np.zeros((n, rows, cols), np.uint8)
    frames[:, :Hs, MARGIN:MARGIN + W] = side
    frames[:, Hs:, MARGIN:MARGIN + W] = bottom
    frames[:, 0, cols - 1] = 255
    frames[:, rows - 1, 0] = 0
    bkg = np.zeros((rows, cols), np.uint8)
    calib = np.arange(rows * cols, dtype=np.int32).reshape(rows, cols)
    bb_x = np.full(n, MARGIN + W - 1, np.uint32)
    bb_y_side = np.full(n, Hs - 1, np.uint32)
    bb_y_bottom = np.full(n, rows - 1, np.uint32)
    if check:
        from oracle import oracle

        assert oracle.check_roi(cfg, model, bb_x[0], bb_y_side[0], bb_y_bottom[0]) == 0
        for f in range(n):
            got, mm = oracle.preprocess(cfg, bkg, calib, frames[f])
            assert (int(mm[0]), int(mm[1])) == (0, 255)
            assert np.array_equal(got, frames[f]), f"frame {f}: the window pixels are not the designed ones"
    return cfg, model, bkg, calib, frames, bb_x, bb_y_side, bb_y_bottom


def box_origin(cfg: Config, view: int):
    """(x0, y0) of the view's box in the calibrated image (view 0 = bottom, 1 = side)."""
    return MARGIN, (cfg.bb_h_side if view == 0 else 0)


# ---- screen_quantize restated -------------------------------------------------------------------------------------------
def lround(x: float) -> int:
    """C's lround: nearest integer, halfway cases away from zero (numpy rounds them to even)."""
    a = abs(x)
    r = math.floor(a)
    if a - r >= 0.5:
        r += 1
    return int(r) if x >= 0 else -int(r)


def screen_quantize(w, rho):
    """The screen's 16-bit weights and rigorous thresholds for template w (float32, row-major taps) and bias rho, in the same
    double-precision operation order as csrc/k_screen.cu screen_quantize, plus k_screen2's 32-bit forms q_need / q_sign."""
    taps = [float(x) for x in np.asarray(w, np.float32).reshape(-1)]
    n = len(taps)
    wmax = wabs = 0.0
    for x in taps:
        wmax = max(wmax, abs(x))
        wabs += abs(x)
    init = float(np.float32(-rho))
    scale = wmax / 32000.0 if wmax > 0.0 else 1.0
    vq = np.zeros(n, np.int64)
    eq = 0.0
    for i, x in enumerate(taps):
        v = max(-32000, min(32000, lround(x / scale)))
        vq[i] = v
        eq += abs(x - scale * float(v))
    rho_f = -init
    u = math.ldexp(1.0, -24)
    efp = (2.0 * n + 2.0) * u * (abs(rho_f) + 255.0 * wabs) * 1.01
    eps = (255.0 * eq + efp) * (1.0 + 1e-9) + 1e-300
    lo = math.floor((rho_f - eps) / scale) - 1.0
    hi = math.ceil((rho_f + eps) / scale) + 1.0
    lim = 4.0e18
    t_lo = int(max(-lim, min(lim, lo)))
    t_hi = int(max(-lim, min(lim, hi)))
    clampi = lambda x: max(-(2 ** 31) + 1, min(2 ** 31 - 2, x))
    return dict(scale=scale, vq=vq.reshape(np.shape(w)), eq=eq, efp=efp, eps=eps, t_lo=t_lo, t_hi=t_hi,
                q_need=clampi(t_lo // 256), q_sign=clampi(t_hi // 256), init=init)


def exact_v(image, vq, x0, y0, width, height):
    """V[y, x] = sum_ij vq[j, i] * I[y0 + y + j - kh/2, x0 + x + i - kw/2] in int64 (the image zero-extended)."""
    kh, kw = vq.shape
    ay, ax = kh // 2, kw // 2
    P = np.zeros((height + kh - 1, width + kw - 1), np.int64)
    ys, xs = np.arange(y0 - ay, y0 - ay + P.shape[0]), np.arange(x0 - ax, x0 - ax + P.shape[1])
    yv = (ys >= 0) & (ys < image.shape[0])
    xv = (xs >= 0) & (xs < image.shape[1])
    P[np.ix_(yv, xv)] = image[np.ix_(ys[yv], xs[xv])]
    V = np.zeros((height, width), np.int64)
    for j, i in zip(*np.nonzero(vq)):
        V += int(vq[j, i]) * P[j:j + height, i:i + width]
    return V


def fp32_scores(w, rho, px, fma_mode=True):
    """The oracle's fp32 scores of a stack of windows (px: [n, kh, kw] pixels under the template): acc = float(-rho), then
    the taps in row-major order, fused or as a product and a sum.  Zero-weight taps are skipped (they can only turn a -0.0
    accumulator into +0.0); used to pick designs, the tests take the oracle's own scores."""
    w = np.asarray(w, np.float32)
    px = np.asarray(px, np.float64).reshape(len(px), -1)
    acc = np.full(px.shape[0], np.float32(-rho), np.float32)
    for t in np.flatnonzero(w.reshape(-1)):
        prod = float(w.reshape(-1)[t]) * px[:, t]          # exact in double (24 x 8 bits)
        acc = (prod + acc.astype(np.float64)).astype(np.float32) if fma_mode else acc + prod.astype(np.float32)
    return acc


# ---- tight templates ----------------------------------------------------------------------------------------------------
S_FIX = 0.5                    # the fixing tap's weight: v = 32000, scale = 0.5 / 32000
SCALE = S_FIX / 32000.0


def tight_template(shape, taps, direction, delta=0.02):
    """A template whose quantisation residuals all have one sign.  taps: [(j, i, k)] -- the first is the fixing tap (k
    ignored, weight S_FIX), the second the unit tap (k = 1, residual s / 100); weight float32(s (k + 1/2 - delta)) for
    direction +1 (residual > 0: rounds down to k), float32(s (k - 1/2 + delta)) for direction -1.  Returns float32 [kh, kw]."""
    w = np.zeros(shape, np.float32)
    for q, (j, i, k) in enumerate(taps):
        # the unit tap's residual is kept small so that stepping its pixel moves V without moving the residual sum
        dq = 0.49 if q == 1 else delta
        w[j, i] = S_FIX if q == 0 else np.float32(SCALE * (k + direction * (0.5 - dq)))
    qz = screen_quantize(w, 0.0)
    assert qz["scale"] == SCALE
    for q, (j, i, k) in enumerate(taps[1:]):
        assert qz["vq"][j, i] == k, (shape, j, i, k)
        r = float(w[j, i]) - SCALE * k
        assert (r > 0) if direction > 0 else (r < 0)
    return w


def tap_layout(shape):
    """Tap positions (j, i, k) for a tight template of the given shape: the fixing tap, the unit tap, then up to seven more
    with assorted k, spread over the template (at most the template's size)."""
    kh, kw = shape
    pos = [(j, i) for j in range(kh) for i in range(kw)]
    if len(pos) > 9:   # spread 9 positions over a large template, the anchor's neighbourhood first
        ay, ax = kh // 2, kw // 2
        want = [(ay, ax), (ay, ax + 1), (ay + 1, ax), (0, 0), (kh - 1, kw - 1), (0, kw - 1), (kh - 1, 0), (ay, 0), (0, ax)]
        pos = [p for p in dict.fromkeys((min(j, kh - 1), min(i, kw - 1)) for j, i in want)]
    ks = [0, 1, 16, 1000, 7, 250, 3, 12000, 60]
    return [(j, i, ks[q]) for q, (j, i) in enumerate(pos[:9])]


def design_windows(w, rho, direction, fma_mode=True):
    """For a tight template w: the window family "fixing tap and k-taps = 255, the k = 16 tap = 255 or 239, the unit tap =
    p" (p = 0..255) -> (pixels uint8 [n, kh, kw], V int64 [n], fp32 score [n]).  Non-tap pixels are 0 except the anchor,
    which is 255 (so that paw / snout outputs are unmasked)."""
    kh, kw = w.shape
    vq = screen_quantize(w, rho)["vq"]
    base = np.zeros((kh, kw), np.uint8)
    base[kh // 2, kw // 2] = 255
    base[w != 0] = 255
    unit, k16 = np.argwhere(vq == 1), np.argwhere(vq == 16)
    qs = (255, 239) if len(k16) else (255,)
    ps = range(256) if len(unit) else (255,)
    px = np.repeat(base[None], len(qs) * len(ps), axis=0)
    for a, q in enumerate(qs):
        for b, p in enumerate(ps):
            if len(k16):
                px[a * len(ps) + b][tuple(k16[0])] = q
            if len(unit):
                px[a * len(ps) + b][tuple(unit[0])] = p
    V = np.tensordot(px.astype(np.int64), vq.astype(np.int64), axes=([1, 2], [0, 1]))
    return px, V, fp32_scores(w, rho, px, fma_mode)


def pick_rho(w, direction):
    """rho for a tight template such that its window family crosses 0 where the 32-bit thresholds cut (when the bound is
    narrow enough for that, else just somewhere inside the family):
    direction +1 (paw / snout): the smallest positive window lies in the block H = q_need and the family has windows in the
    blocks q_need - 1 and q_need + 1;  direction -1 (tail): the largest non-positive window lies in the block H = q_sign."""
    kh, kw = w.shape
    taps = [(j, i) for j, i in zip(*np.nonzero(w))]
    base = float(sum(float(w[j, i]) * 255.0 for j, i in taps))
    unit = [(j, i) for j, i in taps if abs(float(w[j, i]) - SCALE) < SCALE / 2]
    wu = float(w[unit[0]]) if unit else 0.0
    fallback = None
    for pstar in range(40, 250, 3):
        rho = base - wu * (255 - pstar) - 0.5 * wu
        qz = screen_quantize(w, rho)
        _, V, sc = design_windows(w, rho, direction)
        pos = sc > 0
        if not pos.any() or pos.all():
            continue
        if fallback is None:
            fallback = rho
        if direction > 0:
            H = int(V[pos].min()) // 256
            if H == qz["q_need"] and {H - 1, H + 1} <= set((V // 256).tolist()):
                return rho
        elif int(V[~pos].max()) // 256 == qz["q_sign"]:
            return rho
    # large templates: the fp32 term of the bound alone spans more than one block; the family still crosses 0
    assert fallback is not None
    return fallback


def select_edge_windows(w, rho, direction, fma_mode=True):
    """Per 256-unit block H the window with the smallest positive V and the one with the largest non-positive V."""
    px, V, sc = design_windows(w, rho, direction, fma_mode)
    best = {}
    for k in range(len(V)):
        key = (int(V[k]) // 256, bool(sc[k] > 0))
        if key not in best or (V[k] < V[best[key]] if key[1] else V[k] > V[best[key]]):
            best[key] = k
    return [px[best[k]] for k in sorted(best)]


def place(box, w, windows, positions, occupied):
    """Writes designed windows of template w (anchor at the output position) into a box image at the first positions where
    the pixels the output reads (its nonzero taps and its centre) lie inside the box and are read by no output placed
    before (`occupied`, shared by all templates of the view).  A designed output then sees exactly its window.  Returns the
    list of (x, y) used."""
    H, W = box.shape
    kh, kw = w.shape
    ay, ax = kh // 2, kw // 2
    rmask = w != 0
    rmask[ay, ax] = True
    js, is_ = np.nonzero(rmask)
    used = []
    it = iter(windows)
    win = next(it, None)
    for (x, y) in positions:
        if win is None:
            break
        yy, xx = y - ay + js, x - ax + is_
        if yy.min() < 0 or xx.min() < 0 or yy.max() >= H or xx.max() >= W or occupied[yy, xx].any():
            continue
        occupied[yy, xx] = True
        box[yy, xx] = win[js, is_]
        used.append((x, y))
        win = next(it, None)
    return used


def positions(width, height, xs_extra=(), ys_extra=()):
    """Output positions where the tiling can go wrong: x = 0 / 31 (mod 32), the last column, y = 127 / 128 / 255 / 256, the
    box edges -- then a coarse grid to take the remaining windows."""
    xs = sorted({x for x in [0, 31, 32, 63, 64, 95, 96, 127, 128, 159, 160, width - 1, *xs_extra] if 0 <= x < width})
    ys = sorted({y for y in [0, 1, 127, 128, 255, 256, height - 1, *ys_extra] if 0 <= y < height})
    first = [(x, y) for y in ys for x in xs]
    grid = [(x, y) for y in range(2, height, 9) for x in range(2, width, 11)]
    return first + grid


# ---- Part 1 problem: tight templates at the screen's thresholds ---------------------------------------------------------
SMALL_SHAPES = (((2, 2), (3, 5), (3, 3)), ((3, 5), (2, 2), (3, 3)))
MIXED_SHAPES = (((30, 30), (24, 28), (20, 16)), ((27, 30), (30, 22), (15, 17)))
LARGE_SHAPES = (((40, 40),) * 3,) * 2
THRESH_BOX = (170, 260, 100)      # W (tail_w = 102), Hb (two 128-row tiles and a ragged third), Hs (stacked tiles straddle frames)


def tight_model(shapes):
    """Paw / snout templates with residuals > 0 and tail templates with residuals < 0, each with the rho of pick_rho."""
    w = [[None] * 3 for _ in range(2)]
    rho = [[0.0] * 3 for _ in range(2)]
    for v in range(2):
        for k in range(3):
            d = -1 if k == 2 else 1
            w[v][k] = tight_template(shapes[v][k], tap_layout(shapes[v][k]), d)
            rho[v][k] = pick_rho(w[v][k], d)
    return Model(w=w, rho=rho)


def threshold_problem(shapes, fma_mode=True):
    """Three frames (cfg, model, ... as make_problem):
      0: the paw / snout edge windows of both views at the tiling's awkward positions;
      1: bottom: only the tail windows whose score is <= 0 (the oracle's bottom tail map is empty, so one output wrongly
         declared positive changes the tracks); side: all tail windows;
      2: bottom: all tail windows plus a band of 255 over the tail columns (its region is the winner and opens the side
         columns);
         side: the tail windows whose score is <= 0."""
    model = tight_model(shapes)
    W, Hb, Hs = THRESH_BOX
    tail_w = int(float(W) * 0.6)
    bottom = np.zeros((3, Hb, W), np.uint8)
    side = np.zeros((3, Hs, W), np.uint8)
    for v, boxes in ((0, bottom), (1, side)):
        H = boxes.shape[1]
        occ = np.zeros((H, W), bool)
        for k in (0, 1):
            wins = select_edge_windows(model.w[v][k], model.rho[v][k], 1, fma_mode)
            place(boxes[0], model.w[v][k], wins * 3, positions(W, H), occ)
        wt, rt = model.w[v][2], model.rho[v][2]
        wins = select_edge_windows(wt, rt, -1, fma_mode)
        neg = [p for p in wins if not fp32_scores(wt, rt, p[None], fma_mode)[0] > 0]
        tail_pos = [(x, y) for (x, y) in positions(tail_w, H, xs_extra=(tail_w - 1,))]
        for f, sel in ((1, neg if v == 0 else wins), (2, wins if v == 0 else neg)):
            occ = np.zeros((H, W), bool)
            if f == 2 and v == 0:
                boxes[f, H - 5:, :tail_w] = 255
                occ[H - 5:] = True
            place(boxes[f], wt, sel * 3, tail_pos, occ)
    return make_problem(bottom, side, model, fma_mode=fma_mode)


def view_outputs(cfg, model, frame, view, feat, fma_mode):
    """(V int64, fp32 scores in the given mode, centre pixels) of every output of one template over its box."""
    x0, y0 = box_origin(cfg, view)
    width = cfg.tail_w if feat == 2 else cfg.bb_w
    height = cfg.bb_h_bottom if view == 0 else cfg.bb_h_side
    from oracle import oracle

    qz = screen_quantize(model.w[view][feat], model.rho[view][feat])
    V = exact_v(frame, qz["vq"], x0, y0, width, height)
    sc = oracle.correlate(frame, model.w[view][feat], model.rho[view][feat], x0, y0, width, height, fma_mode)
    centre = frame[y0:y0 + height, x0:x0 + width]
    return V, sc, centre, qz


def count_positives(cfg, model, frames):
    """Outputs with score > 0 and centre pixel > 25 over paw and snout in both views (the device's positive-pixel lists)."""
    n = 0
    for f in range(len(frames)):
        for v in (0, 1):
            for k in (0, 1):
                _, sc, centre, _ = view_outputs(cfg, model, frames[f], v, k, cfg.fma_mode)
                n += int(((sc > 0) & (centre > 25)).sum())
    return n


# ---- Part 2 / 3: binary tail maps through 1 x 1 templates -------------------------------------------------------------
MAP_BOX = (170, 40, 30)           # W (tail_w = 102: not a multiple of 32), Hb, Hs


def unit_model(rho_paw=1000.0, rho_snout=1000.0, rho_tail=25.5):
    """1 x 1 templates with w = 1: a view's tail map is `pixel >= 26`; paw / snout outputs are positive iff pixel > rho."""
    one = np.ones((1, 1), np.float32)
    return Model(w=[[one] * 3, [one] * 3], rho=[[rho_paw, rho_snout, rho_tail], [rho_paw, rho_snout, rho_tail]])


def maps_to_boxes(bmaps, smaps, value=255):
    """[n, Hb, tail_w] / [n, Hs, tail_w] 0/1 maps -> box images of MAP_BOX width (pixel `value` where the map is 1)."""
    W = MAP_BOX[0]
    n, Hb, tw = bmaps.shape
    bottom = np.zeros((n, Hb, W), np.uint8)
    side = np.zeros((n, smaps.shape[1], W), np.uint8)
    bottom[:, :, :tw] = np.where(bmaps != 0, value, 0)
    side[:, :, :tw] = np.where(smaps != 0, value, 0)
    return bottom, side


def run_count(binary):
    """Horizontal runs of a 0/1 map (what k_tail's shared-memory path has to hold)."""
    b = (np.asarray(binary) != 0).astype(np.int8)
    return int((np.diff(np.pad(b, ((0, 0), (1, 0))), axis=1) == 1).sum())


def _spiral(n):
    """A square spiral path of width 1 with one free pixel between its arms (n x n)."""
    m = np.zeros((n, n), np.uint8)
    y, x = 0, 0
    lengths = [n - 1, n - 1, n - 1]
    k = n - 3
    while k > 0:
        lengths += [k, k]
        k -= 2
    for q, ln in enumerate(lengths):
        dy, dx = ((0, 1), (1, 0), (0, -1), (-1, 0))[q % 4]
        for _ in range(ln):
            m[y, x] = 1
            y, x = y + dy, x + dx
    m[y, x] = 1
    return m


def _tail_maps():
    """name -> (bottom map [40, 102], side map [30, 102]), 0/1."""
    Hb, Hs, tw = MAP_BOX[1], MAP_BOX[2], int(float(MAP_BOX[0]) * 0.6)
    out = {}

    def new():
        return np.zeros((Hb, tw), np.uint8), np.zeros((Hs, tw), np.uint8)

    # A starts at (1, 2k), B at (0, 2k + 2): B first in raster order, A's 2x2 block first; equal areas
    b, s = new()
    b[1:5, 10] = 1
    b[0, 12:16] = 1
    s[1:5, 10] = 1
    s[0, 12:16] = 1
    out["tie_block_vs_raster"] = (b, s)
    # equal areas in one block row: A at (2, 40) and B at (3, 20) share block row 1.  Under 8-connectivity B's block
    # (column 10 < 20) comes first, so B wins, while a key r * cols + x0 would pick A; under 4-connectivity A comes first in
    # raster order and wins.  A third region of equal area lies further down.
    b, s = new()
    b[2, 40:46] = 1
    b[3, 20:26] = 1
    b[10:13, 60:62] = 1
    s[2, 40:46] = 1
    s[3, 20:26] = 1
    out["tie_same_block_row"] = (b, s)
    # diagonal neighbours: one region under 8-connectivity, a tie that only the 4-connectivity order decides
    b, s = new()
    b[5:7, 30:32] = 1
    b[7:9, 28:30] = 1
    b[20:22, 70:72] = 1
    s[5:7, 30:32] = 1
    s[7:9, 28:30] = 1
    out["tie_diagonal"] = (b, s)
    # three-way tie of vertical bars starting in rows 3, 2 and 1: the bar at column 57 starts first in both orders and wins
    b, s = new()
    b[3:9, 50] = 1
    b[2:8, 53] = 1
    b[1:7, 57] = 1
    s[:, :] = b[:Hs]
    out["tie_three_way"] = (b, s)
    # square spiral (long union-find chains) against a blob one pixel smaller
    b, s = new()
    sp = _spiral(36)
    b[2:38, 0:36] = sp
    blob = np.zeros(Hb * 40, np.uint8)
    blob[:int(sp.sum()) - 1] = 1
    b[:, 50:90] = blob.reshape(Hb, 40)
    s[:, 0:36] = sp[:Hs]
    out["spiral"] = (b, s)
    # comb whose teeth merge only on the last row, against a blob one pixel smaller
    b, s = new()
    b[0:Hb - 1, 0:40:2] = 1
    b[Hb - 1, 0:39] = 1
    area = int(b.sum())
    blob = np.zeros(Hb * 50, np.uint8)
    blob[:area - 1] = 1
    b[:, 50:100] = blob.reshape(Hb, 50)
    s[0:Hs - 1, 1:41:2] = 1
    s[Hs - 1, 1:40] = 1
    out["comb"] = (b, s)
    # U shapes nested, closing only at the bottom
    b, s = new()
    for q in range(6):
        b[q:Hb - q, 2 * q] = 1
        b[q:Hb - q, 60 - 2 * q] = 1
        b[Hb - 1 - q, 2 * q:60 - 2 * q + 1] = 1
    s[:, 3:90:3] = 1
    out["nested_u"] = (b, s)
    # checkerboard: one region under 8-connectivity, all singletons (a 600-way tie) under 4
    b, s = new()
    yy, xx = np.mgrid[0:20, 0:60]
    b[5:25, 20:80] = ((yy + xx) % 2 == 0)
    s[0:20, 30:90] = ((yy + xx) % 2 == 1)
    out["checkerboard"] = (b, s)
    # runs across 32-bit words, a full-width row, the last column
    b, s = new()
    b[4, 28:37] = 1
    b[6, 60:70] = 1
    b[8, 95:tw] = 1
    b[12, :] = 1
    b[13, 30:34] = 1
    s[3, 28:37] = 1
    s[5, :] = 1
    out["word_crossing_runs"] = (b, s)
    # a ring touching all four box edges
    b, s = new()
    b[0, :] = b[Hb - 1, :] = 1
    b[:, 0] = b[:, tw - 1] = 1
    s[0, :] = s[Hs - 1, :] = 1
    s[:, 0] = s[:, tw - 1] = 1
    out["box_edges"] = (b, s)
    # empty bottom map: every track stays -1
    b, s = new()
    s[3:9, 10:40] = 1
    out["empty_bottom"] = (b, s)
    # a winner narrower than n_tail_points: segments of width 0 and 1
    b, s = new()
    b[10:20, 40:50] = 1
    s[5:15, 38:52] = 1
    out["narrow_winner"] = (b, s)
    # a winner whose first segment centroid is column 0 (the side z is only taken for x > 0)
    b, s = new()
    b[0:Hb, 0] = 1
    b[Hb // 2, 0:30] = 1
    s[0:Hs, 0:3] = 1
    out["centroid_column_0"] = (b, s)
    # the side's largest region lies outside the bottom winner's columns
    b, s = new()
    b[10:20, 10:40] = 1
    s[2:28, 60:95] = 1
    s[4:8, 20:30] = 1
    out["side_outside_winner"] = (b, s)
    return out


TAIL_MAPS = _tail_maps()


# ---- scores exactly at 0 -------------------------------------------------------------------------------------------------
def output_score(image, w, rho, x, y, fma_mode):
    """The oracle's fp32 score of the output whose template anchor sits on image pixel (x, y)."""
    from oracle import oracle

    return oracle.correlate(image, w, rho, x, y, 1, 1, fma_mode)[0, 0]


def rho_at_zero(image, w, x, y, fma_mode, span=400):
    """Search rho over the neighbouring float32 values of float(-rho) around the output's real-valued sum: returns
    (rho giving the smallest positive score reached, that score, rho giving exactly +0.0 or None).  The score only depends on
    float(-rho), and it never decreases as float(-rho) grows."""
    kh, kw = w.shape
    ys, xs = np.arange(y - kh // 2, y - kh // 2 + kh), np.arange(x - kw // 2, x - kw // 2 + kw)
    P = np.zeros((kh, kw))
    yv, xv = (ys >= 0) & (ys < image.shape[0]), (xs >= 0) & (xs < image.shape[1])
    P[np.ix_(yv, xv)] = image[np.ix_(ys[yv], xs[xv])]
    init = np.float32(-float((np.asarray(w, np.float64) * P).sum()))
    best, best_rho, zero_rho = None, None, None
    cur = np.nextafter(init, np.float32(-np.inf), dtype=np.float32)
    for _ in range(span):
        cur = np.nextafter(cur, np.float32(-np.inf), dtype=np.float32)
    for _ in range(2 * span):
        rho = -float(cur)
        sc = output_score(image, w, rho, x, y, fma_mode)
        if sc == 0 and not np.signbit(sc) and zero_rho is None:
            zero_rho = rho
        if sc > 0 and (best is None or sc < best):
            best, best_rho = sc, rho
        cur = np.nextafter(cur, np.float32(np.inf), dtype=np.float32)
    return best_rho, best, zero_rho


def zero_score_problems(fma_mode=True):
    """Three models on the same frames, with 3 x 5 paw templates of dyadic weights (k 2^-12, |k| < 2048): on windows of 8-bit
    pixels every product and partial sum is exact in float32, so rho_at_zero finds a float(-rho) at which a designed output
    (centre 200) scores exactly +0.0 ("zero"), and the neighbouring value at which it scores the smallest positive value that
    output can reach ("tiny").  "negzero": all weights negative, the centre weight -0.0 and rho = 0, so an output whose
    window is 0 except for its centre scores -0.0.  Returns {name: (problem, (view, x, y) of the designed output)}."""
    rng = np.random.Generator(np.random.PCG64(77))
    k = rng.integers(-2047, 2048, (3, 5))
    k[1, 2] = 1000
    w = (k * 2.0 ** -12).astype(np.float32)
    W, Hb, Hs = 96, 40, 30
    bottom = np.zeros((2, Hb, W), np.uint8)
    side = np.zeros((2, Hs, W), np.uint8)
    bottom[:, 4:36, 4:90] = rng.integers(0, 256, (2, 32, 86))
    side[:, 4:26, 4:90] = rng.integers(0, 256, (2, 22, 86))
    bx, by = 40, 20
    bottom[0, by, bx] = 200
    negw = -np.abs(w)
    negw[1, 2] = -0.0
    bottom[1, by - 3:by + 4, bx - 4:bx + 5] = 0        # frame 1: the designed output's window is 0 except its centre
    bottom[1, by, bx] = 200
    tail = np.ones((1, 1), np.float32)
    out = {}
    base = make_problem(bottom, side, Model(w=[[w, w, tail], [w, w, tail]], rho=[[0.0, 0.0, 25.5]] * 2), fma_mode=fma_mode)
    image = base[4][0]
    x0, y0 = box_origin(base[0], 0)
    tiny_rho, _, zero_rho = rho_at_zero(image, w, x0 + bx, y0 + by, fma_mode)
    assert zero_rho is not None
    for name, wp, rho in (("zero", w, zero_rho), ("tiny", w, tiny_rho), ("negzero", negw, 0.0)):
        model = Model(w=[[wp, w, tail], [w, w, tail]], rho=[[rho, 1e6, 25.5], [1e6, 1e6, 25.5]])
        out[name] = (make_problem(bottom, side, model, fma_mode=fma_mode), (0, bx, by))
    return out


# ---- Part 3: TAIL_MASK ----------------------------------------------------------------------------------------------------
def tail_mask_problem(conn):
    """Bottom paw positives (1 x 1 template, rho = 100.5: pixels >= 101, written as 200) on designed tail maps (pixels >= 26,
    written as 60).  Every paw pixel lies on a pixel that is already in the tail map, so it never changes the map:
      frame 0: the A / B tie of tie_block_vs_raster, one paw pixel inside A and one inside B, one beyond tail_w;
      frame 1: a 6 x 6 winner with paw pixels inside it and on its border, a one-pixel tail region diagonally next to the
               winner's corner with a paw pixel on it (a separate region under 4-connectivity, part of the winner under 8),
               and a paw pixel beyond tail_w;
      frame 2: a tail region and no bottom paw positive: the side paw list stays empty (Q6) although the side has positives."""
    Hb, Hs, tw = MAP_BOX[1], MAP_BOX[2], int(float(MAP_BOX[0]) * 0.6)
    b = np.zeros((3, Hb, tw), np.uint8)
    s = np.zeros((3, Hs, tw), np.uint8)
    b[0] = TAIL_MAPS["tie_block_vs_raster"][0]
    b[1, 20:26, 40:46] = 1
    b[1, 19, 39] = 1
    b[2, 10:15, 10:20] = 1
    s[:, 10:14, 20:24] = 1
    bottom, side = maps_to_boxes(b, s, value=60)
    for f, pts in ((0, [(2, 10), (0, 13), (5, 120)]), (1, [(22, 42), (20, 40), (25, 43), (19, 39), (30, 150)])):
        for y, x in pts:
            assert x >= tw or b[f, y, x], (f, y, x)
            bottom[f, y, x] = 200
    side[:, 10:14, 20:24] = 200
    return make_problem(bottom, side, unit_model(rho_paw=100.5), conn=conn), b


# ---- pass 1 of the base class on thickened tie maps ------------------------------------------------------------------------
BBOX_TIE_MAPS = ("tie_block_vs_raster", "tie_same_block_row", "tie_three_way", "tie_diagonal", "checkerboard")


def bbox_tie_problem():
    """Each tie map scaled by 3 (every shape at least three pixels thick, so that a 3 x 3 median keeps it) as the bottom and
    side views of one frame.  Returns (cfg, model, bkg, calib, frames, params) for lm_bounding_box_base with a 3 x 3
    median, and the thresholded median images of both views (what the labelling sees)."""
    from locomouse_cpp_b200.types import bb_base_params

    bots, sides = [], []
    for name in BBOX_TIE_MAPS:
        b, s = TAIL_MAPS[name]
        bots.append(np.kron(b, np.ones((3, 3), np.uint8)))
        sides.append(np.kron(s, np.ones((3, 3), np.uint8)))
    bottom = np.where(np.stack(bots) != 0, 255, 0).astype(np.uint8)
    side = np.where(np.stack(sides) != 0, 255, 0).astype(np.uint8)
    cfg, model, bkg, calib, frames, *_ = make_problem(bottom, side, unit_model())
    Hs = side.shape[1]
    params = bb_base_params(cfg, side_h=Hs, sums_as_float=0, median_filter_size=3)
    # median >= 3 of a 0 / 255 image: at least 5 of the zero-extended 3 x 3 window set
    from scipy.ndimage import convolve

    med = np.stack([convolve((f != 0).astype(np.int32), np.ones((3, 3), np.int32), mode="constant") >= 5 for f in frames])
    return (cfg, model, bkg, calib, frames, params), med[:, Hs:], med[:, :Hs]
