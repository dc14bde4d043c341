"""Designed frames for pass 1 (csrc/k_bbox_tm.cu, k_bbox_base.cu, k_bbox.cu) and plain numpy / scipy references of every
stage the device keeps: bwAreaOpen, the disk filter, imfill and the column sums of LocoMouse_TM; the binary image, the
median >= 3 image, the largest components and the four sum vectors of the base class; the column counts of LocoMouse_TM_DE.

The references are written from the reference's description of each stage (LocoMouse_TM.cpp:158-269, LocoMouse_class.cpp
579-653 / 921-997, LocoMouse_TM_DE.cpp:56-113), not from oracle/lm_oracle.cpp; tests/test_pass1_designs.py pins them to the
oracle on every design.  A design is a 0 / 1 pattern that becomes a frame through the real front end: identity calibration,
zero background, pixels 0 / 255 (the normalisation and imadjust_default keep 0 / 255, so the binary stage IS the pattern).
Each design names what it is there to reach (`claims`); measure() counts it, and the CPU test fails a design that no longer
reaches it.  Test infrastructure: imported by tests/ only."""
from __future__ import annotations

import dataclasses

import numpy as np
from scipy import ndimage

F32 = np.float32
STRUCT = {4: ndimage.generate_binary_structure(2, 1), 8: np.ones((3, 3), bool)}


# ---- references ------------------------------------------------------------------------------------------------------
def area_open(b, min_count: int, conn: int):
    """bwAreaOpen: the components (conn-connected) of at least min_count pixels."""
    lab, n = ndimage.label(b, STRUCT[conn])
    keep = np.bincount(lab.ravel(), minlength=n + 1) >= min_count
    keep[0] = False
    return keep[lab].astype(np.uint8)


def filter_bound(kern) -> float:
    """Largest distance between the exact sum of a set of taps and OpenCV's float32 accumulation of it: each of the K * K
    adds rounds by at most 2^-24 of a partial sum bounded by sum |w|."""
    k = np.asarray(kern, np.float64)
    return k.size * 2.0 ** -24 * max(1.0, float(np.abs(k).sum()))


def filter_exact(img, kern):
    """The float64 sum of the taps of filter2D(anchor (K/2, K/2), BORDER_REPLICATE) on a 0 / 1 image (exact to ~1e-15)."""
    K = kern.shape[0]
    an = K // 2
    H, W = img.shape
    pad = np.pad(img.astype(np.float64), ((an, K - 1 - an), (an, K - 1 - an)), mode="edge")
    s = np.zeros((H, W), np.float64)
    for j in range(K):
        for i in range(K):
            if kern[j, i] != 0:
                s += float(kern[j, i]) * pad[j:j + H, i:i + W]
    return s


def filter_replay(img, kern, where):
    """OpenCV's float32 accumulation, tap by tap in row-major order, at the pixels `where` (boolean mask)."""
    K = kern.shape[0]
    an = K // 2
    H, W = img.shape
    rr, cc = np.nonzero(where)
    s = np.zeros(rr.size, F32)
    for j in range(K):
        r = np.clip(rr + j - an, 0, H - 1)
        for i in range(K):
            c = np.clip(cc + i - an, 0, W - 1)
            s = (s + F32(kern[j, i]) * img[r, c].astype(F32)).astype(F32)
    return s


def filter2d(img, kern):
    """filter2D(., CV_8U, kern, (-1, -1), 0, BORDER_REPLICATE) on a 0 / 1 image: the exact sum rounded half to even, except
    where it lies within filter_bound of .5, where the float32 replay decides."""
    kern = np.asarray(kern, F32)
    exact = filter_exact(img, kern)
    near = np.abs(exact - np.floor(exact) - 0.5) <= filter_bound(kern) + 1e-9
    v = np.rint(exact)
    if near.any():
        v[near] = np.rint(filter_replay(img, kern, near).astype(np.float64))
    return np.clip(v, 0, 255).astype(np.uint8)


def imfill(filt):
    """imfill: a flood fill from pixel (0, 0) over 4-connected pixels of its value; reached pixels keep their value, every
    other pixel becomes 255.  Returns (reached bool image, CV_32S column sums of the filled image)."""
    lab, _ = ndimage.label(filt == filt[0, 0], STRUCT[4])
    reached = lab == lab[0, 0]
    H = filt.shape[0]
    n = reached.sum(axis=0).astype(np.int64)
    return reached, (int(filt[0, 0]) * n + 255 * (H - n)).astype(np.int32)


def first_last(sums, th, as_float: bool):
    """firstLastOverT: first index >= th, last one (0 when only one qualifies), (-1, -1) when none; as_float reads the int32
    sums through a float pointer."""
    s = np.ascontiguousarray(sums, np.int32)
    v = s.view(np.float32) if as_float else s.astype(np.float32)
    ok = np.nonzero(v >= np.float32(th))[0]
    if ok.size == 0:
        return -1, -1
    return int(ok[0]), int(ok[-1]) if ok.size > 1 else 0


def window_count(b, k: int):
    """Set pixels in the zero-extended k x k window of every pixel."""
    return ndimage.correlate(b.astype(np.int32), np.ones((k, k), np.int32), mode="constant", cval=0)


def median_major(b, k: int):
    """median >= 3 of a 0 / 255 image padded by k / 2 zeros: at least (k * k + 1) / 2 window pixels set."""
    return (window_count(b, k) >= (k * k + 1) // 2).astype(np.uint8)


def label_keys(lab, conn: int):
    """The order of OpenCV's labels: raster order of a component's first pixel (4), of its first 2 x 2 block (8)."""
    H, W = lab.shape
    r, c = np.mgrid[0:H, 0:W]
    key = r * W + c if conn == 4 else (r // 2) * ((W + 1) // 2) + c // 2
    return key


def largest(b, conn: int):
    """The largest component; ties go to the lowest OpenCV label (largestBWAreaObject / selectLargestRegion)."""
    lab, n = ndimage.label(b, STRUCT[conn])
    if n == 0:
        return np.zeros(b.shape, np.uint8)
    area = np.bincount(lab.ravel(), minlength=n + 1)[1:]
    key = np.asarray(ndimage.minimum(label_keys(lab, conn), lab, np.arange(1, n + 1)), np.int64)
    best = np.lexsort((key, -area))[0] + 1
    return (lab == best).astype(np.uint8)


# ---- pipelines ---------------------------------------------------------------------------------------------------------
def tm_stages(d: "TmDesign", conn: int):
    """opened / filtered / reached images, the column sums and (first, last) of LocoMouse_TM on design d."""
    b = d.binary()
    opened = area_open(b, d.min_count, conn)
    filt = filter2d(opened, d.disk)
    reached, sums = imfill(filt)
    return dict(binary=b, opened=opened, filtered=filt, reached=reached, sums=sums, lims=first_last(sums, d.min_vis, d.as_float))


def base_stages(d: "BaseDesign", conn: int):
    """binary / median images, the four sum vectors and limits of the base class on design d."""
    b = d.pattern.astype(np.uint8)
    major = median_major(b, d.k)
    sums, lims = [], []
    for (x, y, w, h) in (d.side, d.bottom):
        big = largest(major[y:y + h, x:x + w], conn).astype(np.int32)
        sums.append((big.sum(axis=0) * 255, big.sum(axis=1) * 255))
    vecs = [sums[0][0], sums[1][0], sums[0][1], sums[1][1]]   # Row_side, Row_bottom, Col_side, Col_bottom
    lims = np.array([first_last(v, d.min_vis, d.as_float) for v in vecs], np.int32)
    return dict(binary=b, major=major, sums=np.concatenate(vecs).astype(np.int32), lims=lims)


def de_stages(d: "DeDesign"):
    """Column counts and (first, last) of LocoMouse_TM_DE on design d."""
    c0, c1, r0, r1 = d.zero
    m = np.zeros(d.pattern.shape, np.int32)
    m[r0:r1, c0:c1] = d.pattern[r0:r1, c0:c1]
    sums = m.sum(axis=0).astype(np.int32)
    return dict(sums=sums, lims=first_last(sums, d.min_count, False))


def run_count(b) -> int:
    """Horizontal runs of set pixels."""
    b = np.asarray(b, bool)
    return int((b & ~np.pad(b, ((0, 0), (1, 0)))[:, :-1]).sum())


# ---- designs -------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class TmDesign:
    name: str
    pattern: np.ndarray               # H x W 0 / 1: the binary stage
    disk: np.ndarray
    min_count: int = 1
    min_vis: int = 1
    as_float: int = 0
    claims: tuple = ()

    def binary(self):
        return self.pattern.astype(np.uint8)

    def frame(self):
        return (self.pattern * 255).astype(np.uint8)


@dataclasses.dataclass
class BaseDesign:
    name: str
    pattern: np.ndarray               # the whole calibrated image, 0 / 1
    k: int
    side: tuple                       # (x, y, w, h)
    bottom: tuple
    min_vis: int = 1
    as_float: int = 0
    claims: tuple = ()

    def frame(self):
        return (self.pattern * 255).astype(np.uint8)


@dataclasses.dataclass
class DeDesign:
    name: str
    pattern: np.ndarray               # the side view = the whole image, 0 / 1
    min_count: int
    zero: tuple                       # surviving columns [c0, c1), rows [r0, r1)
    claims: tuple = ()

    def frame(self):
        return (self.pattern * 255).astype(np.uint8)


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def _random(H, W, p, seed):
    return (_rng(seed).random((H, W)) < p).astype(np.uint8)


def _k(rows):
    return np.array(rows, F32)


def disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    h = ((x * x + y * y) <= (r + 0.5) ** 2).astype(np.float64)
    return (h / h.sum()).astype(F32)


def _uniform(K, w):
    return np.full((K, K), w, F32)


def _levels(K, n, seed):
    """A K x K kernel with exactly n distinct non-zero weights, positive sum about 1.2."""
    rng = _rng(seed)
    vals = (np.arange(1, n + 1) * 0.37 + 1.0)
    idx = np.concatenate([np.arange(n), rng.integers(0, n, K * K - n)])
    rng.shuffle(idx)
    k = vals[idx].reshape(K, K)
    return (k / k.sum() * 1.2).astype(F32)


def _ballast(p, r0, c0, h=4, w=4):
    """A block far from the pixels a design is about, so that 1 % .. 99 % of the side view is set."""
    p[r0:r0 + h, c0:c0 + w] = 1
    return p


def tm_designs():
    D = []
    # -- disk filter -------------------------------------------------------------------------------------------------------
    # multiples of 0.1f: subsets whose exact sum lies just above .5 accumulate to exactly 0.5f in float32 (round half to
    # even: 0), e.g. 0.1f + 0.4f, 0.2f + 0.3f, 0.1f + 0.1f + 0.3f
    D.append(TmDesign("ties_0.1f_3x3", _random(24, 65, 0.45, 1), _k([[0.1, 0.2, 0.1], [0.3, 0.1, 0.4], [0.1, 0.1, 0.0]]),
                      claims=("replay_disagrees", "replay_on_half")))
    D.append(TmDesign("ties_0.1f_5x5", _random(30, 97, 0.25, 2), _k(np.where(_random(5, 5, 0.45, 3), 0.1, 0.0)),
                      claims=("replay_disagrees", "replay_on_half")))
    # sums 0.5 +- 1e-6 (inside the device's rounding margin, ~2.7e-6 here) and 0.5 +- 4e-6 (just outside)
    m = _k([[0.25 + 1e-6, 0, 0.25 - 1e-6], [0, 0.25, 0], [0.25 + 4e-6, 0, 0.25 - 4e-6]])
    D.append(TmDesign("margin_in_out", _random(24, 65, 0.4, 4), m, claims=("inside_margin", "just_outside_margin")))
    D.append(TmDesign("levels_8", _random(26, 65, 0.5, 5), _levels(5, 8, 6), claims=("levels8",)))
    D.append(TmDesign("levels_9", _random(26, 65, 0.5, 7), _levels(5, 9, 8), claims=("levels9",)))
    D.append(TmDesign("K1", _random(20, 33, 0.3, 9), _k([[1.0]])))
    D.append(TmDesign("K2_even", _random(22, 65, 0.5, 10), _uniform(2, 0.25), claims=("exact_half", "replay_on_half")))
    D.append(TmDesign("K4_even_anchor", _random(22, 65, 0.35, 11), _k([[0.03] * 4] * 3 + [[0.2] * 4]), claims=("empty_word_lit",)))
    blobs = np.zeros((40, 97), np.uint8)
    blobs[5:30, 10:40] = 1
    blobs[12:38, 60:90] = 1
    blobs[20:24, 44:50] = 1
    D.append(TmDesign("K32_exact_ties", blobs, _uniform(32, 1.0 / 1024), claims=("exact_half",)))
    D.append(TmDesign("K33_H_lt_K", blobs[8:28].copy(), _uniform(33, 1.0 / 1089)))
    D.append(TmDesign("K63_H_lt_K", blobs[4:28].copy(), disk(31)))
    # negative taps, positive sum 1.498: the margin scales with sum |w| = 2.198
    neg = _k([[-0.3, 0.5, -0.2], [0.3, 0.499, 0.199], [-0.1, 0.0, -0.1]])
    D.append(TmDesign("negative_taps", _random(24, 65, 0.5, 12), neg, claims=("replay_disagrees_or_near",)))
    for W in (33, 65, 97):
        D.append(TmDesign(f"width_{W}", _random(21, W, 0.3, 13 + W), disk(2), claims=("border_taps",)))
    # single set pixels (and short lines) where the replicated border adds taps: last column, last row, corner
    b = _ballast(np.zeros((20, 65), np.uint8), 8, 20, 4, 5)
    b[0, 64] = b[19, 64] = b[19, 0] = 1          # three corners
    b[9:12, 64] = 1                               # a vertical line in the last column
    b[19, 30:33] = 1                              # a horizontal line in the last row
    D.append(TmDesign("border_singles", b, _uniform(3, 0.15), claims=("border_taps",)))
    # an empty word whose neighbourhood is not: a block that ends in column 31, filtered into word 1
    e = _ballast(np.zeros((20, 97), np.uint8), 14, 70)
    e[3:9, 26:32] = 1
    e[12, 64:70] = 1                              # a row whose rows above are empty: output lands in words of empty rows
    D.append(TmDesign("empty_word_neighbour", e, _uniform(5, 0.05), claims=("empty_word_lit",)))
    # -- bwAreaOpen ------------------------------------------------------------------------------------------------------
    a = np.zeros((24, 65), np.uint8)
    a[1, 2:7] = 1                                 # 5 pixels: kept at min_count 5
    a[4, 2:6] = 1                                 # 4 pixels: removed
    a[7, 10:13] = 1
    a[8, 13:16] = 1                               # 3 + 3 joined diagonally only: kept under 8, removed under 4
    a[12, 28:41] = 1                              # a run across a word boundary
    a[15, 60:65] = 1                              # a run ending in the last column
    a[16, 62:65] = 1
    a[20:23, 30:32] = 1                           # 6 pixels
    a[18, 5:9] = 1
    a[19, 9] = 1                                  # 4 + 1 diagonal: 5 under 8, 4 and 1 under 4
    D.append(TmDesign("area_open", a, _k([[1.0]]), min_count=5, claims=("area_eq", "area_eq_minus1", "diagonal_join")))
    D.append(TmDesign("area_open_noise", _random(26, 97, 0.35, 20), disk(1), min_count=3, claims=("area_eq", "area_eq_minus1", "diagonal_join")))
    # -- imfill ----------------------------------------------------------------------------------------------------------
    f = np.zeros((24, 65), np.uint8)
    f[2:9, 2:9] = 1
    f[4:7, 4:7] = 0                               # an enclosed hole
    f[2:9, 12:19] = 1
    f[4:7, 14:17] = 0
    f[3, 13] = 0                                  # its hole reaches the outside only diagonally: filled
    f[8, 18] = 0
    f[7, 17] = 0                                  # (a diagonal gap at the corner)
    f[10:20, 56:65] = 1
    f[12:18, 60:65] = 0                           # a hole closed by the right edge (last column)
    f[13, 58] = 0
    D.append(TmDesign("imfill_holes", f, _k([[1.0]]), claims=("holes", "diagonal_hole", "last_col_hole")))
    s = np.zeros((25, 33), np.uint8)             # a square spiral: its inside reaches the outside through one corridor
    s[1, 1:32] = s[1:24, 31] = s[23, 1:32] = s[3:24, 1] = 1
    s[3, 1:29] = s[3:21, 28] = s[20, 4:29] = s[6:21, 4] = 1
    s[6, 4:25] = s[6:18, 24] = s[17, 7:25] = s[9:18, 7] = 1
    s[9, 7:21] = 1
    D.append(TmDesign("imfill_spiral", s, _k([[1.0]]), claims=("spiral",)))
    s2 = s.copy()
    s2[2, 1] = 1                                  # the corridor closed: everything inside is filled
    D.append(TmDesign("imfill_spiral_closed", s2, _k([[1.0]]), claims=("holes",)))
    g = np.zeros((20, 65), np.uint8)
    g[0:12, 0:20] = 1
    g[3:6, 3:6] = 0                               # seed pixel set: the fill runs over the object, its hole becomes 255
    g[15:18, 40:45] = 1                           # a second object the fill does not reach
    D.append(TmDesign("imfill_seed_set", g, _k([[1.0]]), claims=("seed_set",)))
    # -- sums and firstLastOverT -----------------------------------------------------------------------------------------
    c = _ballast(np.zeros((20, 33), np.uint8), 2, 26, 2, 4)
    c[4:7, 20] = 1                                # one column with 3 set pixels: sum 765 (the ballast's columns: 510)
    for mv, cl in ((765, ("vis_at_sum", "one_column")), (766, ("vis_above_sum",)), (1, ()), (0, ())):
        D.append(TmDesign(f"sums_vis_{mv}", c, _k([[1.0]]), min_vis=mv, claims=cl))
    D.append(TmDesign("sums_none", c, _k([[1.0]]), min_vis=100000, claims=("no_column",)))
    D.append(TmDesign("sums_as_float_1", c, _k([[1.0]]), min_vis=1, as_float=1, claims=("no_column",)))
    D.append(TmDesign("sums_as_float_0", c, _k([[1.0]]), min_vis=0, as_float=1, claims=("all_columns",)))
    return D


def _base_border_design(k, seed):
    """A random image whose border windows reach exactly (k * k + 1) / 2 set pixels and one fewer (searched over densities)."""
    need = (k * k + 1) // 2
    H, W = max(2 * k + 8, 40), 97
    for t in range(400):
        p = 0.3 + 0.69 * ((t * 0.618) % 1.0) if k > 1 else 0.5
        b = _random(H, W, p, seed * 1000 + t)
        cnt = window_count(b, k)
        border = np.zeros(b.shape, bool)
        h = k // 2
        border[:h + 1, :] = border[-h - 1:, :] = border[:, :h + 1] = border[:, -h - 1:] = True
        if k == 1 or ((cnt[border] == need).any() and (cnt[border] == need - 1).any() and 0 < b.mean() < 1):
            return b
    raise AssertionError(f"no border design for k = {k}")


def base_designs():
    D = []
    for k in (1, 3, 11, 31):
        b = _base_border_design(k, k)
        H, W = b.shape
        sh = H // 2
        D.append(BaseDesign(f"median_k{k}", b, k, side=(3, 0, W - 5, sh), bottom=(7, sh, W - 9, H - sh), claims=("border_need",)))
    t = np.zeros((40, 97), np.uint8)
    t[3:8, 10:15] = t[12:17, 40:45] = 1           # side view: two 5 x 5 squares (a tie)
    t[3:6, 70:74] = 1                             # 12 pixels
    t[24:28, 20:25] = t[30:34, 60:65] = 1         # bottom view: two 4 x 5 rectangles (a tie)
    t[25, 26] = t[26, 27] = 1                     # diagonal specks: join the first rectangle under 8 only
    D.append(BaseDesign("equal_areas", t, 1, side=(5, 0, 90, 20), bottom=(1, 20, 95, 20), claims=("tie",)))
    D.append(BaseDesign("equal_areas_float", t, 1, side=(5, 0, 90, 20), bottom=(1, 20, 95, 20), min_vis=0, as_float=1))
    D.append(BaseDesign("min_vis_at_sum", t, 1, side=(5, 0, 90, 20), bottom=(1, 20, 95, 20), min_vis=5 * 255))
    return D


def de_designs():
    D = []
    rng = _rng(40)
    for W, flip_name in ((65, "w65"), (67, "w67")):
        p = np.zeros((30, W), np.uint8)
        cols = rng.permutation(np.arange(5, W - 5))[:20]
        for i, c in enumerate(cols):
            p[3:3 + (8 if i == 0 else 4 + i % 4), c] = 1   # column counts 4 .. 7 inside the bands (rows 2 .. 27), one of 8
        p[0:2, :] = 1                                  # the zeroed band rows: shape the histogram only
        D.append(DeDesign(f"counts_{flip_name}_min6", p, 6, zero=(2, W - 2, 2, 28), claims=("count_eq", "count_eq_minus1")))
        D.append(DeDesign(f"counts_{flip_name}_min8", p, 8, zero=(2, W - 2, 2, 28), claims=("count_eq", "count_eq_minus1", "one_column")))
    return D


# ---- frames and parameters -------------------------------------------------------------------------------------------
def problem(shape):
    """(cfg, model, bkg, calib) of a zero-background, identity-calibrated image of `shape` (the design's whole frame)."""
    import dataclasses

    import _preprocess_designs as PD
    from locomouse_cpp_b200.types import Config

    H, W = shape
    _, model = PD.small_geometry(False)
    cfg = dataclasses.replace(Config(), vid_rows=H, vid_cols=W, n_rows=H, n_cols=W, bb_w=min(W, 32), bb_h_bottom=8, bb_h_side=8,
                              imadjust=False, cand_cap=64, det_cap=8192, match_cap=256)
    bkg = np.zeros((H, W), np.uint8)
    calib = np.arange(H * W, dtype=np.int32).reshape(H, W)
    return cfg, model, bkg, calib


def tm_params(cfg, d):
    from locomouse_cpp_b200.types import bb_tm_params

    H, W = d.pattern.shape
    return bb_tm_params(cfg, d.disk, side_h=H, side_threshold=3, min_pixel_count=d.min_count, min_pixel_visible=d.min_vis,
                        sums_as_float=d.as_float)


def base_params(cfg, d):
    from locomouse_cpp_b200.types import bb_base_params

    (sx, sy, sw, sh), (bx, by, bw, bh) = d.side, d.bottom
    return bb_base_params(cfg, side_x=sx, side_y=sy, side_w=sw, side_h=sh, bottom_x=bx, bottom_y=by, bottom_w=bw, bottom_h=bh,
                          median_filter_size=d.k, min_pixel_visible=d.min_vis, sums_as_float=d.as_float)


def de_params(cfg, d):
    from locomouse_cpp_b200.types import bb_de_params

    H, W = d.pattern.shape
    c0, c1, r0, r1 = d.zero
    return bb_de_params(cfg, side_h=H, side_w=W, zero_col_pre=c0, zero_col_post=c1, zero_row_pre=r0, zero_row_post=r1,
                        threshold=255 * 0.05, min_count=d.min_count, width_margin=1.1)


# ---- claims ---------------------------------------------------------------------------------------------------------------
def device_margin(kern) -> float:
    """The rounding margin k_bbtm_disk decides by counting outside of (lm_launch_bbox_tm)."""
    k = np.asarray(kern, F32)
    return 4.0 * k.size * 5.9604644775390625e-8 * max(1.0, float(np.abs(k.astype(np.float64)).sum())) + 1e-9


def measure_tm(d: TmDesign, conn: int):
    st = tm_stages(d, conn)
    opened, filt = st["opened"], st["filtered"]
    kern = d.disk
    exact = filter_exact(opened, kern)
    dist = np.abs(exact - 0.5)
    near = dist <= 1e-3
    rep = filter_replay(opened, kern, near) if near.any() else np.zeros(0, F32)
    rep_round = np.rint(rep.astype(np.float64))
    ex_round = np.rint(exact[near])
    marg = device_margin(kern)
    H, W = opened.shape
    # the filter with a zero border instead of the replicated one
    K = kern.shape[0]
    an = K // 2
    zpad = np.pad(opened.astype(np.float64), ((an, K - 1 - an), (an, K - 1 - an)))
    zsum = sum(float(kern[j, i]) * zpad[j:j + H, i:i + W] for j in range(K) for i in range(K))
    zero_border = np.clip(np.rint(zsum), 0, 255).astype(np.uint8)
    wpr = (W + 31) // 32
    wpad = np.pad(opened, ((0, 0), (0, wpr * 32 - W))).reshape(H, wpr, 32).any(axis=2)
    fpad = np.pad(filt, ((0, 0), (0, wpr * 32 - W))).reshape(H, wpr, 32).any(axis=2)
    lab4 = ndimage.label(st["binary"], STRUCT[4])
    lab8 = ndimage.label(st["binary"], STRUCT[8])
    areas = np.bincount(ndimage.label(st["binary"], STRUCT[conn])[0].ravel())[1:]
    reached4 = st["reached"]
    lab_same8 = ndimage.label(filt == filt[0, 0], STRUCT[8])[0]
    reached8 = lab_same8 == lab_same8[0, 0]
    sums = st["sums"]
    nz = np.unique(np.abs(kern[kern != 0]))
    return {
        "replay_disagrees": int((rep_round != ex_round).sum()),
        "replay_on_half": int((rep == F32(0.5)).sum()),
        "replay_disagrees_or_near": int((dist < 1e-3).sum()),
        "exact_half": int((exact == 0.5).sum()),
        "inside_margin": int(((dist > 0) & (dist <= marg)).sum()),
        "just_outside_margin": int(((dist > marg) & (dist <= 2 * marg)).sum()),
        "levels8": int(np.unique(kern[kern != 0]).size == 8 and nz.size > 0),
        "levels9": int(np.unique(kern[kern != 0]).size == 9),
        "border_taps": int((zero_border != filt).sum()),
        "empty_word_lit": int((fpad & ~wpad).sum()),
        "area_eq": int((areas == d.min_count).sum()),
        "area_eq_minus1": int((areas == d.min_count - 1).sum()),
        "diagonal_join": int(lab4[1] - lab8[1]),
        "holes": int((~reached4 & (filt == filt[0, 0])).sum()),
        "diagonal_hole": int((reached8 & ~reached4).sum()),
        "spiral": int((reached4 & (filt == filt[0, 0])).sum() - (filt == filt[0, 0]).sum() == 0 and reached4[12, 16]),
        "last_col_hole": int((~reached4[:, -1] & (filt[:, -1] == filt[0, 0])).sum()),
        "seed_set": int(filt[0, 0] == 1 and (~reached4 & (filt == 1)).any()),
        "vis_at_sum": int((sums == d.min_vis).sum()),
        "vis_above_sum": int((sums == d.min_vis - 1).sum()),
        "one_column": int(st["lims"][1] == 0 and st["lims"][0] >= 0),
        "no_column": int(st["lims"] == (-1, -1)),
        "all_columns": int(st["lims"] == (0, W - 1)),
    }


def measure_base(d: BaseDesign, conn: int):
    st = base_stages(d, conn)
    need = (d.k * d.k + 1) // 2
    cnt = window_count(d.pattern, d.k)
    h = d.k // 2
    border = np.zeros(cnt.shape, bool)
    border[:h + 1, :] = border[-h - 1:, :] = border[:, :h + 1] = border[:, -h - 1:] = True
    ties = 0
    for (x, y, w, hh) in (d.side, d.bottom):
        lab, n = ndimage.label(st["major"][y:y + hh, x:x + w], STRUCT[conn])
        a = np.sort(np.bincount(lab.ravel())[1:])[::-1]
        ties += int(a.size > 1 and a[0] == a[1])
    return {"border_need": int((cnt[border] == need).any() and (cnt[border] == need - 1).any()), "tie": ties}


def measure_de(d: DeDesign):
    st = de_stages(d)
    return {"count_eq": int((st["sums"] == d.min_count).sum()), "count_eq_minus1": int((st["sums"] == d.min_count - 1).sum()),
            "one_column": int(st["lims"][1] == 0 and st["lims"][0] >= 0)}
