"""The grid-bucketed NMS kernels (k_nms_bottom = nmsMax, k_nms_side = peakClustering) on lists built to probe the cell
geometry: cells are ceil(w/3) x ceil(h/3) pixels and an overlap search reads the 3 x 3 cells around a detection, so the
cases below put overlapping pairs at the largest overlapping distance, pairs exactly on the overlap bound, suppression
chains across cell borders, ties spread over cells, clusters larger than 64 and 1024 members (lists past the shared-memory
capacity run on the global scratch slice), a list filling det_cap exactly and more clusters than cand_cap.  Each result is
compared bit for bit with the oracle and, where the reference's own code is built (oracle/_ref), with it.

Not reachable through lm_debug_nms, which zeroes the tail mask, gives the side view's feature one bottom detection and
returns an error instead of candidates when a flag is set: tail-masked pixels, an empty bottom list beside a non-empty
side list (Q6), a list longer than det_cap, and the content of a truncated candidate list.  Those paths run in the whole
pipeline, whose results test_gpu_parity.py compares with the oracle.  Needs a B200: pytest -m gpu."""
import numpy as np
import pytest

from locomouse_cpp_b200.api import OverflowError_
from locomouse_cpp_b200.types import Config, Model

pytestmark = pytest.mark.gpu

SIZES = [(9, 9), (10, 11), (11, 10), (31, 9), (9, 31), (31, 31), (30, 30)]


def _detector(rows, cols, bw, bh, cand_cap=1024, det_cap=8192):
    from locomouse_cpp_b200.api import Detector

    cfg = Config(vid_rows=2 * rows, vid_cols=cols, n_rows=2 * rows, n_cols=cols, bb_w=cols, bb_h_bottom=rows, bb_h_side=rows,
                 cand_cap=cand_cap, det_cap=det_cap, match_cap=256)
    w = np.zeros((bh, bw), np.float32)
    model = Model(w=[[w, w, w], [w, w, w]], rho=[[1.0] * 3, [1.0] * 3])
    bkg = np.zeros((cfg.vid_rows, cfg.vid_cols), np.uint8)
    calib = np.arange(cfg.n_rows * cfg.n_cols, dtype=np.int32).reshape(cfg.n_rows, cfg.n_cols)
    return Detector(cfg, model, bkg, calib, device=0)


def _tuples(c):
    return [(int(r["x"]), int(r["y"]), float(r["s"])) for r in c]


def _check(oracle, s, bw, bh, **kw):
    """Both kernels (feature 0 bottom, feature 1 side) == oracle (== the reference's code where it is built)."""
    from oracle import reference_nms

    det = _detector(s.shape[0], s.shape[1], bw, bh, **kw)
    try:
        got_b, got_s = det.debug_nms(0, 0, s), det.debug_nms(1, 1, s)
    finally:
        det.close()
    assert _tuples(got_b) == oracle.nms_max(s, bw, bh), f"nmsMax differs, box {bw}x{bh}"
    assert _tuples(got_s) == oracle.peak_clustering(s, bw, bh), f"peakClustering differs, box {bw}x{bh}"
    if reference_nms.available(build=False):
        assert _tuples(got_b) == _tuples(reference_nms.nms_max(s, bw, bh))
        assert _tuples(got_s) == _tuples(reference_nms.peak_clustering(s, bw, bh))
    return got_b, got_s


def _overlap(dx, dy, w, h):
    dx, dy = abs(dx), abs(dy)
    return dx < w and dy < h and 3 * (w - dx) * (h - dy) > 2 * w * h


def _pairs(rng, rows, cols, offsets, n_pairs):
    """Score map with n_pairs detection pairs (p, p + offset), offsets drawn from `offsets`, random distinct scores."""
    s = np.full((rows, cols), -1.0, np.float32)
    for _ in range(n_pairs):
        dx, dy = offsets[rng.integers(len(offsets))]
        x, y = int(rng.integers(0, cols - abs(dx))), int(rng.integers(0, rows - abs(dy)))
        x0, y0 = (x if dx >= 0 else x - dx), (y if dy >= 0 else y - dy)
        s[y0, x0] = rng.random() + 0.01
        s[y0 + dy, x0 + dx] = rng.random() + 0.01
    return s


@pytest.mark.parametrize("bw,bh", SIZES)
def test_pairs_at_the_cell_distance(oracle, bw, bh):
    cx, cy = -(-bw // 3) - 1, -(-bh // 3) - 1
    assert _overlap(cx, 0, bw, bh) and _overlap(0, cy, bw, bh) and not _overlap(cx + 1, 0, bw, bh)
    offs = [(cx, 0), (-cx, 0), (0, cy), (0, -cy)] + [(dx, dy) for dx in (-cx, cx) for dy in (-cy, cy) if _overlap(dx, dy, bw, bh)]
    rng = np.random.Generator(np.random.PCG64(bw * 100 + bh))
    b, s = _check(oracle, _pairs(rng, 96, 128, offs, 40), bw, bh)
    assert len(b) > 0 and len(s) > 0


@pytest.mark.parametrize("bw,bh", SIZES)
def test_pairs_on_the_overlap_bound_do_not_merge(oracle, bw, bh):
    edge = [(dx, dy) for dx in range(bw) for dy in range(bh) if 3 * (bw - dx) * (bh - dy) == 2 * bw * bh]
    near = [(dx, dy) for dx in range(bw) for dy in range(bh) if 3 * (bw - dx) * (bh - dy) in (2 * bw * bh + 1, 2 * bw * bh + 3)]
    offs = [(sx * dx, sy * dy) for dx, dy in edge + near for sx in (1, -1) for sy in (1, -1)] or [(bw // 3, 0)]
    rng = np.random.Generator(np.random.PCG64(7 + bw * bh))
    _check(oracle, _pairs(rng, 96, 128, offs, 40), bw, bh)


@pytest.mark.parametrize("bw,bh", [(9, 9), (10, 11), (31, 9)])
def test_suppression_chains_across_cells(oracle, bw, bh):
    """Rows of detections one cell distance apart with decreasing scores: every link of a chain crosses a cell border,
    and the chain's end is far outside its root's neighbourhood (discarded detections keep suppressing, Q3)."""
    rows, cols = 64, 160
    s = np.full((rows, cols), -1.0, np.float32)
    step = -(-bw // 3) - 1
    for r in range(4, rows, bh + 4):
        xs = np.arange(1 + r % 3, cols, step)
        s[r, xs] = np.linspace(1.0, 0.5, len(xs), dtype=np.float32)
    b, _ = _check(oracle, s, bw, bh)
    assert len(b) > 0


@pytest.mark.parametrize("levels,dens", [(2, 0.3), (4, 0.6), (1, 0.05)])
def test_equal_scores_over_many_cells(oracle, levels, dens):
    rng = np.random.Generator(np.random.PCG64(levels * 10))
    for bw, bh in [(9, 9), (10, 11), (30, 30)]:
        s = rng.integers(1, levels + 1, (72, 120)).astype(np.float32)
        s[rng.random(s.shape) > dens] = -1.0
        _check(oracle, s, bw, bh)


def test_empty_lists(oracle):
    s = np.full((40, 64), -1.0, np.float32)
    b, side = _check(oracle, s, 9, 9)
    assert len(b) == 0 and len(side) == 0


@pytest.mark.parametrize("blob,bw,bh", [(12, 30, 30), (40, 60, 60)])
def test_large_clusters(oracle, blob, bw, bh):
    """One dense blob: a cluster of blob**2 members (> 64; > 1024 for the 40 x 40 blob, whose list exceeds the kernels'
    shared-memory capacity)."""
    rng = np.random.Generator(np.random.PCG64(blob))
    s = np.full((96, 128), -1.0, np.float32)
    s[30:30 + blob, 40:40 + blob] = rng.random((blob, blob)).astype(np.float32) + 0.01
    s[5, 5] = 0.5
    b, side = _check(oracle, s, bw, bh)
    assert len(b) >= 2 and len(side) >= 2


def test_list_at_det_cap(oracle):
    rng = np.random.Generator(np.random.PCG64(3))
    s = rng.random((48, 64)).astype(np.float32)
    s[rng.random(s.shape) > 0.4] = -1.0
    n = int((s > 0).sum())
    _check(oracle, s, 10, 11, det_cap=n)


def test_more_roots_than_cand_cap(oracle):
    """Isolated detections: every one is a root / maximum, so the slots follow the rank order of all 450.  With cand_cap
    below their number the kernels raise the candidate-overflow flag."""
    s = np.full((60, 120), -1.0, np.float32)
    rng = np.random.Generator(np.random.PCG64(11))
    s[::4, ::4] = rng.random((15, 30)).astype(np.float32) + 0.01
    b, side = _check(oracle, s, 9, 9)
    assert len(b) == 450 and len(side) == 450
    det = _detector(60, 120, 9, 9, cand_cap=64)
    try:
        for view in (0, 1):
            with pytest.raises(OverflowError_):
                det.debug_nms(view, 0, s)
    finally:
        det.close()
