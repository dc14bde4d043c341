"""The tensor-core screen (csrc/k_screen.cu) must never change a result: with the screen on (int8 tcgen05
implicit GEMM + sparse exact re-evaluation) and off (dense exact FP32 kernel) every output byte is identical,
and both equal the oracle.  Needs a B200:  pytest -m gpu.
"""
import numpy as np
import pytest

from locomouse_cpp_b200 import synth
from locomouse_cpp_b200.types import Model, diff_results

pytestmark = pytest.mark.gpu


def _detector(cfg, model, bkg, calib, screen):
    from locomouse_cpp_b200.api import Detector

    d = Detector(cfg, model, bkg, calib, device=0)
    d.set_option("screen", screen)
    return d


def _run_both(spec, n, seed, model_edit=None, **kw):
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=seed)
    if model_edit is not None:
        model = model_edit(model)
    frames = frames.numpy()
    out = []
    for screen in (2, 1, 0):
        det = _detector(cfg, model, bkg, calib, screen)
        r = det.detect_batch(frames, bx, bs, bb, **kw)
        out.append((r, det.info("screen_active")))
        det.close()
    return out, (cfg, model, bkg, calib, frames, bx, bs, bb)


@pytest.mark.parametrize("kw", [dict(), dict(method="TM_DE", flip=True), dict(method="base", fma_mode=False),
                                dict(warp=True, vid_pad=5, conn=4)])
def test_screen_equals_dense_and_oracle(oracle, kw):
    (pair, pair_active), (on, on_active), (off, off_active) = _run_both(synth.SynthSpec(**kw), 6, 1000)[0]
    assert pair_active == 2.0 and on_active == 1.0 and off_active == 0.0
    assert diff_results(on, off) == [] and on.checksum() == off.checksum()
    assert diff_results(pair, off) == [] and pair.checksum() == off.checksum()


def test_screen_vs_oracle_mixed_template_shapes(oracle):
    """Per-feature different template sizes: different anchors shift the Toeplitz band (dx, dy != 0), and the
    sparse exact kernel runs one launch per padded kernel width."""
    shapes = (((30, 30), (24, 28), (20, 16)), ((27, 30), (30, 22), (15, 17)))
    spec = synth.SynthSpec(tshapes=shapes)
    ((pair, a2), (on, a1), (off, a0)), (cfg, model, bkg, calib, frames, bx, bs, bb) = _run_both(spec, 4, 1001)
    assert a2 == 2.0 and a1 == 1.0
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    assert diff_results(pair, ref) == [] and diff_results(on, ref) == [] and diff_results(off, ref) == []


def test_screen_large_batch_property():
    """Size-independent property at benchmark scale: 700 device-rendered frames (three sub-batches), screen on
    and off give the same checksum of every result byte."""
    import torch

    spec = synth.SynthSpec()
    cfg, model, bkg, calib, _, _, _, _ = synth.make_problem(spec, 8, seed=1000)
    frames, bx, bs, bb = synth.make_video(spec, 700, 1234, "cuda", bkg)
    torch.cuda.synchronize()
    sums = []
    for screen in (2, 1, 0):
        det = _detector(cfg, model, bkg, calib, screen)
        r = det.detect_batch(frames, bx, bs, bb)
        sums.append((r.checksum(), int(r.n_bottom.sum()), int(r.n_side.sum()), int(r.match_n.sum())))
        det.close()
    assert sums[0] == sums[2] and sums[1] == sums[2]
    assert sums[0][1] > 1000


def test_screen_dense_threshold_and_degenerate_templates(oracle):
    """Stress the decision thresholds: (a) biases lowered so that a large share of all outputs is positive (many
    survivors, overflow allowed), (b) an all-zero template with rho = 0 (every score is exactly -0.0 -> no
    detection, quantisation scale degenerate).  Outputs placed exactly on the screen's thresholds, and scores of exactly 0
    and the smallest subnormal, are in tests/test_gpu_designed_frames.py."""
    def lower_rho(m):
        return Model(w=m.w, rho=[[r * 0.25 for r in row] for row in m.rho])

    ((pair, a2), (on, a1), (off, _)), _ = _run_both(synth.SynthSpec(), 3, 1002, model_edit=lower_rho, allow_overflow=True)
    assert a2 == 2.0 and a1 == 1.0
    # overflowing lists keep an unspecified subset of detections; compare only frames without overflow
    for got in (pair, on):
        ok = (got.flags == 0) & (off.flags == 0)
        assert np.array_equal(got.flags != 0, off.flags != 0)
        for name in got.ARRAYS:
            assert np.array_equal(getattr(got, name)[ok], getattr(off, name)[ok]), name

    def zero_paw(m):
        w = [[a.copy() for a in row] for row in m.w]
        w[0][0][:] = 0.0
        rho = [list(row) for row in m.rho]
        rho[0][0] = 0.0
        return Model(w=w, rho=rho)

    ((pair, a2), (on, a1), (off, _)), (cfg, model, bkg, calib, frames, bx, bs, bb) = _run_both(synth.SynthSpec(), 3, 1002, model_edit=zero_paw)
    assert a2 == 2.0 and a1 == 1.0 and diff_results(on, off) == [] and diff_results(pair, off) == []
    assert int(on.n_bottom[:, 0].sum()) == 0
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    assert diff_results(pair, ref) == []


def test_screen_large_templates_digit_split_and_dense_fallback(oracle):
    """40x40 templates: one template's Toeplitz operand no longer fits next to another's, so the CTA-pair kernel
    runs one template per job (hi digits in CTA 0, lo digits in CTA 1) while the single-CTA screen falls back to
    the dense kernel.  64x64 templates fit neither: every mode runs the dense exact kernel.  Results never change."""
    shapes = (((40, 40), (40, 40), (40, 40)), ((40, 40), (40, 40), (40, 40)))
    ((pair, a2), (on, a1), (off, a0)), (cfg, model, bkg, calib, frames, bx, bs, bb) = _run_both(synth.SynthSpec(tshapes=shapes), 2, 1000)
    assert a2 == 2.0 and a1 == 0.0 and a0 == 0.0
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    assert diff_results(pair, ref) == [] and diff_results(on, ref) == []
    shapes = (((64, 64), (64, 64), (64, 64)), ((64, 64), (64, 64), (64, 64)))
    ((pair, a2), (on, a1), (off, a0)), (cfg, model, bkg, calib, frames, bx, bs, bb) = _run_both(synth.SynthSpec(tshapes=shapes), 2, 1000)
    assert a2 == 0.0 and a1 == 0.0 and a0 == 0.0
    assert diff_results(pair, off) == []


def test_screen_config5_upsampled_60x60(oracle):
    """SURVEY config 5 (800x3400 frames, 60x60 templates, boxes 800 x 470 / 300): the pair kernel runs three
    digit-split jobs per view with a two-stage window ring and two y-tile pairs; bit-exact vs dense and oracle."""
    spec = synth.SynthSpec(scale=2, det_cap=8192, cand_cap=128, match_cap=512)
    ((pair, a2), (on, a1), (off, a0)), (cfg, model, bkg, calib, frames, bx, bs, bb) = _run_both(spec, 2, 1000, allow_overflow=True)
    assert a2 == 2.0 and a0 == 0.0
    assert diff_results(pair, off) == []
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    assert diff_results(pair, ref) == []


@pytest.mark.parametrize("kw,n,sub", [(dict(), 40, 16), (dict(method="TM_DE", flip=True), 9, 4),
                                      (dict(tshapes=(((30, 30), (24, 28), (20, 16)), ((27, 30), (30, 22), (15, 17)))), 7, 3)])
def test_screen2_job_layouts_are_equivalent(oracle, kw, n, sub):
    """k_screen2's job layouts -- tail planes sharing the paw + snout operand (N = 192, N = 128 right of the tail box) and
    y tiles stacked over the frames of a sub-batch (tiles straddle frames; ragged last tile) -- never change a result:
    all four combinations equal the oracle bit for bit."""
    from locomouse_cpp_b200.api import Detector

    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(synth.SynthSpec(**kw), n, seed=1003)
    frames = frames.numpy()
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    seen = set()
    for layout in (3, 2, 1, 0):
        det = Detector(cfg, model, bkg, calib, device=0)
        det.set_option("screen", 2)
        det.set_option("screen_layout", layout)
        det.set_option("subbatch", sub)
        got = det.detect_batch(frames, bx, bs, bb)
        assert det.info("screen_active") == 2.0
        seen.add((det.info("screen2_merged"), det.info("screen2_stacked")))
        det.close()
        assert diff_results(got, ref) == [], f"layout {layout}"
    assert (0.0, 0.0) in seen and len(seen) >= 3   # the layouts were really different


@pytest.mark.parametrize("seed", list(range(1, 37)))
def test_screen2_random_geometries_equal_oracle(oracle, seed, monkeypatch):
    """Random geometries for the CTA-pair screen's tiling: image / box sizes (boxes lower than one 128-row tile so that stacked
    tiles span several frames, and taller than 256 rows so that a frame needs two tile pairs), tail boxes whose width is
    not a multiple of the 32-column tile, template shapes that differ per feature and view, odd sub-batch sizes.  Every
    result byte equals the oracle for the default layout and with merging / stacking off.  The contexts run in guard mode
    (LM_GUARD: every scratch allocation between two pattern-filled 4 kB regions; compute-sanitizer is closed on the pool), and
    no kernel may have written outside its allocations."""
    from locomouse_cpp_b200.api import Detector

    monkeypatch.setenv("LM_GUARD", "1")
    rng = np.random.Generator(np.random.PCG64(9000 + seed))
    side_h = int(rng.choice([60, 96, 140, 165, 300]))
    bottom_h = int(rng.choice([70, 120, 235, 280]))
    bb_w = int(rng.choice([150, 250, 400, 430]))
    n_cols = int(bb_w * rng.uniform(1.6, 3.0)) & ~3
    tsh = lambda: (int(rng.integers(8, 31)), int(rng.integers(8, 31)))
    shapes = tuple(tuple(tsh() for _ in range(3)) for _ in range(2))
    method = str(rng.choice(["TM", "TM_DE"]))
    # seeds above 6 (the memory-safety fuzz that used to live in tools/fuzz_geometries.py only) also draw a warped calibration
    # (the gather tiers of k_prep), the connectivity, the stream count and the base method
    extra = dict(warp=bool(rng.integers(0, 2)), conn=int(rng.choice([4, 8]))) if seed > 6 else {}
    if seed > 6 and rng.integers(0, 3) == 0:
        method = "base"
    spec = synth.SynthSpec(method=method, n_rows=side_h + bottom_h, n_cols=n_cols, side_h=side_h, bb_w=bb_w,
                           bb_h_side_tm=max(40, side_h - 15), tshapes=shapes, mouse_scale=min(1.0, bb_w / 400, bottom_h / 235, side_h / 165),
                           flip=bool(rng.integers(0, 2)), cand_cap=128, match_cap=1024, **extra)
    n = int(rng.integers(5, 12))
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=1000 + seed)
    frames = frames.numpy()
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    for layout in (3, 0):
        det = Detector(cfg, model, bkg, calib, device=0)
        det.set_option("screen_layout", layout)
        det.set_option("subbatch", int(rng.integers(2, 8)))
        if seed > 6:
            det.set_option("streams", int(rng.integers(1, 5)))
        got = det.detect_batch(frames, bx, bs, bb, allow_overflow=True)
        active = det.info("screen_active")
        regions, violated = det.info("guard_regions"), det.info("guard_violations")
        det.close()
        assert regions > 20 and violated == 0.0, f"seed {seed}, layout {layout}: {violated} guard bytes overwritten"
        assert active >= 1.0, "the screen should handle templates up to 30 x 30"
        assert diff_results(got, ref) == [], f"seed {seed}, layout {layout}: side_h {side_h}, bottom_h {bottom_h}, bb_w {bb_w}, shapes {shapes}"


@pytest.mark.gpu
def test_guard_regions_stay_intact_on_the_benchmark_geometry(oracle, monkeypatch):
    """Config 1's geometry, several sub-batches on four streams, the dense fallback and the single-CTA screen as well: no kernel
    of the detection path writes outside its scratch allocations (guard mode, see lm_api.cu), and a deliberate overwrite of a
    guard region is noticed."""
    from locomouse_cpp_b200.api import Detector

    monkeypatch.setenv("LM_GUARD", "1")
    spec = synth.SynthSpec()
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 70, seed=1234)
    frames = frames.numpy()
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    for screen in (2, 1, 0):
        det = Detector(cfg, model, bkg, calib, device=0)
        det.set_option("screen", screen)
        det.set_option("subbatch", 16)
        got = det.detect_batch(frames, bx, bs, bb)
        violated = det.info("guard_violations")
        control = det.info("guard_selftest")          # three guard bytes overwritten on purpose, counted, restored
        again = det.info("guard_violations")
        det.close()
        assert violated == 0.0, f"screen={screen}: {violated} guard bytes overwritten"
        assert control == 3.0 and again == 0.0
        assert diff_results(got, ref) == []
