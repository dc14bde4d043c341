"""One context's device memory (lm_api.cu): every buffer an entry point uses is an allocation of the context, between guard
regions in guard mode, counted in lm_get_info("device_allocs") and kept for the next call.  On one context created with
LM_GUARD=1, a PNG decode, a detection call, the three pass-1 entry points from host and from device frames (with the
global-memory labelling forced by LM_BBOX_RUNCAP=16) and both cost builders give the results of a context without guard
mode, and no kernel writes outside its buffers; the first pass-1 and cost-builder calls add guard regions; a repeated round
allocates nothing, and a smaller geometry after a larger one runs in the grown allocations.  Needs a B200: pytest -m gpu."""
import numpy as np
import pytest

from _png_avi import make_png
from locomouse_cpp_b200 import synth
from locomouse_cpp_b200.types import Results, bb_base_params, bb_de_params, bb_tm_params, diff_results, location_priors, pairwise_params

pytestmark = pytest.mark.gpu

PRIOR_ROWS = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
              (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0)]


def _disk(r):
    y, x = np.mgrid[-r:r + 1, -r:r + 1]
    h = ((x * x + y * y) <= (r + 0.5) ** 2).astype(np.float64)
    return (h / h.sum()).astype(np.float32)


def _problem(spec, n, seed):
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=seed)
    frames = frames.numpy()
    pngs = [make_png(f) for f in frames]
    offs = np.concatenate([[0], np.cumsum([len(p) for p in pngs])]).astype(np.int64)
    return dict(spec=spec, setup=(cfg, model, bkg, calib), frames=frames, boxes=(bx, bs, bb), payload=np.frombuffer(b"".join(pngs), np.uint8),
                offs=offs)


def _round(det, pb, regions):
    """Every entry point once on problem `pb`.  `regions` receives guard_regions after the detection call and after the first
    pass-1 call of each class and the cost builders."""
    import torch

    spec, cfg, frames = pb["spec"], pb["setup"][0], pb["frames"]
    out = {"decoded": det.decode_png(pb["payload"], pb["offs"]).cpu().numpy()}
    res = det.detect_batch(frames, *pb["boxes"], allow_overflow=True)
    out["detect"] = res
    regions.append(det.info("guard_regions"))
    tm = bb_tm_params(cfg, _disk(5), side_h=spec.side_h, side_threshold=40, min_pixel_count=25, sums_as_float=0)
    for src, f in (("host", frames), ("device", torch.from_numpy(frames).cuda(det.device))):
        out["tm_de", src] = det.bounding_box_tm_de(f, bb_de_params(cfg, side_h=spec.side_h))
        regions.append(det.info("guard_regions"))
        out["base", src] = det.bounding_box_base(f, bb_base_params(cfg, side_h=spec.side_h, sums_as_float=0))
        regions.append(det.info("guard_regions"))
        out["tm", src] = det.bounding_box_tm(f, tm)
        regions.append(det.info("guard_regions"))
    pri, pw = location_priors(PRIOR_ROWS), pairwise_params(cfg.bb_w, cfg.bb_h_bottom)
    for feat in range(2):
        out["unary", feat] = det.unary_costs(res, feat, cfg.bb_w, cfg.bb_h_bottom, pri)
        out["pairwise", feat] = det.pairwise_costs(res, feat, pw)
    regions.append(det.info("guard_regions"))
    return out


def _check(got, want):
    assert got.keys() == want.keys()
    for key, w in want.items():
        g = got[key]
        if isinstance(w, Results):
            assert diff_results(g, w) == [], key
            continue
        for a, b in zip(g if isinstance(g, tuple) else (g,), w if isinstance(w, tuple) else (w,)):
            assert a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes(), key


def test_every_buffer_is_guarded_counted_and_kept(monkeypatch):
    from locomouse_cpp_b200.api import Detector

    monkeypatch.setenv("LM_BBOX_RUNCAP", "16")
    small = _problem(synth.SynthSpec(method="TM"), 24, seed=5100)
    big = _problem(synth.SynthSpec(method="TM", n_rows=480, n_cols=1900), 24, seed=5200)
    monkeypatch.delenv("LM_GUARD", raising=False)
    plain = Detector(*small["setup"], device=0)
    try:
        want_small = _round(plain, small, [])
        assert np.array_equal(want_small["decoded"], small["frames"])
        plain.configure(*big["setup"])
        want_big = _round(plain, big, [])
    finally:
        plain.close()

    monkeypatch.setenv("LM_GUARD", "1")
    det = Detector(*small["setup"], device=0)
    try:
        regions = []
        _check(_round(det, small, regions), want_small)
        # the first call of each pass-1 class and the cost builders allocate guarded buffers; the device-frame calls reuse them
        first = regions[:4] + regions[-1:]
        assert all(b > a for a, b in zip(first, first[1:])), f"guard regions {regions}"
        assert regions[4:7] == [regions[3]] * 3, f"guard regions {regions}"
        assert det.info("guard_violations") == 0.0
        allocs = det.info("device_allocs")
        _check(_round(det, small, []), want_small)
        assert det.info("device_allocs") == allocs, "a repeated round must reuse every allocation"
        det.configure(*big["setup"])
        _check(_round(det, big, []), want_big)
        assert det.info("guard_violations") == 0.0
        allocs = det.info("device_allocs")
        det.configure(*small["setup"])
        _check(_round(det, small, []), want_small)
        assert det.info("device_allocs") == allocs, "a smaller geometry must run in the grown allocations"
        assert det.info("guard_violations") == 0.0
        assert det.info("guard_selftest") == 3.0
        assert det.info("guard_violations") == 0.0
    finally:
        det.close()
