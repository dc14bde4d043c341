"""Pass 1 on the device stage by stage (lm_debug_fetch items 4 .. 6) against the plain references of tests/_pass1_designs.py
on every designed frame, bit for bit: LocoMouse_TM's opened and filtered images and column sums, the base class's binary and
median images and four sum vectors, LocoMouse_TM_DE's column counts, and each method's limits.  Both connectivities; the
shared-memory labelling with the run capacity at the design's run count and the global-memory path one run below; host and
device frames; one pass in guard mode.  Needs a B200:  pytest -m gpu."""
import dataclasses

import numpy as np
import pytest

import _pass1_designs as P
from _pass1_designs import base_params, de_params, problem, tm_params

pytestmark = pytest.mark.gpu

TM = P.tm_designs()
BASE = P.base_designs()
DE = P.de_designs()


def _detector(d, conn):
    from locomouse_cpp_b200.api import Detector

    cfg, model, bkg, calib = problem(d.pattern.shape)
    cfg = dataclasses.replace(cfg, conn=conn)
    return cfg, Detector(cfg, model, bkg, calib, device=0)


def _frames(d, on_device):
    f = d.frame()[None]
    if on_device:
        import torch

        return torch.from_numpy(f).cuda()
    return f


def _fetch(det, what, frame=0):
    return det.debug_fetch(what, frame)[0]


def _diff(name, got, want):
    if np.array_equal(got, want):
        return []
    bad = np.argwhere(np.asarray(got) != np.asarray(want))
    return [f"{name}: {len(bad)} entries differ, first at {bad[0].tolist()}"]


def _check_tm(det, d, conn, frames):
    st = P.tm_stages(d, conn)
    raw, lims = det.bounding_box_tm(frames, tm_params(det.cfg, d))
    errs = _diff("opened", _fetch(det, 5), st["opened"]) + _diff("filtered", _fetch(det, 4), st["filtered"])
    errs += _diff("sums", _fetch(det, 6), st["sums"]) + _diff("lims", tuple(lims[0]), st["lims"])
    errs += _diff("bb_x", raw[0], float(st["lims"][1]))
    return errs


@pytest.mark.parametrize("conn", [4, 8])
def test_tm_stages_equal_reference(conn, monkeypatch):
    """Every TM design with the run capacity at the larger run count of the two labelled images (both stages on the
    shared-memory path, host frames) and one run below (the larger one on the global-memory path, device frames); then
    with min_pixel_count = 1, where the opened image is the binary image."""
    failures = []
    for d in TM:
        cfg, det = _detector(d, conn)
        try:
            st = P.tm_stages(d, conn)
            filt = st["filtered"]
            runs = max(P.run_count(st["binary"]), P.run_count(filt == filt[0, 0]))
            for cap, dev in ((runs, False), (runs - 1, True)):
                monkeypatch.setenv("LM_BBOX_RUNCAP", str(cap))
                failures += [f"{d.name} cap {cap}: {e}" for e in _check_tm(det, d, conn, _frames(d, dev))]
            monkeypatch.delenv("LM_BBOX_RUNCAP")
            d1 = dataclasses.replace(d, min_count=1)
            failures += [f"{d.name} min_count 1: {e}" for e in _check_tm(det, d1, conn, _frames(d, False))]
            assert np.array_equal(_fetch(det, 5), d.binary()), d.name
        finally:
            det.close()
    assert not failures, failures[:10]


def _check_base(det, d, conn, frames):
    st = P.base_stages(d, conn)
    _, lims = det.bounding_box_base(frames, base_params(det.cfg, d))
    errs = _diff("binary", _fetch(det, 4), st["binary"]) + _diff("median", _fetch(det, 5), st["major"])
    errs += _diff("sums", _fetch(det, 6), st["sums"]) + _diff("lims", lims[0], st["lims"])
    return errs


@pytest.mark.parametrize("conn", [4, 8])
def test_base_stages_equal_reference(conn, monkeypatch):
    """Every base-class design with the run capacity at the larger view's run count (k_bbb_cc) and one run below
    (k_bbb_cc_slow for that view)."""
    failures = []
    for d in BASE:
        cfg, det = _detector(d, conn)
        try:
            st = P.base_stages(d, conn)
            runs = max(P.run_count(st["major"][y:y + h, x:x + w]) for (x, y, w, h) in (d.side, d.bottom))
            for cap, dev in ((runs, False), (runs - 1, True)):
                monkeypatch.setenv("LM_BBOX_RUNCAP", str(cap))
                failures += [f"{d.name} cap {cap}: {e}" for e in _check_base(det, d, conn, _frames(d, dev))]
        finally:
            det.close()
    assert not failures, failures[:10]


@pytest.mark.parametrize("on_device", [False, True])
def test_de_counts_equal_reference(on_device):
    """Column counts of exactly min_count and one below, side views 65 (a partial 16-pixel segment) and 67 pixels wide (the
    kept differences stored byte by byte on alternate rows)."""
    failures = []
    for d in DE:
        cfg, det = _detector(d, 8)
        try:
            st = P.de_stages(d)
            _, raw, lims = det.bounding_box_tm_de(_frames(d, on_device), de_params(cfg, d))
            failures += [f"{d.name}: {e}" for e in _diff("counts", _fetch(det, 6), st["sums"]) + _diff("lims", tuple(lims[0]), st["lims"])]
            failures += [f"{d.name}: {e}" for e in _diff("bb_x", raw[0], min(d.pattern.shape[1] - 1, st["lims"][1] * 1.1))]
            with pytest.raises(ValueError):   # TM_DE keeps no bit images
                det.debug_fetch(4, 0)
        finally:
            det.close()
    assert not failures, failures[:10]


def test_guard_mode_and_chunks(monkeypatch):
    """Guard mode (every buffer between guard regions): a TM call of 300 frames (two chunks) and a base call leave every
    guard byte untouched; the items address frames of the last chunk only, and need no lm_detect_batch."""
    monkeypatch.setenv("LM_GUARD", "1")
    d = next(d for d in TM if d.name == "imfill_holes")
    cfg, det = _detector(d, 8)
    try:
        with pytest.raises(RuntimeError):   # no pass-1 call yet
            det.debug_fetch(6, 0)
        frames = np.repeat(d.frame()[None], 300, axis=0)
        st = P.tm_stages(d, 8)
        raw, lims = det.bounding_box_tm(frames, tm_params(cfg, d))
        assert (lims == np.array(st["lims"])).all()
        for f in (256, 299):
            assert np.array_equal(_fetch(det, 6, f), st["sums"])
            assert np.array_equal(_fetch(det, 4, f), st["filtered"])
        for f in (255, 300):
            with pytest.raises(ValueError):
                det.debug_fetch(6, f)
        assert det.info("guard_violations") == 0
    finally:
        det.close()
    d = next(d for d in BASE if d.name == "median_k3")
    cfg, det = _detector(d, 4)
    try:
        assert _check_base(det, d, 4, _frames(d, True)) == []
        assert det.info("guard_violations") == 0
    finally:
        det.close()
