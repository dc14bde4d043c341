"""The plain references of tests/_pass1_designs.py against the oracle on every designed pass-1 frame, and every design against
what it claims to reach.  CPU only; the device side is tests/test_gpu_pass1_stages.py."""
import numpy as np
import pytest

import _pass1_designs as P
from _pass1_designs import base_params, de_params, problem, tm_params

TM = P.tm_designs()
BASE = P.base_designs()
DE = P.de_designs()


@pytest.mark.parametrize("d", TM, ids=[d.name for d in TM])
def test_tm_references_equal_oracle(oracle, d):
    """Every stage of the numpy reference equals the oracle's (oracle.mouse_box_tm on the side view, oracle.filter2d_u8 on
    the opened image) and the end-to-end limits through the front end; the binary stage is the design's pattern."""
    frame = d.frame()
    assert 0.01 < d.pattern.mean() < 0.99
    cfg, model, bkg, calib = problem(frame.shape)
    for conn in (4, 8):
        st = P.tm_stages(d, conn)
        bbx, lims, ost = oracle.mouse_box_tm(frame, d.disk, threshold=3, min_pixel_count=d.min_count, min_pixel_visible=d.min_vis,
                                             conn=conn, sums_as_float=d.as_float)
        assert np.array_equal(ost["binary"], d.binary())
        assert np.array_equal(ost["opened"], st["opened"]), conn
        assert np.array_equal(ost["filtered"], st["filtered"]), conn
        assert np.array_equal(oracle.filter2d_u8(st["opened"], d.disk), st["filtered"])
        assert np.array_equal(ost["row_sums"], st["sums"]), conn
        assert tuple(lims) == st["lims"] and bbx == float(st["lims"][1])
        import dataclasses

        raw, ol = oracle.bounding_box_tm(dataclasses.replace(cfg, conn=conn), bkg, calib, frame[None], tm_params(cfg, d))
        assert tuple(ol[0]) == st["lims"] and raw[0] == float(st["lims"][1])
    assert st["filtered"].max() <= 1


@pytest.mark.parametrize("d", TM, ids=[d.name for d in TM])
def test_tm_designs_reach_their_claims(d):
    got = {c: max(P.measure_tm(d, conn)[c] for conn in (4, 8)) for c in d.claims}
    assert all(v > 0 for v in got.values()), got


@pytest.mark.parametrize("d", BASE, ids=[d.name for d in BASE])
def test_base_references_equal_oracle(oracle, d):
    """Binary image through the front end, median >= 3 against cv2.medianBlur on the zero-padded image, largest components
    against oracle.largest_region, limits against oracle.bounding_box_base."""
    import dataclasses

    frame = d.frame()
    cfg, model, bkg, calib = problem(frame.shape)
    I, _ = oracle.preprocess(dataclasses.replace(cfg, imadjust=False), bkg, calib, frame)
    assert np.array_equal((I >= 3).astype(np.uint8), d.pattern)
    st = P.base_stages(d, 8)
    if d.k > 1:
        cv2 = pytest.importorskip("cv2")
        h = d.k // 2
        pad = np.pad(d.frame(), h)
        med = cv2.medianBlur(pad, d.k)[h:-h, h:-h]
        assert np.array_equal((med >= 3).astype(np.uint8), st["major"])
    for conn in (4, 8):
        st = P.base_stages(d, conn)
        for (x, y, w, h) in (d.side, d.bottom):
            view = st["major"][y:y + h, x:x + w]
            assert np.array_equal((oracle.largest_region(view, conn) != 0).astype(np.uint8), P.largest(view, conn)), conn
        _, ol = oracle.bounding_box_base(dataclasses.replace(cfg, conn=conn), bkg, calib, frame[None], base_params(cfg, d))
        assert np.array_equal(ol[0], st["lims"]), conn


@pytest.mark.parametrize("d", BASE, ids=[d.name for d in BASE])
def test_base_designs_reach_their_claims(d):
    got = {c: max(P.measure_base(d, conn)[c] for conn in (4, 8)) for c in d.claims}
    assert all(v > 0 for v in got.values()), got


def test_base_tie_breaks_differ_between_views_and_connectivities():
    """The tie design's winners are not the first components the scan meets in every case: a reversed tie rule changes
    its sums."""
    d = next(d for d in BASE if d.name == "equal_areas")
    for conn in (4, 8):
        st = P.base_stages(d, conn)
        x, y, w, h = d.side
        lab, n = P.ndimage.label(st["major"][y:y + h, x:x + w], P.STRUCT[conn])
        areas = np.bincount(lab.ravel())[1:]
        tied = np.nonzero(areas == areas.max())[0] + 1
        assert tied.size >= 2
        sums = [(lab == t).sum(axis=0) for t in tied]
        assert not np.array_equal(sums[0], sums[-1])


@pytest.mark.parametrize("d", DE, ids=[d.name for d in DE])
def test_de_references_equal_oracle(oracle, d):
    frame = d.frame()
    cfg, model, bkg, calib = problem(frame.shape)
    st = P.de_stages(d)
    _, raw, ol = oracle.bounding_box_tm_de(cfg, bkg, calib, frame[None], de_params(cfg, d))
    assert tuple(ol[0]) == st["lims"]
    assert raw[0] == min(d.pattern.shape[1] - 1, st["lims"][1] * 1.1)
    got = P.measure_de(d)
    assert all(got[c] > 0 for c in d.claims), got


def test_first_last_reads_integer_sums_as_floats():
    s = np.array([0, 765, 0, 255 * 20], np.int32)
    assert P.first_last(s, 1, False) == (1, 3)
    assert P.first_last(s, 765, False) == (1, 3) and P.first_last(s, 766, False) == (3, 0)
    assert P.first_last(s, 1, True) == (-1, -1) and P.first_last(s, 0, True) == (0, 3)
