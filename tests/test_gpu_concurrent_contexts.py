"""Several contexts on one device, driven from their own host threads, and re-configuration that keeps a context's device
allocations (lm_api.cu: per-context stream synchronisation, retained scratch blocks, lm_get_info("device_allocs")).  Every
result equals the same call made alone, and in guard mode no kernel writes outside its (retained) allocations."""
import threading

import pytest

from locomouse_cpp_b200 import synth
from locomouse_cpp_b200.types import diff_results

pytestmark = pytest.mark.gpu


def _problems():
    """Three different problems: methods, backgrounds, geometries, sides."""
    specs = [synth.SynthSpec(method="TM", flip=False),
             synth.SynthSpec(method="TM_DE", flip=True),
             synth.SynthSpec(method="base", n_rows=300, n_cols=1200, side_h=130, bb_w=320, bb_h_side_tm=115, mouse_scale=0.7)]
    out = []
    for i, spec in enumerate(specs):
        cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, 40 + 13 * i, seed=3000 + 17 * i)
        out.append((cfg, model, bkg, calib, frames.numpy(), bx, bs, bb))
    return out


def _alone(p):
    from locomouse_cpp_b200.api import Detector

    cfg, model, bkg, calib, frames, bx, bs, bb = p
    det = Detector(cfg, model, bkg, calib, device=0)
    try:
        return det.detect_batch(frames, bx, bs, bb, allow_overflow=True)
    finally:
        det.close()


def test_three_contexts_from_three_threads_equal_the_calls_alone(monkeypatch):
    from locomouse_cpp_b200.api import Detector

    monkeypatch.setenv("LM_GUARD", "1")
    probs = _problems()
    want = [_alone(p) for p in probs]
    dets = [Detector(*p[:4], device=0) for p in probs]
    got = [[None] * 3 for _ in probs]
    errors = []
    start = threading.Barrier(len(probs))

    def run(i):
        try:
            cfg, model, bkg, calib, frames, bx, bs, bb = probs[i]
            start.wait()
            for rep in range(3):   # host frames, device-resident frames, host frames again
                if rep == 1:
                    import torch
                    frames_d = torch.from_numpy(frames).cuda(0)
                    got[i][rep] = dets[i].detect_batch(frames_d, bx, bs, bb, allow_overflow=True)
                else:
                    got[i][rep] = dets[i].detect_batch(frames, bx, bs, bb, allow_overflow=True)
        except Exception as e:  # noqa: BLE001 - reported below
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(probs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    try:
        assert not errors, errors
        for i in range(len(probs)):
            for rep in range(3):
                assert diff_results(got[i][rep], want[i]) == [], f"problem {i}, repetition {rep}"
            assert dets[i].info("guard_violations") == 0.0
    finally:
        for d in dets:
            d.close()


def test_reconfigure_keeps_allocations_and_results(monkeypatch):
    from locomouse_cpp_b200.api import Detector

    monkeypatch.setenv("LM_GUARD", "1")
    spec = synth.SynthSpec(method="TM")
    a = synth.make_problem(spec, 50, seed=4000)
    b = synth.make_problem(spec, 50, seed=4100)    # same geometry, another background / video
    a = a[:4] + (a[4].numpy(),) + a[5:]
    b = b[:4] + (b[4].numpy(),) + b[5:]
    big_spec = synth.SynthSpec(method="TM", n_rows=480, n_cols=1900, side_h=190, bb_w=440, bb_h_side_tm=175, mouse_scale=1.0)
    c = synth.make_problem(big_spec, 70, seed=4200)
    c = c[:4] + (c[4].numpy(),) + c[5:]
    det = Detector(*a[:4], device=0)
    try:
        det.detect_batch(*a[4:], allow_overflow=True)
        n0 = det.info("device_allocs")
        assert n0 > 0
        det.configure(*b[:4])
        got_b = det.detect_batch(*b[4:], allow_overflow=True)
        assert det.info("device_allocs") == n0, "a video of the same geometry must reuse every allocation"
        assert diff_results(got_b, _alone(b)) == []
        assert det.info("guard_violations") == 0.0
        det.configure(*c[:4])
        got_c = det.detect_batch(*c[4:], allow_overflow=True)
        assert det.info("device_allocs") > n0, "a larger geometry grows the allocations"
        assert diff_results(got_c, _alone(c)) == []
        det.configure(*a[:4])   # back to the smaller geometry, in the grown blocks
        got_a = det.detect_batch(*a[4:], allow_overflow=True)
        assert diff_results(got_a, _alone(a)) == []
        assert det.info("guard_regions") > 0 and det.info("guard_violations") == 0.0
    finally:
        det.close()


def _in_threads(jobs):
    """Runs each job (a callable) in its own thread, all released at once; returns their results or raises the first error."""
    out, errors = [None] * len(jobs), []
    start = threading.Barrier(len(jobs))

    def run(i):
        try:
            start.wait()
            out[i] = jobs[i]()
        except Exception as e:  # noqa: BLE001 - reported below
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    return out


def test_concurrent_ffv1_decodes_with_different_work_memory(tmp_path):
    """Two contexts decode FFV1 at once: a cv2-written stream (its large context table puts the chains' work memory in global
    slots) and a hand-built small-model stream (work memory in shared memory), so the two launches ask for different dynamic
    shared memory.  The decoder's shared-memory limit is a property of the kernel on the device, set once; each decode equals
    VideoCapture."""
    cv2 = pytest.importorskip("cv2")
    import numpy as np
    from _ffv1_avi import encode_avi, read_avi_ffv1, write_cv2_ffv1
    from test_gpu_png_ingest import _detector

    rng = np.random.Generator(np.random.PCG64(11))
    big = rng.integers(0, 256, (24, 400, 640), dtype=np.uint8)
    small = rng.integers(0, 256, (13, 21, 31), dtype=np.uint8)
    want_big = write_cv2_ffv1(cv2, tmp_path / "big.avi", big)
    _, _, want_small = encode_avi(cv2, tmp_path / "small.avi", small)
    streams = [(read_avi_ffv1(tmp_path / "big.avi"), want_big), (read_avi_ffv1(tmp_path / "small.avi"), want_small)]
    dets = [_detector(*s[0][3][1:]) for s in streams]
    try:
        def job(k):
            (ex, payload, offs, _), want = streams[k]
            return lambda: [np.array_equal(dets[k].decode_ffv1(ex, payload, offs).cpu().numpy(), want) for _ in range(6)]

        assert _in_threads([job(0), job(1)]) == [[True] * 6, [True] * 6]
    finally:
        for d in dets:
            d.close()


def test_dense_correlation_from_two_threads_on_different_geometries():
    """The dense exact kernel (option screen = 0) needs per-view, per-geometry dynamic shared memory: two contexts of different
    geometries run it at once and give the results of the default path alone."""
    from locomouse_cpp_b200.api import Detector

    probs = [p for i, p in enumerate(_problems()) if i != 1]
    want = [_alone(p) for p in probs]
    dets = [Detector(*p[:4], device=0) for p in probs]
    try:
        for d in dets:
            d.set_option("screen", 0)

        def job(k):
            return lambda: [dets[k].detect_batch(*probs[k][4:], allow_overflow=True) for _ in range(2)]

        got = _in_threads([job(0), job(1)])
        for k in range(2):
            assert dets[k].info("screen_active") == 0.0
            for g in got[k]:
                assert diff_results(g, want[k]) == [], f"problem {k}"
    finally:
        for d in dets:
            d.close()
