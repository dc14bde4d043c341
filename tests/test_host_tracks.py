"""The driver stages after the per-frame loop (main.cpp:85-91): computeBottomTracks, computeSideTracks, exportResults ->
output_<stem>.yml (SURVEY 8b caveat / 8f-3 / 8f-4).

CPU: the side-view transition builder equals the REFERENCE's own pairwisePotential_SideView (compiled from
/root/reference) on committed vectors and fresh inputs; the YAML writer is byte-identical to cv2.FileStorage.
GPU (-m gpu): the C++ driver (reference call sequence on files) writes an output_<stem>.yml whose matrices equal the
tracker run on the ORACLE's candidates (tests/_tracks_model.py; tracker = the reference's compiled match2nd when
oracle/_ref is present), and whose bytes equal what the real OpenCV writes for those matrices."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _tracks_model as tm  # noqa: E402
from test_match2nd import _host, _ref, REF_LIB  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "reference_side_transitions.npz")


def side_cases(seed=77, n=40):
    rng = np.random.Generator(np.random.PCG64(seed))
    cases = []
    for it in range(n):
        ni, nj = int(rng.integers(0, 5)), int(rng.integers(0, 5))
        if it == 0:
            ni, nj = 0, 3
        if it == 1:
            ni, nj = 3, 0
        side_h = int(rng.choice([150, 165, 300]))
        spacing = int(rng.choice([20, 20, 35]))
        c = int(rng.integers(10, side_h - 10))
        zi = [int(np.clip(c + rng.integers(-20, 21), 0, side_h - 1)) for _ in range(ni)]
        zj = [int(np.clip(c + rng.integers(-20, 21), 0, side_h - 1)) for _ in range(nj)]
        cases.append(dict(zi=zi, zj=zj, lowest=float(side_h - 1 - spacing // 2), spacing=float(spacing),
                          nong=(side_h - spacing) // spacing + 1, max_disp=float(rng.choice([15, 15, 40])),
                          alpha=float(rng.choice([100.0, 100.0, 0.0, 0.1])), occ=float(rng.choice([1e-2, 1e-2, 0.0]))))
    return cases


def _side(lib, name, c):
    return tm.side_transitions(lib, name, c["zi"], c["zj"], c["lowest"], c["spacing"], c["nong"], c["max_disp"], c["alpha"], c["occ"])


def _same(a, b):
    return (a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
            and np.array_equal(a[4].view(np.uint64), b[4].view(np.uint64)))


def _ref_nms():
    p = os.path.join(os.path.dirname(REF_LIB), "libref_nms.so")
    if _ref() is None or not os.path.exists(p):
        return None
    return C.CDLL(p)


def make_golden():
    R = _ref_nms()
    assert R is not None
    out = {}
    for i, c in enumerate(side_cases()):
        r = _side(R, "ref_pairwise_potential_side", c)
        out[f"dims_{i}"] = np.array(r[:2])
        out[f"jc_{i}"], out[f"ir_{i}"], out[f"pr_{i}"] = r[2], r[3], r[4]
    np.savez_compressed(GOLD, **out)


def test_side_view_transitions_equal_reference_golden():
    H = _host()
    G = np.load(GOLD)
    stored = 0
    for i, c in enumerate(side_cases()):
        got = _side(H, "lmh_pairwise_potential_side", c)
        want = (int(G[f"dims_{i}"][0]), int(G[f"dims_{i}"][1]), G[f"jc_{i}"], G[f"ir_{i}"], G[f"pr_{i}"])
        assert _same(got, want), i
        stored += len(want[3])
    assert stored > 200


def test_side_view_transitions_equal_reference_fresh():
    R = _ref_nms()
    if R is None:
        pytest.skip("reference library not built (no LocoMouse_cpp checkout, see oracle/reference_nms.py); golden vectors cover it")
    H = _host()
    for c in side_cases(seed=123, n=150):
        assert _same(_side(H, "lmh_pairwise_potential_side", c), _side(R, "ref_pairwise_potential_side", c))


def _yaml_write(path, items):
    H = _host()
    names = "\n".join(k for k, _ in items).encode()
    rows = np.array([m.shape[0] for _, m in items], np.int32)
    cols = np.array([m.shape[1] for _, m in items], np.int32)
    data = np.concatenate([np.ascontiguousarray(m, np.int32).reshape(-1) for _, m in items])
    p = lambda a: C.c_void_p(a.ctypes.data)
    H.lmh_yaml_write.restype = C.c_int
    assert H.lmh_yaml_write(str(path).encode(), names, len(items), p(rows), p(cols), p(data)) == 0


def test_yaml_writer_is_byte_identical_to_opencv(tmp_path):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.Generator(np.random.PCG64(3))
    items = [(f"paw_tracks{k}", rng.integers(-1, 1700, (int(rng.integers(1, 200)), 3)).astype(np.int32)) for k in range(4)]
    items.append(("snout_tracks0", -np.ones((57, 3), np.int32)))
    items.append(("tracks_tail", rng.integers(-1, 400, (3, 15 * 23)).astype(np.int32)))
    _yaml_write(tmp_path / "ours.yml", items)
    fs = cv2.FileStorage(str(tmp_path / "cv.yml"), cv2.FILE_STORAGE_WRITE)
    for k, m in items:
        fs.write(k, m)
    fs.release()
    assert (tmp_path / "ours.yml").read_bytes() == (tmp_path / "cv.yml").read_bytes()
    fs = cv2.FileStorage(str(tmp_path / "ours.yml"), cv2.FILE_STORAGE_READ)
    for k, m in items:
        assert np.array_equal(fs.getNode(k).mat(), m)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["TM", "TM_DE"])
def test_driver_track_file_equals_tracker_on_oracle_candidates(tmp_path, oracle, method):
    cv2 = pytest.importorskip("cv2")
    from locomouse_cpp_b200 import synth
    from locomouse_cpp_b200.types import location_priors, pairwise_params
    from test_host_cpp import _build_driver, write_problem_files

    exe = _build_driver()
    spec = synth.SynthSpec(method=method)
    n = 40
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, n, seed=1000)
    frames = frames.numpy()
    ref = oracle.detect(cfg, model, bkg, calib, frames, bx, bs, bb, n_threads=8)
    assert ref.rc == 0
    rows = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
            (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0), (0.95, 0.5, 0.6, 0.5, 1.0, 0.0, 1.0)]
    flat = ", ".join(repr(float(v)) for r in rows for v in r)
    write_problem_files(tmp_path, cfg, model, bkg, calib, frames, bx, bs, bb, spec.side_h,
                        extra_cfg=f"batch_frames: 16\nlocation_prior: [{flat}]\nmax_displacement_bottom: 40\nmax_displacement_side: 25\ntracker_threads: 3\n")
    meth = {"TM": "1", "TM_DE": "2"}[method]
    p = subprocess.run([exe, meth, str(tmp_path / "config.yml"), str(tmp_path / "video.lmv"), str(tmp_path / "bkg.lmi"),
                        str(tmp_path / "model.lmm"), str(tmp_path / "calib.lmc"), "R", str(tmp_path)], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    # ---- the same stages on the oracle's candidates ----------------------------------------------------------------
    pri = [location_priors(rows[:4]), location_priors(rows[4:])]
    P = pairwise_params(cfg.bb_w, cfg.bb_h_bottom, max_displacement=40)
    nong = P.ong_w * P.ong_h
    unary, trans = [[], []], [[], []]
    for feat in range(2):
        for f in range(n):
            c = ref.candidates_bottom(f, feat)
            unary[feat].append(oracle.unary_cost_box(c, cfg.bb_w, cfg.bb_h_bottom, pri[feat]).reshape(len(c), 4 if feat == 0 else 1))
            if f:
                _r, _c, jc, ir, pr = oracle.pairwise_potential(ref.candidates_bottom(f - 1, feat), c, P)
                trans[feat].append((jc, ir, pr))
    paw, snout = tm.bottom_tracks(unary[0], trans[0], unary[1], trans[1], nong)
    p22 = [[ref.p22d(f, feat) for f in range(n)] for feat in range(2)]
    paw_side = tm.side_tracks(paw, p22[0], cfg.bb_h_side, max_disp_side=25)
    snout_side = tm.side_tracks(snout, p22[1], cfg.bb_h_side, max_disp_side=25)
    want = [(f"paw_tracks{k}", m) for k, m in enumerate(tm.export_points(paw, paw_side, p22[0], bx, bs, bb, cfg.bb_w, cfg.bb_h_bottom, cfg.bb_h_side))]
    want += [("snout_tracks0", tm.export_points(snout, snout_side, p22[1], bx, bs, bb, cfg.bb_w, cfg.bb_h_bottom, cfg.bb_h_side)[0])]
    want += [("tracks_tail", tm.export_tail(ref.tail[:n], bx, bs, bb, cfg.bb_w, cfg.bb_h_bottom, cfg.bb_h_side))]
    # ---- what the driver wrote, read back by the real OpenCV ----------------------------------------------------------
    out = tmp_path / "output_video.yml"
    assert out.exists(), p.stdout
    fs = cv2.FileStorage(str(out), cv2.FILE_STORAGE_READ)
    tracked = 0
    for k, m in want:
        got = fs.getNode(k).mat()
        assert got is not None and np.array_equal(got, m), k
        tracked += int((m[:, 0] >= 0).sum()) if k != "tracks_tail" else 0
    assert tracked > n  # the tracks follow real candidates, not only occlusion nodes
    fs2 = cv2.FileStorage(str(tmp_path / "cv.yml"), cv2.FILE_STORAGE_WRITE)
    for k, m in want:
        fs2.write(k, m)
    fs2.release()
    assert out.read_bytes() == (tmp_path / "cv.yml").read_bytes()


if __name__ == "__main__":
    make_golden()
    print("wrote", GOLD)
