"""Host tracker (SURVEY 8f-4, north_star "match2nd interface"): locomouse_cpp_b200/host/match2nd.cpp against the REFERENCE'S
OWN tracker (match2nd/match2nd.cpp + match2nd.h + MyMat.cpp compiled unchanged from /root/reference by `make -C oracle ref`
into oracle/_ref/libref_match2nd.so): identical label matrices on committed vectors the reference produced
(tests/golden/reference_match2nd.npz) and, where the reference library is present, on fresh random trellises; plus the
re-entrancy the reference lacks (its state is global): the same jobs on several threads give the serial answer."""
import ctypes as C
import os

import numpy as np
import pytest

from locomouse_cpp_b200.types import pairwise_params, location_priors
from oracle import oracle, reference_nms

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(HERE, "golden", "reference_match2nd.npz")
HOST_LIB = os.path.join(ROOT, "locomouse_cpp_b200", "host", "libmatch2nd_host.so")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libref_match2nd.so")
PRIOR_ROWS = [(0.8, 0.25, 0.5, 0.4, 1.0, 0.0, 0.5), (0.8, 0.75, 0.5, 0.4, 1.0, 0.5, 1.0), (0.3, 0.25, 0.4, 0.0, 0.6, 0.0, 0.5),
              (0.3, 0.75, 0.35, 0.0, 0.6, 0.5, 1.0)]


def _host():
    if not os.path.exists(HOST_LIB):
        import subprocess
        subprocess.run(["make", "-C", os.path.dirname(HOST_LIB), "libmatch2nd_host.so"], check=True, capture_output=True)
    return C.CDLL(HOST_LIB)


def _ref():
    if not os.path.exists(REF_LIB):
        if os.path.isdir(os.path.join(reference_nms.REF_ROOT, "match2nd")):
            reference_nms.make_ref()
        else:
            return None
    return C.CDLL(REF_LIB)


class Trellis:
    """Packed trellis: what lm_unary_costs / lm_pairwise_costs return, frame by frame."""

    def __init__(self, points, nong, n_loc, unary, trans):
        self.points, self.nong = points, nong
        self.n_loc = np.asarray(n_loc, np.int32)
        self.frames = len(n_loc)
        self.unary_off = np.zeros(self.frames + 1, np.int64)
        for f in range(self.frames):
            self.unary_off[f + 1] = self.unary_off[f] + int(n_loc[f]) * points
        self.unary = np.concatenate([np.asarray(u, np.float64).reshape(-1, order="F") for u in unary] + [np.zeros(1)])
        self.jc_off = np.zeros(max(self.frames - 1, 1), np.int64)
        self.nz_off = np.zeros(max(self.frames - 1, 1), np.int64)
        jc, ir, pr = [], [], []
        o_jc = o_nz = 0
        for f, (j, i, p) in enumerate(trans):
            self.jc_off[f], self.nz_off[f] = o_jc, o_nz
            jc.append(np.asarray(j, np.int32))
            ir.append(np.asarray(i, np.int32))
            pr.append(np.asarray(p, np.float64))
            o_jc += len(j)
            o_nz += len(i)
        self.jc = np.concatenate(jc + [np.zeros(1, np.int32)])
        self.ir = np.concatenate(ir + [np.zeros(1, np.int32)])
        self.pr = np.concatenate(pr + [np.zeros(1)])

    def args(self):
        p = lambda a: C.c_void_p(a.ctypes.data)
        return (self.frames, self.points, p(self.n_loc), p(self.unary), p(self.unary_off), self.nong, p(self.jc), p(self.jc_off),
                p(self.ir), p(self.pr), p(self.nz_off))


def run(lib, name, T, occ_cost, bam, perm):
    fn = getattr(lib, name)
    fn.restype = C.c_int
    perm = np.asarray(perm, np.int32)
    out = np.full((T.points, T.frames), 77, np.int32)
    fn(*T.args(), C.c_double(occ_cost), C.c_double(bam), C.c_void_p(perm.ctypes.data), C.c_void_p(out.ctypes.data))
    return out


def cost(lib, name, T, perm, labels):
    fn = getattr(lib, name)
    fn.restype = C.c_double
    perm = np.asarray(perm, np.int32)
    labels = np.ascontiguousarray(labels, np.int32)
    p = lambda a: C.c_void_p(a.ctypes.data)
    return fn(T.frames, T.points, p(T.n_loc), p(T.unary), p(T.unary_off), p(perm), p(labels))


def random_sparse_trellis(rng, frames, points, nong, max_loc, density, zero_unary=0.2):
    n_loc = rng.integers(0, max_loc + 1, frames)
    unary = []
    for f in range(frames):
        u = rng.uniform(0.0, 2.0, (int(n_loc[f]), points))
        u[rng.uniform(size=u.shape) < zero_unary] = 0.0
        unary.append(u)
    trans = []
    for f in range(frames - 1):
        cols, rows = int(n_loc[f]) + nong, int(n_loc[f + 1]) + nong
        jc, ir, pr = [0], [], []
        for c in range(cols):
            r = np.nonzero(rng.uniform(size=rows) < density)[0]
            ir += list(r)
            pr += list(rng.choice([0.001, 0.05, 0.1, 0.37, 1.0], len(r)) * rng.choice([1.0, 1.0, 0.5], len(r)))
            jc.append(len(ir))
        trans.append((jc, ir, pr))
    return Trellis(points, nong, n_loc, unary, trans)


def tracker_like_trellis(rng, frames, points, move=6.0):
    """Candidates that drift like paws + the oracle's own cost builders: the structure the tracker really sees."""
    bw, bh = 400, 235
    pw = pairwise_params(bw, bh)
    pw.grid_spacing = 60.0          # a small occlusion grid keeps the dense detour of the reference checker cheap
    pw.ong_w, pw.ong_h = 3, 2
    pri = location_priors(PRIOR_ROWS[:points])
    centres = rng.uniform([40, 30], [360, 200], (points, 2))
    cands = []
    for f in range(frames):
        centres += rng.normal(0, move, centres.shape)
        centres = np.clip(centres, [5, 5], [bw - 6, bh - 6])
        c = []
        for k in range(points):
            if rng.uniform() < 0.85:
                c.append((int(centres[k, 0] + rng.integers(-2, 3)), int(centres[k, 1] + rng.integers(-2, 3)), float(np.float32(rng.uniform(0.2, 2.5)))))
        for _ in range(int(rng.integers(0, 4))):
            c.append((int(rng.integers(0, bw)), int(rng.integers(0, bh)), float(np.float32(rng.uniform(0.05, 1.0)))))
        if rng.uniform() < 0.08:
            c = []
        cands.append(c)
    n_loc = [len(c) for c in cands]
    unary = [oracle.unary_cost_box(c, bw, bh, pri).reshape(len(c), points) for c in cands]
    trans = []
    for f in range(frames - 1):
        _r, _c, jc, ir, pr = oracle.pairwise_potential(cands[f], cands[f + 1], pw)
        trans.append((jc, ir, pr))
    return Trellis(points, pw.ong_w * pw.ong_h, n_loc, unary, trans)


def golden_cases():
    rng = np.random.Generator(np.random.PCG64(20261018))
    cases = []
    for it in range(36):
        points = int(rng.choice([1, 2, 4, 4]))
        if it % 3 == 0:
            T = tracker_like_trellis(rng, int(rng.integers(3, 40)), points)
        else:
            T = random_sparse_trellis(rng, int(rng.integers(2, 30)), points, int(rng.integers(1, 4)), int(rng.integers(1, 7)),
                                      float(rng.choice([0.15, 0.4, 0.8])))
        perm = list(rng.permutation(points))
        occ_cost, bam = (0.0, 0.0) if it % 4 else (float(rng.choice([0.0, 0.01])), float(rng.choice([0.0, 0.05, np.inf])))
        cases.append((T, perm, occ_cost, bam))
    # degenerate: no edges at all (every margin is -inf, messages become NaN), one frame pair, no candidates anywhere
    cases.append((random_sparse_trellis(rng, 5, 2, 2, 3, 0.0), [1, 0], 0.0, 0.0))
    cases.append((random_sparse_trellis(rng, 2, 4, 1, 5, 0.5), [0, 1, 2, 3], 0.0, 0.0))
    cases.append((random_sparse_trellis(rng, 12, 4, 3, 0, 0.6), [3, 2, 1, 0], 0.0, 0.0))
    return cases


def make_golden():
    R = _ref()
    assert R is not None, "needs a LocoMouse_cpp checkout (see oracle/reference_nms.py)"
    out = {}
    for i, (T, perm, occ_cost, bam) in enumerate(golden_cases()):
        lab = run(R, "ref_match2nd", T, occ_cost, bam, perm)
        out[f"labels_{i}"] = lab
        if T.points == 4 and (lab >= 0).all():  # a label of -1 makes the reference read outside its unary matrix
            out[f"cost_{i}"] = np.array([cost(R, "ref_cost_track", T, perm, lab)])
    np.savez_compressed(GOLD, **out)


def test_tracker_equals_reference_golden_vectors():
    H = _host()
    G = np.load(GOLD)
    n_occ = n_unsat = 0
    for i, (T, perm, occ_cost, bam) in enumerate(golden_cases()):
        got = run(H, "lmh_match2nd", T, occ_cost, bam, perm)
        want = G[f"labels_{i}"]
        assert np.array_equal(got, want), f"case {i}: labels differ\n{got}\n{want}"
        n_occ += int((want >= T.n_loc[None, :]).sum())
        n_unsat += int((want < 0).sum())
        if T.points == 4:
            # the label matrices never hold -1 where a cost is committed (the reference reads out of bounds there)
            if (want >= 0).all():
                c = cost(H, "lmh_cost_track", T, perm, want)
                assert np.float64(c).view(np.uint64) == np.float64(G[f"cost_{i}"][0]).view(np.uint64)
    assert n_occ > 0 and n_unsat > 0  # the vectors exercise occlusion labels and unsatisfiable tracks


def test_tracker_equals_reference_on_fresh_trellises():
    R = _ref()
    if R is None:
        pytest.skip("reference library not built (no LocoMouse_cpp checkout, see oracle/reference_nms.py); golden vectors cover it")
    H = _host()
    rng = np.random.Generator(np.random.PCG64(99))
    for it in range(150):
        points = int(rng.choice([1, 2, 3, 4]))
        if it % 5 == 0:
            T = tracker_like_trellis(rng, int(rng.integers(2, 60)), min(points, 4))
        else:
            T = random_sparse_trellis(rng, int(rng.integers(2, 25)), points, int(rng.integers(1, 4)), int(rng.integers(0, 7)),
                                      float(rng.choice([0.05, 0.2, 0.5, 1.0])))
        perm = list(rng.permutation(points))
        occ_cost, bam = float(rng.choice([0.0, 0.0, 0.02])), float(rng.choice([0.0, 0.0, 0.1, np.inf]))
        a = run(H, "lmh_match2nd", T, occ_cost, bam, perm)
        b = run(R, "ref_match2nd", T, occ_cost, bam, perm)
        assert np.array_equal(a, b), f"trellis {it}\n{a}\n{b}"


def test_tracker_is_reentrant():
    H = _host()
    rng = np.random.Generator(np.random.PCG64(5))
    T = tracker_like_trellis(rng, 80, 4)
    fn = H.lmh_match2nd_concurrent_check
    fn.restype = C.c_int
    perm = np.array([2, 0, 3, 1], np.int32)
    assert fn(*T.args(), C.c_double(0.0), C.c_double(0.0), C.c_void_p(perm.ctypes.data), 12, 4) == 1


def test_degenerate_inputs():
    H = _host()
    rng = np.random.Generator(np.random.PCG64(6))
    T = random_sparse_trellis(rng, 1, 2, 1, 3, 0.5)  # fewer than two frames: zeros, as the reference returns
    assert not run(H, "lmh_match2nd", T, 0.0, 0.0, [0, 1]).any()


if __name__ == "__main__":
    make_golden()
    print("wrote", GOLD)
