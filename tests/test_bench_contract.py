"""The reference arm of bench.py (`--impl reference`: the oracle port on the host cores, the one place besides tests / smoke
where bench.py executes oracle/) prints ONE JSON line with the fields the round driver reads.  Runs on CPU; the GPU arm's line is
checked on the GPU box by the driver itself."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "detection_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["data"] == "synthetic"
    assert "workload" in d["config"] and "configs[1]" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_dump_outputs_writes_a_seeded_sample_of_the_result_arrays_exactly(oracle, small_problem, tmp_path, monkeypatch):
    """bench.py --dump-outputs: the same frames are sampled every time and every result value survives the float dtypes."""
    import bench

    p = small_problem
    res = oracle.detect(p["cfg"], p["model"], p["bkg"], p["calib"], p["frames"], p["bb_x"], p["bb_y_side"], p["bb_y_bottom"],
                        n_threads=2)
    monkeypatch.setattr(bench, "DUMP_FRAMES", 4)
    bench.dump_outputs(res, str(tmp_path / "a"))
    bench.dump_outputs(res, str(tmp_path / "b"))
    idx = np.load(tmp_path / "a" / "frame_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "frame_index.npy"))
    idx = idx.astype(np.int64)
    assert len(idx) == 4 and np.all(np.diff(idx) > 0) and idx[-1] < res.n
    want = {"frame_index": idx}
    for name in res.ARRAYS:
        a = getattr(res, name)[idx]
        if a.dtype.names:
            want.update({f"{name}_{f}": a[f] for f in a.dtype.names})
        else:
            want[name] = a
    assert sorted(f[:-4] for f in os.listdir(tmp_path / "a")) == sorted(want)
    for name, w in want.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype in (np.float32, np.float64), name
        assert np.array_equal(got, w, equal_nan=got.dtype == np.float64), name
