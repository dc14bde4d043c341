"""locomouse_b200_batch's pre-flight (CPU): the list file is checked before any CUDA call.  Every refusal names its list line and
the program exits with EXIT_FAILURE without creating a context (no summary file is written)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "locomouse_cpp_b200", "host")


@pytest.fixture(scope="module")
def exe():
    if not os.path.exists(os.path.join(ROOT, "locomouse_cpp_b200", "liblocomouse_b200.so")):
        pytest.skip("CUDA library not built")
    p = subprocess.run(["make", "-C", HOST, "locomouse_b200_batch"], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    return os.path.join(HOST, "locomouse_b200_batch")


def _touch(path):
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_bytes(b"x")
    return path


def _run(exe, tmp_path, lines, side="R", cwd=None):
    (tmp_path / "config.yml").write_text("conn_comp_connectivity: 8\n")
    lst = tmp_path / "list.tsv"
    lst.write_text("".join(line + "\n" for line in lines))
    out = tmp_path / "out"
    out.mkdir(exist_ok=True)
    p = subprocess.run([exe, "1", str(tmp_path / "config.yml"), str(lst), str(tmp_path / "m"), str(tmp_path / "c"), side, str(out)],
                       capture_output=True, text=True, cwd=cwd)
    assert not (out / "batch_summary.tsv").exists(), "the pre-flight must stop before any video is run"
    assert "lm_create" not in p.stdout
    return p


def test_missing_video_or_background(exe, tmp_path):
    v, b = _touch(tmp_path / "a.lmv"), _touch(tmp_path / "bkg.lmi")
    p = _run(exe, tmp_path, [f"{v}\t{b}", f"{tmp_path / 'gone.lmv'}\t{b}", f"{v.with_name('c.lmv')}\t{tmp_path / 'nobkg.lmi'}"])
    assert p.returncode == 1
    assert f"list line 2: video file {tmp_path / 'gone.lmv'} does not exist" in p.stdout
    assert f"list line 3: video file {tmp_path / 'c.lmv'} does not exist" in p.stdout
    assert f"list line 3: background file {tmp_path / 'nobkg.lmi'} does not exist" in p.stdout
    assert "list line 1" not in p.stdout


def test_bad_side_character(exe, tmp_path):
    b = _touch(tmp_path / "bkg.lmi")
    v = [_touch(tmp_path / f"v{i}.lmv") for i in range(4)]
    p = _run(exe, tmp_path, [f"{v[0]}\t{b}\tL", f"{v[1]}\t{b}\tX", f"{v[2]}\t{b}\tR", f"{v[3]}\t{b}\tLR"])
    assert p.returncode == 1
    assert "list line 2: side 'X' must be either" in p.stdout and "list line 4: side 'LR'" in p.stdout
    assert "list line 1" not in p.stdout and "list line 3" not in p.stdout
    # the command line's side applies to lines without their own
    p = _run(exe, tmp_path, [f"{v[0]}\t{b}\tL", f"{v[1]}\t{b}"], side="Q")
    assert p.returncode == 1 and "list line 2: side 'Q' must be either \"L\" or \"R\" (from the command line)" in p.stdout
    assert "list line 1" not in p.stdout


def test_duplicate_output_stems(exe, tmp_path):
    b = _touch(tmp_path / "bkg.lmi")
    v1, v2, v3 = _touch(tmp_path / "a" / "trial.avi"), _touch(tmp_path / "b" / "trial.lmv"), _touch(tmp_path / "b" / "other.avi")
    p = _run(exe, tmp_path, [f"{v1}\t{b}", f"{v3}\t{b}", f"{v2}\t{b}"])
    assert p.returncode == 1
    assert "list line 3: output stem 'trial' is also the stem of line 1" in p.stdout
    assert "list line 2" not in p.stdout


def test_comment_and_blank_lines_keep_the_line_numbers(exe, tmp_path):
    b = _touch(tmp_path / "bkg.lmi")
    v = _touch(tmp_path / "v.lmv")
    p = _run(exe, tmp_path, ["# session 3", "", "   ", f"#{tmp_path / 'gone.lmv'}\t{b}", f"{tmp_path / 'gone.lmv'}\t{b}", f"{v}\t{b}",
                             f"{v}"])
    assert p.returncode == 1
    assert "list line 5: video file" in p.stdout
    assert "list line 7: expected video<TAB>background[<TAB>side], found 1 field(s)" in p.stdout
    for n in (1, 2, 3, 4, 6):
        assert f"list line {n}:" not in p.stdout
    # only comments: nothing to run is a refusal too
    p = _run(exe, tmp_path, ["# nothing", ""])
    assert p.returncode == 1 and "names no video" in p.stdout


def test_relative_paths_resolve_against_the_list_directory(exe, tmp_path):
    _touch(tmp_path / "videos" / "v1.lmv")
    _touch(tmp_path / "bkg" / "b1.lmi")
    elsewhere = tmp_path / "elsewhere"
    elsewhere.mkdir()
    _touch(elsewhere / "videos" / "v2.lmv")   # exists relative to the working directory only
    p = _run(exe, tmp_path, ["videos/v1.lmv\tbkg/b1.lmi", "videos/v2.lmv\tbkg/b1.lmi"], cwd=str(elsewhere))
    assert p.returncode == 1
    assert f"list line 2: video file {tmp_path}/videos/v2.lmv does not exist" in p.stdout
    assert "list line 1" not in p.stdout
