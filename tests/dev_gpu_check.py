"""Development aid (lives under tests/ because it uses the oracle): run the CUDA path and the oracle on the same small
synthetic problem and print where they differ, stage by stage.  Not collected by pytest; run it directly:
    python tests/dev_gpu_check.py --frames 8"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from locomouse_cpp_b200 import synth  # noqa: E402
from locomouse_cpp_b200.api import Detector  # noqa: E402
from locomouse_cpp_b200.types import diff_results  # noqa: E402
from oracle import oracle  # noqa: E402

import _preprocess_designs as designs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--method", default="TM")
    ap.add_argument("--flip", action="store_true")
    ap.add_argument("--warp", action="store_true")
    ap.add_argument("--muladd", action="store_true")
    ap.add_argument("--device-frames", action="store_true")
    ap.add_argument("--bench", type=int, default=0, help="also time this many device-resident frames")
    args = ap.parse_args()

    spec = synth.SynthSpec(method=args.method, flip=args.flip, warp=args.warp, fma_mode=not args.muladd)
    cfg, model, bkg, calib, frames, bx, bs, bb = synth.make_problem(spec, args.frames, seed=1000)
    frames_np = frames.numpy()
    t = time.time()
    ref = oracle.detect(cfg, model, bkg, calib, frames_np, bx, bs, bb, n_threads=8)
    print(f"oracle: {time.time() - t:.2f}s  n_bottom={ref.n_bottom.sum(0)} n_side={ref.n_side.sum(0)} rc={ref.rc}")

    det = Detector(cfg, model, bkg, calib)
    pads, canvas = det.geometry()
    opads, ocanvas = oracle.geometry(cfg, model)
    print("geometry equal:", np.array_equal(pads, opads) and np.array_equal(canvas, ocanvas))
    if args.device_frames:
        import torch

        fr = torch.from_numpy(frames_np).cuda()
    else:
        fr = frames_np
    t = time.time()
    got = det.detect_batch(fr, bx, bs, bb, allow_overflow=True)
    print(f"gpu: {time.time() - t:.3f}s rc={got.rc} timing={det.last_timing()}")

    # stage diagnostics on the last sub-batch (windows placed and sized by tests/_preprocess_designs.py)
    for f in range(args.frames):
        I, mm = oracle.preprocess(cfg, bkg, calib, frames_np[f])
        try:
            gmm, _ = det.debug_fetch(3, f)
        except Exception:  # frame not in last sub-batch
            continue
        if not np.array_equal(gmm, mm):
            print(f"frame {f}: minmax gpu {gmm} oracle {mm}")
        for v, ypos in ((0, bb[f]), (1, bs[f])):
            win, dims = det.debug_fetch(v, f)
            x0, y0, win_w, _ = designs.window_origin(cfg, model, v, bx[f], ypos)
            exp = designs.expected_window(I, x0, y0, win.shape[0], win.shape[1], win_w)
            ncmp = (win != exp)
            if ncmp.any():
                idx = np.argwhere(ncmp)
                print(f"frame {f} view {v}: window differs at {len(idx)} px, first {idx[0]} gpu {win[tuple(idx[0])]} exp {exp[tuple(idx[0])]}")
    d = diff_results(got, ref)
    print("DIFF:", "none (bit-exact)" if not d else "")
    for line in d[:20]:
        print("  ", line)
    if d:
        for f in range(args.frames):
            for k in range(2):
                if got.candidates_bottom(f, k) != ref.candidates_bottom(f, k):
                    print(f"f{f} feat{k} bottom gpu {got.candidates_bottom(f, k)[:6]}\n            ref {ref.candidates_bottom(f, k)[:6]}")
                if got.candidates_side(f, k) != ref.candidates_side(f, k):
                    print(f"f{f} feat{k} side   gpu {got.candidates_side(f, k)[:6]}\n            ref {ref.candidates_side(f, k)[:6]}")
            if not np.array_equal(got.tail[f], ref.tail[f]):
                print(f"f{f} tail gpu\n{got.tail[f]}\nref\n{ref.tail[f]}")

    if args.bench:
        import torch

        n = args.bench
        fr, bx2, bs2, bb2 = synth.make_video(spec, n, 1000, "cuda", bkg)
        torch.cuda.synchronize()
        for it in range(3):
            t = time.time()
            r = det.detect_batch(fr, bx2, bs2, bb2, allow_overflow=True)
            dt = time.time() - t
            tm, nl = det.last_timing()
            print(f"bench n={n}: wall {dt * 1e3:.1f} ms -> {n / dt:.0f} frames/s; device stages(ms) {tm} launches {nl}")
        print("flags any:", int((r.flags != 0).sum()), "n_bottom mean", r.n_bottom.mean(0), "n_side mean", r.n_side.mean(0))


if __name__ == "__main__":
    main()
