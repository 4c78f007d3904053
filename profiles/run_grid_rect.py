"""Cost of angular window tiling on a rectangular grid (scene.super_resolve_grid with n = (N_u, N_v), --full_grid 1
--grid_views) next to the square 9x9 grid of profiles/r04_grid_tiling_b200.json: views of 432x624 HR at x4 (LR 108x156,
70 patches of 32 per window), MyEfficientLFNet with seeded random weights.

Per grid (9x13 and 9x9) and angular stride (t = 4, 2) it reports:
  windows / wall   super_resolve_grid, CUDA events, median of 5 after a warm-up; and super_resolve_scene on one 5x5
                   window for the cost of one window
  accumulate       lfsr_window_accumulate_uv alone into the 9x13 mosaic, "add" mode over a whole window (one read of the
                   window mosaic, one read-modify-write of its footprint): CUDA events over 200 launches that cycle through
                   4 window / grid buffer pairs (~300 MB touched in turn, more than the 126 MB L2), bytes counted from the
                   shapes and TB/s
Prints the card name, power limit and max SM clock; writes JSON to --out.

    python profiles/run_grid_rect.py [--out grid_rect.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from run_grid_tiling import card  # noqa: E402

A, SCALE, H, W = 5, 4, 432, 624
GRIDS = [(9, 13), (9, 9)]


def timed(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="grid_rect.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_grid_rect.py measures the GPU path: no CUDA device")
    import lfsr_b200
    from lfsr_b200 import scene
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)
    net = lfsr_b200.load_net("MyEfficientLFNet", A, SCALE).eval().to(dev)
    h0, w0 = H // SCALE, W // SCALE
    res = {"card": card(), "geometry": "views of 432x624 HR at x4 (LR 108x156), windows of 5x5, MyEfficientLFNet"}
    with torch.no_grad():
        one = torch.from_numpy(np.random.RandomState(1).random_sample((A * h0, A * w0)).astype(np.float32)).to(dev)
        res["one_window_scene_ms"] = timed(lambda: scene.super_resolve_scene(net, one, A, SCALE))
        print("one window", res["one_window_scene_ms"])
        for nu, nv in GRIDS:
            lr = torch.from_numpy(np.random.RandomState(0).random_sample((nu * h0, nv * w0)).astype(np.float32)).to(dev)
            r = {}
            for t in (4, 2):
                n_win = len(scene.window_plan((nu, nv), A, t))
                ms = timed(lambda: scene.super_resolve_grid(net, lr, (nu, nv), A, SCALE, ang_stride=t))
                r["t%d" % t] = {"windows": n_win, "wall_ms": ms, "per_window_ms": ms / n_win}
            res["%dx%d" % (nu, nv)] = r
            print("%dx%d" % (nu, nv), json.dumps(r))
        # the accumulate kernel alone, into the 9x13 mosaic
        ops = lfsr_b200.kernels.default_ops()
        nu, nv = GRIDS[0]
        hs, ws = H, W
        wins = [torch.rand((A * hs, A * ws), device=dev) for _ in range(4)]
        grids = [torch.rand((nu * hs, nv * ws), device=dev) for _ in range(4)]
        modes = [1] * (A * A)
        for k in range(4):
            ops.window_accumulate_uv(wins[k], grids[k], A, nu, nv, hs, ws, 4, 8, modes)
        torch.cuda.synchronize()
        n = 200
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            ops.window_accumulate_uv(wins[i % 4], grids[i % 4], A, nu, nv, hs, ws, 4, 8, modes)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / n
        nbytes = 3 * A * A * hs * ws * 4                  # window read + footprint read + footprint write
        res["accumulate_uv"] = {"grid": "%dx%d" % (nu, nv), "mode": "add", "bytes": nbytes, "us": ms * 1e3,
                                "TB_per_s": nbytes / (ms * 1e-3) / 1e12}
        print("accumulate_uv", json.dumps(res["accumulate_uv"]))
    print(res["card"])
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
