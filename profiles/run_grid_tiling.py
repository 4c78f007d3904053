"""Cost of angular window tiling (scene.super_resolve_grid, --full_grid 1) at the NTIRE geometry: a 9x9 grid of views of
432x624 HR at x4 (LR 108x156, 70 patches of 32 per window), MyEfficientLFNet with seeded random weights.

Per scene it reports:
  windows / wall   super_resolve_grid at angular stride t = 4, 2 and 1 (4, 9 and 25 windows), CUDA events, median of 3
                   after a warm-up; and super_resolve_scene on the central 5x5 for the cost of one window
  accumulate       lfsr_window_accumulate alone, "add" mode over a whole window (one read of the window mosaic, one
                   read-modify-write of its footprint in the 9x9 mosaic): CUDA events over 200 launches that cycle through
                   4 window / grid buffer pairs (216 MB touched in turn, so the launches do not run out of the 126 MB L2),
                   bytes and TB/s
and the same walls with the x8 self-ensemble. Prints the card name, power limit and max SM clock; writes JSON to --out.

    python profiles/run_grid_tiling.py [--out grid_tiling.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

A, SCALE, H, W, GRID = 5, 4, 432, 624, 9


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, reps=3):
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
    ap.add_argument("--out", default="grid_tiling.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_grid_tiling.py measures the GPU path: no CUDA device")
    import lfsr_b200
    from lfsr_b200 import scene
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(1234)
    net = lfsr_b200.load_net("MyEfficientLFNet", A, SCALE).eval().to(dev)
    h0, w0 = H // SCALE, W // SCALE
    lr = torch.from_numpy(np.random.RandomState(0).random_sample((GRID * h0, GRID * w0)).astype(np.float32)).to(dev)
    centre = lr.view(GRID, h0, GRID, w0)[2:7, :, 2:7, :].reshape(A * h0, A * w0)
    res = {"card": card(), "geometry": "9x9 views of 432x624 HR at x4 (LR 108x156), windows of 5x5, MyEfficientLFNet"}
    with torch.no_grad():
        for ens in (False, True):
            key = "self_ensemble" if ens else "plain"
            r = {"one_window_scene_ms": timed(lambda: scene.super_resolve_scene(net, centre, A, SCALE, self_ensemble=ens))}
            for t in (4, 2, 1):
                n_win = len(scene.window_plan(GRID, A, t))
                ms = timed(lambda: scene.super_resolve_grid(net, lr, GRID, A, SCALE, ang_stride=t, self_ensemble=ens))
                r["t%d" % t] = {"windows": n_win, "wall_ms": ms, "per_window_ms": ms / n_win}
            res[key] = r
            print(key, json.dumps(r))
        # the accumulate kernel alone
        ops = lfsr_b200.kernels.default_ops()
        hs, ws = H, W
        wins = [torch.rand((A * hs, A * ws), device=dev) for _ in range(4)]
        grids = [torch.rand((GRID * hs, GRID * ws), device=dev) for _ in range(4)]
        modes = [1] * (A * A)
        for k in range(4):
            ops.window_accumulate(wins[k], grids[k], A, GRID, hs, ws, 4, 4, modes)
        torch.cuda.synchronize()
        n = 200
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            ops.window_accumulate(wins[i % 4], grids[i % 4], A, GRID, hs, ws, 4, 4, modes)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / n
        nbytes = 3 * A * A * hs * ws * 4                  # window read + footprint read + footprint write
        res["accumulate"] = {"mode": "add", "bytes": nbytes, "us": ms * 1e3, "TB_per_s": nbytes / (ms * 1e-3) / 1e12}
        print("accumulate", json.dumps(res["accumulate"]))
    print(res["card"])
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
