"""Cost and parity of the x8 geometric self-ensemble (scene.SceneRunner(self_ensemble=True)).

  python profiles/run_self_ensemble.py OUT_DIR      -> OUT_DIR/self_ensemble.json (also printed)

(a) the Track-2 model (MyEfficientLFNet x4, seeded constructor-default weights as in bench.py) on bench.py's scene
    (128 x 128 views = 64 patches) through SceneRunner.run_resident with LR / HR already in HBM: ms per step without and
    with the ensemble, timed alternately in this process after warm-up, >= 2 s per timed window, CUDA events
(b) lfsr_divide_rows_d8 / lfsr_integrate_rows_d8 at that geometry timed alone (CUDA events, 200 launches) with their
    algorithmic bytes computed from shapes, next to the plain divide / integrate kernels
(c) max-abs error and |dPSNR| of the ensemble scene against the CPU oracle composition on a small non-square scene
(d) the device name, power limit and max SM clock, read in the same run
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import lfsr_b200                                                         # noqa: E402
from lfsr_b200 import kernels as K                                       # noqa: E402

A, P, S = 5, 32, 16


def events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def device_info(dev):
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        pl, mx = [x.strip() for x in q.split(",")]
        info.update(power_limit=pl, clocks_max_sm=mx)
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        info.update(power_limit=None, error=repr(e)[:200])
    return info


def scene_cost(dev, min_s=2.0, rounds=3):
    """(a): plain and ensemble steps alternate in windows of >= min_s seconds"""
    scale, h0 = 4, 128
    torch.manual_seed(1234)
    net = lfsr_b200.load_net("MyEfficientLFNet", A, scale).eval().to(dev)
    rs = np.random.RandomState(0)
    lr = torch.from_numpy(rs.random_sample((A * h0, A * h0)).astype(np.float32)).to(dev)
    hr = torch.from_numpy(rs.random_sample((A * h0 * scale, A * h0 * scale)).astype(np.float32)).to(dev)
    runners = {k: lfsr_b200.scene.SceneRunner(net, A, scale, h0, h0, P, S, minibatch=64, device=dev, world=1, rank=0,
                                              depth=1, self_ensemble=(k == "ensemble")) for k in ("plain", "ensemble")}
    steps = {}
    for k, r in runners.items():
        slot = r.device_slot(0)
        step = (lambda r=r, slot=slot: r.run_resident(lr, slot["mosaic"], hr, slot["acc"]))
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        one = events_ms(step, 3) / 3
        steps[k] = (step, max(3, int(min_s * 1e3 / one) + 1))
    windows = {k: [] for k in runners}
    for _ in range(rounds):
        for k, (step, n) in steps.items():
            windows[k].append(events_ms(step, n) / n)
    ms = {k: float(np.median(v)) for k, v in windows.items()}
    r8 = runners["ensemble"]
    out = {"workload": f"MyEfficientLFNet x{scale}, {h0}x{h0} views = {r8.num_u * r8.num_v} patches, LR/HR resident, "
                       "divide -> forwards -> integrate -> PSNR/SSIM sums (SceneRunner.run_resident)",
           "forward_batch": {k: (r.rows_per_mb * r.nvar * r.num_v) for k, r in runners.items()},
           "ms_per_step": ms, "windows_ms": windows, "steps_per_window": {k: n for k, (_, n) in steps.items()},
           "ratio": ms["ensemble"] / ms["plain"],
           "psnr_ssim": {k: [float(x) for x in r.metrics_from_sums(r.device_slot(0)["acc"].cpu().numpy())]
                         for k, r in runners.items()}}
    del runners, net
    torch.cuda.empty_cache()
    return out


def gather_rates(dev, iters=200):
    """(b): each gather alone at the bench geometry (x4), with the plain kernels for scale"""
    ops = K.default_ops()
    scale, h0 = 4, 128
    _, nu, nv = lfsr_b200.lfutils.divide_geometry(h0, h0, P, S)
    n = nu * nv
    L, pz, ss = A * P, P * scale, S * scale
    Lz, hs = A * pz, h0 * scale
    g = torch.Generator(device=dev).manual_seed(0)
    lr = torch.rand((A * h0, A * h0), device=dev, generator=g)
    sub1 = torch.empty((n, 1, L, L), device=dev)
    sub8 = torch.empty((8 * n, 1, L, L), device=dev)
    sr1 = torch.rand((n, 1, Lz, Lz), device=dev, generator=g)
    sr8 = torch.rand((8 * n, 1, Lz, Lz), device=dev, generator=g)
    mosaic = torch.empty((A * hs, A * hs), device=dev)
    calls = {
        "divide_rows_d8": (lambda: ops.divide_rows_d8(lr, sub8, A, h0, h0, P, S, 0, nu), 8 * n * L * L * 4 + lr.numel() * 4),
        "integrate_rows_d8": (lambda: ops.integrate_rows_d8(sr8, mosaic, A, pz, ss, hs, hs, nu, nv, 0, nu),
                              8 * mosaic.numel() * 4 + mosaic.numel() * 4),
        "divide_rows": (lambda: ops.divide_rows(lr, sub1, A, h0, h0, P, S, 0, nu), n * L * L * 4 + lr.numel() * 4),
        "integrate_rows": (lambda: ops.integrate_rows(sr1, mosaic, A, pz, ss, hs, hs, nu, nv, 0, nu), 2 * mosaic.numel() * 4),
    }
    out = {"geometry": f"{n} patches of 5x5x32x32 (x{scale}); bytes = output written + input read once (reads of the d8 "
                       "integrate: the 8 centre crops of every patch; of the divides: the LR scene)",
           "l2_note": "divide outputs (52 MB d8) fit the 126 MB L2 across repeats; the integrate inputs (839 MB d8) do not"}
    for k, (fn, nbytes) in calls.items():
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        ms = events_ms(fn, iters) / iters
        out[k] = {"us": ms * 1e3, "bytes": int(nbytes), "bytes_per_source_patch": nbytes / n, "gbs": nbytes / (ms * 1e-3) / 1e9}
    del sub1, sub8, sr1, sr8
    torch.cuda.empty_cache()
    return out


def parity(dev):
    """(c): ensemble scene (non-square 16 x 24 views, 2 patches = 16 network patches) against the CPU oracle composition"""
    from oracle import lf_oracle, weights
    from test_self_ensemble_cpu import oracle_ensemble_scene
    name, scale, h0, w0 = "MyEfficientLFNet", 4, 16, 24
    sd = weights.make_state_dict(name, scale, 1234)
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(sd, strict=True)
    net = net.to(dev)
    rs = np.random.RandomState(11)
    lr = rs.random_sample((A * h0, A * w0)).astype(np.float32)
    hr = rs.random_sample((A * h0 * scale, A * w0 * scale)).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr = lfsr_b200.scene.test_scene(net, torch.from_numpy(lr).to(dev), torch.from_numpy(hr).to(dev), A, scale,
                                                    P, S, 16, self_ensemble=True)
    sr = sr.cpu().numpy()
    torch.set_num_threads(os.cpu_count() or 1)
    want = oracle_ensemble_scene(name, lr, sd, A, scale, P, S, h0, w0)
    p_or = float(lf_oracle.cal_metrics(hr, want, A)[0])
    err = float(np.abs(sr - want).max())
    dps = abs(float(psnr) - p_or)
    return {"scene": f"{name} x{scale}, {h0}x{w0} views, seeded weights (oracle.weights, seed 1234)", "max_abs": err,
            "dpsnr_db": dps, "psnr": float(psnr), "psnr_oracle": p_or, "tol_max_abs": 1e-3, "tol_dpsnr_db": 0.01,
            "ok": bool(err <= 1e-3 and dps <= 0.01)}


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    out_dir = sys.argv[1]
    if not torch.cuda.is_available():
        sys.exit("run_self_ensemble.py measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"device": device_info(dev)}
    res["scene"] = scene_cost(dev)
    res["kernels"] = gather_rates(dev)
    res["parity"] = parity(dev)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "self_ensemble.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
