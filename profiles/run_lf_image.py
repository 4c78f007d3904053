"""Cost of reading a light field stored as one lenslet image (utils_datasets.ImageTestSet, lfutils.prepare_image) at the
geometry of a decoded Lytro Illum capture: 14x14 views of 376x541, one seeded 8-bit PNG of 5264x7574 px.

It reports:
  decode      read_lf_image (Pillow PNG decode on the host)
  stage       the copy of the decoded image into the pinned staging buffer (host)
  h2d         the pinned host-to-device copy of the whole image (CUDA events)
  gather      lfsr_image_to_views_u8 alone (CUDA events over repeated launches that cycle through 4 device copies of the
              image and 4 output buffers, so that the working set exceeds the 126 MB L2), for the central 9x9 views
              cropped to x4 and for all 196 views; GB/s of the bytes the gather must move (read + write of the selected
              views) against 7.7 TB/s
  numpy       the same 9x9 gather on the host with numpy (reshape, transpose, contiguous copy), for comparison
  prepare     lfutils.prepare_image on the image against lfutils.prepare_views on the same views (host views), host
              clock around a device synchronise: kind "hr" on the central 5x5, kind "lr" on the central 9x9, x4
  inference   inference.py --input_layout lenslet --input_grid 14x14 --full_grid 1 --grid_views 9x9 --save_layout lenslet
              (MyEfficientLFNet x4, random init) on 3 copies of the scene: wall time and the time between the per-scene
              lines it prints
Prints the card name and power limit; writes JSON to --out.

    python profiles/run_lf_image.py [--out lf_image.json]     (profiles/r05_lf_image_b200.json is one such run)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

U = V = 14
H, W, SCALE, A = 376, 541, 4, 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def lenslet(seed=0):
    """uint8 [(H U), (W V), 3]: each view a window of one seeded smooth, noisy image, shifted by 1 px per angular step"""
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, H + U), np.linspace(0, 1, W + V), indexing="ij")
    f = rs.uniform(4, 12, (3, 2))
    big = np.stack([np.sin(f[c, 0] * yy * 3) * np.cos(f[c, 1] * xx * 3) for c in range(3)], -1)
    big = np.clip(np.round(127.5 + 90 * big + rs.normal(0, 4, big.shape)), 0, 255).astype(np.uint8)
    g = np.stack([np.stack([big[u:u + H, v:v + W] for v in range(V)]) for u in range(U)])
    return np.ascontiguousarray(g.transpose(2, 0, 3, 1, 4)).reshape(H * U, W * V, 3)


def host_ms(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def gather_rate(lib, imgs, nu, nv, reps=40):
    hc, wc = H - H % SCALE, W - W % SCALE
    u0, v0 = (U - nu) // 2, (V - nv) // 2
    outs = [torch.empty((nu, nv, hc, wc, 3), dtype=torch.uint8, device="cuda") for _ in imgs]
    stream = torch.cuda.current_stream().cuda_stream

    def launch(k):
        st = lib.lfsr_image_to_views_u8(imgs[k % len(imgs)].data_ptr(), 2, U, V, H, W, u0, v0, nu, nv, hc, wc,
                                        outs[k % len(outs)].data_ptr(), stream)
        assert st == 0
    for k in range(8):
        launch(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(reps):
        launch(k)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = 2 * nu * nv * hc * wc * 3
    return {"views": "%dx%d" % (nu, nv), "us": us, "bytes": nbytes, "GBps": nbytes / us / 1e3,
            "share_of_7_7_TBps": nbytes / us / 1e6 / 7.7}


def inference_run(tmp, png):
    data = os.path.join(tmp, "data", "Set")
    os.makedirs(data)
    for i in range(3):
        os.link(png, os.path.join(data, "scene_%d.png" % i))
    cmd = [sys.executable, "-u", "inference.py", "--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4",
           "--use_pre_ckpt", "", "--path_for_test", os.path.join(tmp, "data") + "/", "--input_layout", "lenslet",
           "--input_grid", "14x14", "--full_grid", "1", "--grid_views", "9x9", "--save_layout", "lenslet", "--path_log",
           os.path.join(tmp, "log") + "/"]
    t0 = time.perf_counter()
    p = subprocess.Popen(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    marks = []
    for line in p.stdout:
        if line.startswith("scene "):
            marks.append(time.perf_counter() - t0)
    err = p.stderr.read()
    assert p.wait() == 0, err[-3000:]
    wall = time.perf_counter() - t0
    out = [os.path.join(dp, f) for dp, _, fs in os.walk(os.path.join(tmp, "log")) for f in fs if f.endswith(".bmp")]
    return {"wall_s": wall, "scene_done_s": marks, "per_scene_s_warm": float(np.mean(np.diff(marks))),
            "bmp_files": len(out), "bmp_bytes": os.path.getsize(out[0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="lf_image.json")
    a = ap.parse_args()
    from PIL import Image
    from lfsr_b200 import _native as N, lfutils
    from utils.utils_datasets import read_lf_image
    from test_lf_image_cpu import image_to_views
    res = {"card": card(), "geometry": "14x14 views of 376x541 as one 5264x7574 lenslet PNG; x4 crop to 376x540",
           "torch": torch.__version__}
    img = lenslet()
    with tempfile.TemporaryDirectory() as tmp:
        png = os.path.join(tmp, "lf.png")
        t0 = time.perf_counter()
        Image.fromarray(img).save(png)
        res["encode_png_s"] = time.perf_counter() - t0
        res["png_bytes"] = os.path.getsize(png)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            dec = read_lf_image(png, "lenslet", (U, V))
            ts.append((time.perf_counter() - t0) * 1e3)
        assert np.array_equal(dec, img)
        res["decode_png_ms"] = float(np.median(ts))

        dev = torch.device("cuda", 0)
        pinned = torch.empty(img.shape, dtype=torch.uint8, pin_memory=True)
        res["stage_pinned_ms"] = host_ms(lambda: pinned.numpy().__setitem__(Ellipsis, img), 5)
        d = torch.empty(img.shape, dtype=torch.uint8, device=dev)
        d.copy_(pinned, non_blocking=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            d.copy_(pinned, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        res["h2d_bytes"] = img.nbytes
        res["h2d_ms"] = e0.elapsed_time(e1) / 10

        lib = N.load()
        imgs = [d] + [d.clone() for _ in range(3)]
        res["gather"] = [gather_rate(lib, imgs, 9, 9), gather_rate(lib, imgs, U, V)]
        del imgs

        hc, wc = H - H % SCALE, W - W % SCALE
        t0 = time.perf_counter()
        u0 = (U - 9) // 2
        for _ in range(3):
            np_views = np.ascontiguousarray(
                img.reshape(H, U, W, V, 3)[:hc, u0:u0 + 9, :wc, u0:u0 + 9].transpose(1, 3, 0, 2, 4))
        res["numpy_gather_9x9_ms"] = (time.perf_counter() - t0) * 1e3 / 3
        all_views = image_to_views(img, "lenslet", U, V)
        assert np.array_equal(np_views, all_views[u0:u0 + 9, u0:u0 + 9, :hc, :wc])

        res["prepare"] = []
        for kind, sel in (("hr", A), ("lr", 9)):
            got = lfutils.prepare_image(img, "lenslet", (U, V), sel, SCALE, kind)
            want = lfutils.prepare_views(all_views, sel, SCALE, kind)
            same = all(x is None and y is None or torch.equal(x, y) for x, y in zip(got, want))
            del got, want
            t_img = host_ms(lambda: lfutils.prepare_image(img, "lenslet", (U, V), sel, SCALE, kind), 5)
            t_views = host_ms(lambda: lfutils.prepare_views(all_views, sel, SCALE, kind), 5)
            res["prepare"].append({"kind": kind, "views": "%dx%d" % (sel, sel), "prepare_image_ms": t_img,
                                   "prepare_views_ms": t_views, "bit_identical": bool(same)})
        torch.cuda.empty_cache()
        res["inference_py"] = inference_run(tmp, png)
    print(json.dumps(res, indent=1))
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
