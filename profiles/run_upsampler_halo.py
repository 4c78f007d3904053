"""Times the two upsampler convs of MyEfficientLFNet x4 at batch 64 (up.0: 3x3 64->224 @160^2 + PixelShuffle + LReLU, fp16
out; up.3: 3x3 56->224 @320^2 + PixelShuffle + LReLU + head-conv tap projection) with CUDA events: 10 warm-up calls, then
50 timed calls, median and min per call. Run it once on the product library (halo-block kernel) and once with
LFSR_PROBE_LIB=1 LFSR_TC_NO_HALO=1 (per-tap kernel) for an A/B pair.

    python profiles/run_upsampler_halo.py out.json
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import lfsr_b200  # noqa: E402
from lfsr_b200 import _native as N, kernels as K  # noqa: E402
from oracle import weights  # noqa: E402


def main(out_path):
    dev = torch.device("cuda:0")
    lib = N.load()
    ops = K.default_ops()
    net = lfsr_b200.load_net("MyEfficientLFNet", 5, 4).eval()
    net.load_state_dict(weights.make_state_dict("MyEfficientLFNet", 4, 1234), strict=True)
    net = net.to(dev)
    pk = net._get_packed(dev, ops)
    B, width = 64, pk["CU"]
    calls, h = [], 160
    for j, (pcv, r) in enumerate(pk["up"]):
        x = (torch.rand(B, h, h, pcv.cin, device=dev) * 2 - 1).half()
        shuffle = (r, r, N.SHUF_CHANNEL_MAJOR)
        if j == len(pk["up"]) - 1:
            y = net._buf("head_taps", B, h * r, h * r, 9, dev)
            calls.append((f"up{j} {h}^2 tail", lambda x=x, pcv=pcv, y=y, s=shuffle: ops.conv(
                x, pcv, y, act=N.ACT_LRELU, slope=0.1, shuffle=s, tail=(pk["tail_w"], 9, width))))
        else:
            y = net._buf16(f"up{j}", B, h * r, h * r, width, dev)
            calls.append((f"up{j} {h}^2 fp16 out", lambda x=x, pcv=pcv, y=y, s=shuffle: ops.conv(
                x, pcv, None, out16=y, act=N.ACT_LRELU, slope=0.1, shuffle=s)))
        h *= r
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "library": "probe" if os.environ.get("LFSR_PROBE_LIB") == "1" else "product",
           "no_halo": os.environ.get("LFSR_TC_NO_HALO") == "1", "batch": B, "layers": {}}
    for name, fn in calls:
        c0 = lib.lfsr_conv_tc_halo_count()
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(50)]
        for a, b in ev:
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        res["layers"][name] = {"median_ms": ms[len(ms) // 2], "min_ms": ms[0],
                               "halo_launches": lib.lfsr_conv_tc_halo_count() - c0}
    print(json.dumps(res))
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
