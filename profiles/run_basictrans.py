"""The fused EPIT BasicTrans kernel on its production shape (B patches of 5x5x32x32, 64 channels): CUDA-event time per call,
useful TFLOP/s (SURVEY 8d: 4.8235 GMAC per call per patch), and the whole EPIT forward.
usage: python profiles/run_basictrans.py [batch] [forward: 0|1]"""
import os, sys, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lfsr_b200
from lfsr_b200 import kernels as K

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
do_fwd = int(sys.argv[2]) if len(sys.argv) > 2 else 1
dev = "cuda"
ops = K.default_ops()
torch.manual_seed(1234)
net = lfsr_b200.load_net("EPIT", 5, 4).eval().to(dev)
pk = net._get_packed(torch.device(dev, 0), ops)
al = pk["alt"][0]
A, h, W = 5, 32, 160
x = (torch.rand(B, W, W, 64, device=dev) - 0.5).half()
y = torch.empty_like(x)
passes = [dict(A=A, S=h, stride_a=h * W, stride_s=W, stride_b=W * W, stride_p=h, stride_q=1, np_=A, nq=h),
          dict(A=A, S=h, stride_a=h, stride_s=1, stride_b=W * W, stride_p=h * W, stride_q=W, np_=A, nq=h)]
for name, p in zip(("H pass (columns)", "V pass (rows)"), passes):
    call = lambda: ops.basictrans(x, al["bt"][0], al["bt"][1], y, p["A"], p["S"], 5, B, p["np_"], p["nq"], p["stride_a"],
                                  p["stride_s"], p["stride_b"], p["stride_p"], p["stride_q"])
    for _ in range(3):
        assert call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    fl = 2 * 4.8235e9 * B
    tiles = B * 160 * 2
    print(f"basictrans {name} batch {B}: {ms:.3f} ms/call, {fl / ms / 1e9:.1f} useful TFLOP/s, "
          f"{ms * 1e-3 * 1.965e9 / (tiles / 148):.0f} cycles/tile @1965 MHz")
if do_fwd:
    xin = torch.rand(B, 1, 160, 160, device=dev)
    for _ in range(2):
        net.forward_static(xin)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        net.forward_static(xin)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    print(f"EPIT forward batch {B}: {ms:.2f} ms, {B / ms * 1e3:.0f} patches/s")
