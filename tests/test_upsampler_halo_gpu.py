"""The halo-block CTA-pair kernel (conv_tc_halo_kernel) against the per-tap kernel it replaces for the upsampler convs of
MyEfficientLFNet: both layers at x4 (fp16 output, tail projection) and the single layer at x2, at batch 1, 3 and 64, and
whole forwards. Both kernels issue the same MMAs in the same order and share the epilogue arithmetic, so the outputs must be
bit-identical. The per-tap kernel is selected with the probe library's LFSR_TC_NO_HALO switch; each side runs in its own
process, because the library reads its switches once."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCHES = (1, 3, 64)


def _run_layers(path):
    """every upsampler conv of MyEfficientLFNet x4 / x2 on seeded fp16 inputs, called as lfnets.common.upsample_tail calls
    them, plus two whole forwards; saves the outputs and the halo-kernel launch count"""
    import lfsr_b200
    from lfsr_b200 import _native as N, kernels as K
    from oracle import weights
    dev = torch.device("cuda:0")
    lib = N.load()
    ops = K.default_ops()
    res, launches = {}, 0
    for scale in (4, 2):
        net = lfsr_b200.load_net("MyEfficientLFNet", 5, scale).eval()
        net.load_state_dict(weights.make_state_dict("MyEfficientLFNet", scale, 1234), strict=True)
        net = net.to(dev)
        pk = net._get_packed(dev, ops)
        width, n_up = pk["CU"], len(pk["up"])
        g = torch.Generator(device=dev).manual_seed(11)
        for B in BATCHES:
            h = 160
            for j, (pcv, r) in enumerate(pk["up"]):
                x = (torch.rand(B, h, h, pcv.cin, device=dev, generator=g) * 2 - 1).half()
                shuffle = (r, r, N.SHUF_CHANNEL_MAJOR)
                c0 = lib.lfsr_conv_tc_halo_count()
                if j == n_up - 1:
                    assert ops.tail_supported(pcv, width, shuffle)
                    y = net._buf("head_taps", B, h * r, h * r, 9, dev)
                    y.fill_(float("nan"))
                    ops.conv(x, pcv, y, act=N.ACT_LRELU, slope=0.1, shuffle=shuffle, tail=(pk["tail_w"], 9, width))
                else:
                    y = net._buf16(f"up{j}", B, h * r, h * r, width, dev)
                    y.fill_(float("nan"))
                    ops.conv(x, pcv, None, out16=y, act=N.ACT_LRELU, slope=0.1, shuffle=shuffle)
                torch.cuda.synchronize()
                launches += lib.lfsr_conv_tc_halo_count() - c0
                res[f"x{scale}_up{j}_b{B}"] = y.clone().cpu()
                h *= r
        xin = weights.synthetic_patches(3, 5, 32, seed=3).to(dev)
        res[f"x{scale}_forward"] = net(xin, [5, 5]).cpu()
    res["halo_launches"] = launches
    torch.save(res, path)


def _side(tmp_path, name, env):
    path = str(tmp_path / f"{name}.pt")
    code = ("import sys; sys.path[:0]=['.','tests']; import test_upsampler_halo_gpu as t; t._run_layers(%r)" % path)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    return torch.load(path)


def test_halo_kernel_bit_identical_to_per_tap(tmp_path):
    new = _side(tmp_path, "halo", {"LFSR_PROBE_LIB": "0"})
    old = _side(tmp_path, "per_tap", {"LFSR_PROBE_LIB": "1", "LFSR_TC_NO_HALO": "1"})
    # x4: up.0 and up.3, x2: the single layer, at each batch; the whole forwards add two x4 and one x2 launch each
    layers = len(BATCHES) * 3
    assert new.pop("halo_launches") >= layers, "the halo-block kernel did not take the upsampler convs"
    assert old.pop("halo_launches") == 0
    assert new.keys() == old.keys()
    for k in new:
        assert not torch.isnan(new[k].float()).any(), k
        assert torch.equal(new[k], old[k]), k
