"""CPU checks of the host-side launch plans: each drop-in module, with the torch statement of the
kernel contracts (tests/opref.RefOps) injected as backend, must reproduce the oracle (and through
it the reference - oracle/make_golden.py pins oracle == reference bit-exactly) and the goldens."""
import numpy as np
import pytest
import torch

import lfsr_b200
from opref import RefOps
from oracle import nets as onets, weights

CASES = [("MyEfficientLFNet", 4), ("MyEfficientLFNet", 2), ("EPIT", 4), ("DistgSSR", 4), ("DistgSSR", 2),
         ("LF_InterNet", 4), ("MyEfficientLFNetV4_5", 4)]


def _have(name):
    try:
        lfsr_b200.net_module(name)
        return True
    except ModuleNotFoundError:
        return False


@pytest.mark.parametrize("name,scale", CASES)
def test_state_dict_matches_reference_spec(name, scale):
    if not _have(name):
        pytest.skip(f"{name} not built yet")
    net = lfsr_b200.load_net(name, 5, scale)
    spec = weights.load_spec(name, scale)
    sd = net.state_dict()
    assert list(sorted(sd.keys())) == sorted(n for n, _, _ in spec)
    for n, shape, dtype in spec:
        assert tuple(sd[n].shape) == tuple(shape), n
        assert str(sd[n].dtype).replace("torch.", "") == dtype, n
    gold = np.load(f"{weights.GOLDEN_DIR}/{name}_x{scale}.npz")
    assert sum(p.numel() for p in net.parameters()) == int(gold["nparams"])


@pytest.mark.parametrize("name,scale", CASES)
def test_launch_plan_matches_oracle_p8(name, scale):
    if not _have(name):
        pytest.skip(f"{name} not built yet")
    net = lfsr_b200.load_net(name, 5, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    net.set_backend(RefOps())
    x = weights.synthetic_patches(2, 5, 8, seed=7)
    y = net(x, [5, 5])
    gold = np.load(f"{weights.GOLDEN_DIR}/{name}_x{scale}.npz")["p8_out"]
    y_or = onets.forward(name, x, sd, 5, scale)
    assert y.shape == y_or.shape
    assert np.abs(y_or.numpy() - gold).max() <= 1e-5          # oracle == committed reference output
    assert (y - y_or).abs().max().item() <= 2e-5              # launch plan == oracle


@pytest.mark.parametrize("name,scale", [("DistgSSR", 4), ("DistgSSR", 2), ("LF_InterNet", 4), ("EPIT", 4), ("MyEfficientLFNet", 4),
                                         ("MyEfficientLFNet", 2)])
def test_fp16_operand_plan_matches_oracle_p8(name, scale):
    """the launch plans that exchange fp16 activations between tensor-core layers (residual trunks stay fp32): the torch
    backend rounds the same tensors through fp16, so the plan (which buffer feeds which layer) is checked on the CPU"""
    net = lfsr_b200.load_net(name, 5, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    net.set_backend(RefOps(fp16_operands=True))
    x = weights.synthetic_patches(2, 5, 8, seed=7)
    y = net(x, [5, 5])
    assert net._packed["f16"]
    y_or = onets.forward(name, x, sd, 5, scale)
    err = (y - y_or).abs().max().item()
    assert 0 < err <= 1e-3, err                              # fp16 rounding of the operands is visible, and inside the budget


def test_cpu_input_without_backend_raises():
    net = lfsr_b200.load_net("MyEfficientLFNet", 5, 4)
    with pytest.raises(lfsr_b200.LfsrError):
        net(torch.zeros(1, 1, 40, 40))


def test_oracle_imresize_matches_reference_golden(monkeypatch):
    """oracle.lf_oracle.imresize == outputs of the unmodified utils/imresize.py (oracle/make_golden.py, SURVEY 8f-3), and
    the product's host-side contribution tables equal the oracle's"""
    from oracle import lf_oracle
    g = np.load(f"{weights.GOLDEN_DIR}/imresize.npz")
    kws = {"y_down4": dict(scalar_scale=0.25), "cbcr_up4": dict(scalar_scale=4), "tri_down2": dict(scalar_scale=0.5, method="bilinear"),
           "shape": dict(output_shape=(45, 20)), "u8_down3": dict(scalar_scale=1.0 / 3)}
    for key, kw in kws.items():
        out = lf_oracle.imresize(g[key + "_in"], **kw)
        assert out.dtype == g[key + "_out"].dtype and np.abs(out.astype(np.float64) - g[key + "_out"].astype(np.float64)).max() <= 1e-13
    for n_in, n_out, sc, m in ((64, 16, 0.25, "bicubic"), (24, 96, 4.0, "bicubic"), (37, 19, 0.5, "bilinear"), (50, 20, 0.4, "bicubic")):
        w0, i0 = lf_oracle.imresize_contributions(n_in, n_out, sc, m)
        w1, i1 = lfsr_b200.lfutils.resize_contributions(n_in, n_out, sc, m)
        assert np.array_equal(w0, w1) and np.array_equal(i0, i1)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)        # host inputs go to the GPU when there is one
    with pytest.raises(lfsr_b200.LfsrError):
        lfsr_b200.lfutils.imresize(np.zeros((8, 8)), scalar_scale=2)        # no CPU fallback


def test_oracle_colour_tail_and_bmp_writer(tmp_path, monkeypatch):
    """oracle colour tail == the reference's (committed golden); write_bmp == Pillow's bytes (host logic, no GPU)"""
    from oracle import lf_oracle
    g = np.load(f"{weights.GOLDEN_DIR}/colour_tail.npz")
    assert np.array_equal(lf_oracle.sai_to_rgb8_views(g["sr_y"][0, 0], g["sr_cbcr"][0], 5), g["views"])
    p = tmp_path / "v.bmp"
    lfsr_b200.lfutils.write_bmp(str(p), g["views"][1, 3])
    assert np.array_equal(np.frombuffer(p.read_bytes(), dtype=np.uint8), g["bmp_view_1_3"])
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)        # host inputs go to the GPU when there is one
    with pytest.raises(lfsr_b200.LfsrError):
        lfsr_b200.lfutils.sai_to_rgb8_views(torch.zeros(10, 10), torch.zeros(2, 10, 10), 5)
