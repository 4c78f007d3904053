"""GPU parity of the drop-in networks: CUDA forward vs the oracle (== reference, bit-exact on CPU)
on seeded weights/inputs, and vs the committed outputs of the unmodified reference."""
import json
import os

import numpy as np
import pytest
import torch

import lfsr_b200
from oracle import lf_oracle, nets as onets, weights

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3          # north_star: max abs error <= 1e-3 on [0,1] outputs
CASES = [("MyEfficientLFNet", 4), ("MyEfficientLFNet", 2), ("EPIT", 4), ("DistgSSR", 4), ("DistgSSR", 2),
         ("LF_InterNet", 4), ("MyEfficientLFNetV4_5", 4)]
REPORT = {}


def _have(name):
    try:
        lfsr_b200.net_module(name)
        return True
    except ModuleNotFoundError:
        return False


def _net(name, scale):
    net = lfsr_b200.load_net(name, 5, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    return net.to(DEV), sd


def _dump():
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/net_parity.json", "w") as f:
        json.dump(REPORT, f, indent=1)


@pytest.mark.parametrize("name,scale", CASES)
def test_forward_p8_vs_reference_golden(name, scale, golden_dir):
    if not _have(name):
        pytest.skip(f"{name} not built yet")
    net, sd = _net(name, scale)
    x = weights.synthetic_patches(2, 5, 8, seed=7)
    y = net(x.to(DEV), [5, 5]).cpu().numpy()
    gold = np.load(f"{golden_dir}/{name}_x{scale}.npz")["p8_out"]
    err = float(np.abs(y - gold).max())
    REPORT[f"{name}_x{scale}_p8_maxabs"] = err
    _dump()
    assert err <= TOL, f"max abs err {err}"


@pytest.mark.parametrize("name,scale", CASES)
def test_forward_p32_vs_oracle(name, scale, golden_dir):
    if not _have(name):
        pytest.skip(f"{name} not built yet")
    net, sd = _net(name, scale)
    x = weights.synthetic_patches(3, 5, 32, seed=0)          # patch 0 == the golden's input
    y = net(x.to(DEV), [5, 5]).cpu()
    g = np.load(f"{golden_dir}/{name}_x{scale}.npz")
    err_g = float(np.abs(y[0, 0].numpy()[::8, ::8] - g["p32_sub"][0, 0]).max())
    torch.set_num_threads(os.cpu_count() or 1)
    y_or = onets.forward(name, x[1:2], sd, 5, scale)
    err_o = float((y[1:2] - y_or).abs().max())
    # |dPSNR| against a fixed pseudo ground truth
    hr = np.random.RandomState(5).random_sample(y_or.shape[-2:]).astype(np.float32)
    dpsnr = abs(lf_oracle.psnr_view(hr, y[1, 0].numpy()) - lf_oracle.psnr_view(hr, y_or[0, 0].numpy()))
    REPORT[f"{name}_x{scale}_p32"] = dict(maxabs_vs_golden=err_g, maxabs_vs_oracle=err_o, dpsnr=dpsnr,
                                          sum=float(y[0].double().sum()), golden_sum=float(g["p32_sum"]))
    _dump()
    assert err_g <= TOL and err_o <= TOL, (err_g, err_o)
    assert dpsnr <= 0.01


@pytest.mark.parametrize("name,scale", CASES)
def test_forward_batch64_default_init_vs_oracle(name, scale):
    """bench.py times seeded constructor-default weights at batch 64: the same weights, the same batch, against the oracle
    (first, middle and last patch of the batch; 1e-3 / 0.01 dB as everywhere)."""
    if not _have(name):
        pytest.skip(f"{name} not built yet")
    torch.manual_seed(1234)
    net = lfsr_b200.load_net(name, 5, scale).eval()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.to(DEV)
    B = 64
    x = weights.synthetic_patches(B, 5, 32, seed=21)
    y = net(x.to(DEV), [5, 5]).cpu()
    torch.set_num_threads(os.cpu_count() or 1)
    worst, worst_dp = 0.0, 0.0
    for i in (0, 31, 63):
        with torch.no_grad():
            y_or = onets.forward(name, x[i:i + 1], sd, 5, scale)
        worst = max(worst, float((y[i:i + 1] - y_or).abs().max()))
        hr = np.random.RandomState(5).random_sample(y_or.shape[-2:]).astype(np.float32)
        worst_dp = max(worst_dp, abs(lf_oracle.psnr_view(hr, y[i, 0].numpy()) - lf_oracle.psnr_view(hr, y_or[0, 0].numpy())))
    REPORT[f"{name}_x{scale}_b64_default_init"] = dict(maxabs_vs_oracle=worst, dpsnr=worst_dp,
                                                        out_absmax=float(y.abs().max()))
    _dump()
    assert worst <= TOL and worst_dp <= 0.01, (worst, worst_dp)


def test_epi_branch_packer_fallback_matches_default(monkeypatch):
    """the hybrid EPI block (depthwise taps on the CUDA cores, 1x1s on tcgen05), which runs when the operand packer returns
    None, against the default plan (taps as shifted-row tcgen05 MMAs over the fp16 trunk copy the SA tail writes): same
    network output to well inside the tolerance"""
    torch.manual_seed(1234)
    net = lfsr_b200.load_net("MyEfficientLFNet", 5, 4).eval().to(DEV)
    x = weights.synthetic_patches(4, 5, 32, seed=9).to(DEV)
    y0 = net(x, [5, 5]).clone()
    ops = net._backend(x)          # (the package is importable under two names: patch the instance the net uses)
    assert all(st["epi_img"] is not None for st in net._get_packed(x.device, ops)["stages"])
    monkeypatch.setattr(ops, "mel_epi_pack", lambda *a, **k: None)
    net.invalidate()
    y1 = net(x, [5, 5]).clone()
    d = float((y0 - y1).abs().max())
    assert 0.0 < d <= 3e-4, d


def test_invalidate_after_data_edit():
    """ADVICE r1: edits through `.data` bypass the version counter; invalidate() (also run by load_state_dict) repacks."""
    net, sd = _net("MyEfficientLFNet", 4)
    x = weights.synthetic_patches(1, 5, 8, seed=3).to(DEV)
    y0 = net(x).clone()
    for p in net.parameters():
        p.data.mul_(0.5)
    net.invalidate()
    y1 = net(x).clone()
    assert not torch.equal(y0, y1)
    net.load_state_dict(sd)                 # post-hook invalidates
    assert torch.equal(net(x), y0)


def test_scene_runner_pipeline_matches_sync(golden_dir):
    """submit()/result() with host tensors (pinned and pageable), two scenes in flight, equals the synchronous driver."""
    net, _ = _net("MyEfficientLFNet", 4)
    A, s, h0, w0 = 5, 4, 40, 48
    r = lfsr_b200.scene.SceneRunner(net, A, s, h0, w0, minibatch=6, device=DEV, world=1, rank=0, depth=2)
    scenes = []
    for k in range(3):
        rs = np.random.RandomState(40 + k)
        lr = torch.from_numpy(rs.random_sample((A * h0, A * w0)).astype(np.float32))
        hr = torch.from_numpy(rs.random_sample((A * h0 * s, A * w0 * s)).astype(np.float32))
        scenes.append((lr.pin_memory() if k % 2 == 0 else lr, hr))
    want = []
    for lr, hr in scenes:          # (the returned mosaic is the runner's slot buffer: copy it before the slot is reused)
        p, q, sr = lfsr_b200.scene.test_scene(net, lr.to(DEV), hr.to(DEV), A, s, minibatch=6)
        want.append((p, q, sr.cpu().clone()))
    tickets, got = [], []
    for lr, hr in scenes:
        tickets.append(r.submit(lr, hr))
        if len(tickets) == 2:
            p, q, sr = r.result(tickets.pop(0))
            got.append((p, q, sr.clone()))
    while tickets:
        p, q, sr = r.result(tickets.pop(0))
        got.append((p, q, sr.clone()))
    for (p0, q0, s0), (p1, q1, s1) in zip(want, got):
        assert torch.equal(s0, s1) and abs(p0 - p1) < 1e-9 and abs(q0 - q1) < 1e-9


def test_batch_slices_and_repeatability():
    net, _ = _net("MyEfficientLFNet", 4)
    x = weights.synthetic_patches(4, 5, 8, seed=3).to(DEV)
    full = net(x)
    one = torch.cat([net(x[i:i + 1]) for i in range(4)])
    assert (full - one).abs().max().item() <= 1e-5
    assert torch.equal(net(x), full)


def test_scene_loop_vs_reference_test_golden(golden_dir):
    """row L: reference train.test() on a synthetic 5x5x40x48 scene (oracle/make_golden.py)."""
    g = np.load(f"{golden_dir}/test_loop.npz")
    h0, w0 = int(g["h0"]), int(g["w0"])
    lr = np.random.RandomState(int(g["lr_seed"])).random_sample((1, 1, 5 * h0, 5 * w0)).astype(np.float32)
    hr = np.random.RandomState(int(g["hr_seed"])).random_sample((1, 1, 20 * h0, 20 * w0)).astype(np.float32)
    net, _ = _net("MyEfficientLFNet", 4)
    psnr, ssim, sr = lfsr_b200.scene.test_scene(net, torch.from_numpy(lr[0, 0]).to(DEV), torch.from_numpy(hr[0, 0]).to(DEV),
                                                5, 4, minibatch=5)
    err = float(np.abs(sr.cpu().numpy()[::4, ::4] - g["sr_sub"]).max())
    REPORT["test_loop"] = dict(maxabs=err, psnr=float(psnr), psnr_ref=float(g["psnr"]), ssim=float(ssim),
                               ssim_ref=float(g["ssim"]))
    _dump()
    assert err <= TOL
    assert abs(psnr - float(g["psnr"])) <= 0.01 and abs(ssim - float(g["ssim"])) <= 1e-4


@pytest.mark.parametrize("name", ["MyEfficientLFNet", "MyEfficientLFNetV4_5", "EPIT"])
def test_graph_replay_equals_direct_launches(name, monkeypatch):
    """SURVEY 8f-2: the per-shape CUDA graph of a forward gives bit-identical results to launching every kernel,
    survives shape changes, and is dropped when the weights change."""
    import sys
    net, _ = _net(name, 4)
    common = sys.modules[[c for c in type(net).__mro__ if c.__name__ == "LFNetBase"][0].__module__]
    xa = weights.synthetic_patches(2, 5, 8, seed=11).to(DEV)
    xb = weights.synthetic_patches(1, 5, 16, seed=12).to(DEV)
    monkeypatch.setattr(common, "USE_CUDA_GRAPH", False)
    da, db = net(xa), net(xb)
    assert not net._graphs
    monkeypatch.setattr(common, "USE_CUDA_GRAPH", True)
    for _ in range(3):
        assert torch.equal(net(xa), da) and torch.equal(net(xb), db)
    assert len(net._graphs) == 2 and net.graph_launches > 0
    xa2 = weights.synthetic_patches(2, 5, 8, seed=13).to(DEV)          # same shape, new data -> same graph, new result
    ga2 = net(xa2)
    monkeypatch.setattr(common, "USE_CUDA_GRAPH", False)
    assert torch.equal(ga2, net(xa2)) and not torch.equal(ga2, da)
    monkeypatch.setattr(common, "USE_CUDA_GRAPH", True)
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(0.5)
    out = net(xa)                                                       # repacks and re-captures
    monkeypatch.setattr(common, "USE_CUDA_GRAPH", False)
    assert torch.equal(out, net(xa)) and not torch.equal(out, da)
