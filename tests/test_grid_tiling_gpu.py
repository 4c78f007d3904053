"""Angular window tiling on the B200: lfsr_window_accumulate bit-exact against torch's fp32 `+` and `/` in window order,
scene.super_resolve_grid / test_grid against super_resolve_scene / test_scene and against the CPU oracle, and test.py /
inference.py with --full_grid 1 (one GPU and torchrun on two) on datasets of View_u_v.png|bmp folders larger than 5x5."""
import os

import numpy as np
import pytest
import torch

import lfsr_b200
from lfsr_b200 import lfutils, scene
from oracle import lf_oracle, weights
from test_grid_tiling_cpu import oracle_grid, window_pairs
from test_multi_gpu_eval_gpu import _eval_values, _need_two, _numbers, _run
from test_view_input_cpu import _grid, _write_grid
from test_view_input_gpu import _entry

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A = 5


def torch_merge(wins, n, ang, stride=None):
    """the definition in torch fp32 on the device: per view the windows that contain it in window order, summed with `+`,
    divided by their count (as a tensor: a Python scalar divisor may become a multiply by its reciprocal)"""
    h, w = wins[0].shape[0] // ang, wins[0].shape[1] // ang
    out = torch.empty((n, h, n, w), dtype=torch.float32, device=wins[0].device)
    pairs = window_pairs(n, ang, stride)
    for u in range(n):
        for v in range(n):
            parts = [wk.view(ang, h, ang, w)[u - ou, :, v - ov, :] for wk, (ou, ov) in zip(wins, pairs)
                     if ou <= u < ou + ang and ov <= v < ov + ang]
            acc = parts[0].clone()
            for p in parts[1:]:
                acc = acc + p
            out[u, :, v, :] = acc if len(parts) == 1 else acc / torch.full_like(acc, float(len(parts)))
    return out.view(n * h, n * w)


# ---- kernel ---------------------------------------------------------------------------------------------------------------
_GEOMS = [(8, 12), (7, 9), (6, 10), (5, 16), (9, 3)]          # float4 path, odd, non-square (scalar), float4, scalar


@pytest.mark.parametrize("ang", [3, 5])
@pytest.mark.parametrize("n", list(range(5, 15)))
def test_window_accumulate_bit_exact(ang, n):
    ops = lfsr_b200.kernels.default_ops()
    h, w = _GEOMS[n % len(_GEOMS)]
    g = torch.Generator(device=DEV).manual_seed(n * 100 + ang)
    for t in ([None] + ([1] if n > ang else [])):
        plan = scene.window_plan(n, ang, t)
        wins = [torch.rand((ang * h, ang * w), generator=g, device=DEV) * 4 - 2 for _ in plan]
        grid = torch.full((n * h, n * w), float("nan"), device=DEV)      # every pixel is stored before it is read
        for (ou, ov, modes), wk in zip(plan, wins):
            ops.window_accumulate(wk, grid, ang, n, h, w, ou, ov, modes)
        want = torch_merge(wins, n, ang, t)
        assert torch.equal(grid, want), (t, float((grid - want).abs().max()))
        used = {m if m < 2 else 2 for _, _, modes in plan for m in modes}
        assert used == ({0} if n == ang else {0, 1, 2})


def test_window_accumulate_rejects_bad_input():
    ops = lfsr_b200.kernels.default_ops()
    LfsrError = lfsr_b200.kernels.N.LfsrError           # the class of the package the launcher lives in
    win = torch.zeros((3 * 4, 3 * 4), device=DEV)
    grid = torch.zeros((5 * 4, 5 * 4), device=DEV)
    ok = [0] * 9
    ops.window_accumulate(win, grid, 3, 5, 4, 4, 2, 2, ok)
    for args, words in [((3, 5, 4, 4, 3, 0, ok), "outside"), ((3, 5, 4, 4, 0, -1, ok), "outside"),
                        ((3, 2, 4, 4, 0, 0, ok), "smaller"), ((3, 5, 4, 4, 0, 0, [0] * 8 + [-1]), "bad mode"),
                        ((3, 5, 4, 4, 0, 0, [0] * 8 + [10]), "bad mode")]:
        with pytest.raises(LfsrError, match=words):
            ops.window_accumulate(win, grid, *args)
    with pytest.raises(LfsrError, match="overlap"):
        ops.window_accumulate(grid.view(-1)[:144].view(12, 12), grid, 3, 5, 4, 4, 0, 0, ok)
    torch.cuda.synchronize()


# ---- scene driver ---------------------------------------------------------------------------------------------------------
def _load(name, scale):
    net = lfsr_b200.load_net(name, A, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    return net.to(DEV), sd


def test_single_window_is_the_scene():
    net, _ = _load("MyEfficientLFNet", 4)
    rs = np.random.RandomState(1)
    lr = torch.from_numpy(rs.random_sample((A * 32, A * 48)).astype(np.float32)).to(DEV)
    hr = torch.from_numpy(rs.random_sample((A * 128, A * 192)).astype(np.float32)).to(DEV)
    with torch.no_grad():
        sr1 = scene.super_resolve_scene(net, lr, A, 4).clone()
        sr2 = scene.super_resolve_grid(net, lr, A, A, 4)
        p1, s1, t1 = scene.test_scene(net, lr, hr, A, 4)
        t1 = t1.clone()
        p2, s2, t2 = scene.test_grid(net, lr, hr, A, A, 4)
    torch.cuda.synchronize()
    assert torch.equal(sr1, sr2) and torch.equal(t1, t2) and torch.equal(sr1, t1)
    # the per-view metric sums are fp64 atomics, so equal mosaics give equal metrics up to their summation order
    np.testing.assert_allclose([p2, s2], [p1, s1], rtol=1e-9)


@pytest.mark.parametrize("t,ens", [(None, False), (2, False), (None, True)])
def test_grid_equals_torch_composition(t, ens):
    n, scale, h0, w0 = 9, 4, 32, 32
    net, _ = _load("MyEfficientLFNet", scale)
    lr = torch.from_numpy(np.random.RandomState(2).random_sample((n * h0, n * w0)).astype(np.float32)).to(DEV)
    views = lr.view(n, h0, n, w0)
    with torch.no_grad():
        got = scene.super_resolve_grid(net, lr, n, A, scale, ang_stride=t, self_ensemble=ens)
        wins = [scene.super_resolve_scene(net, views[ou:ou + A, :, ov:ov + A, :].reshape(A * h0, A * w0), A, scale,
                                          self_ensemble=ens).clone() for ou, ov in window_pairs(n, A, t)]
    assert len(wins) == (4 if t is None else 9)
    want = torch_merge(wins, n, A, t)
    torch.cuda.synchronize()
    assert torch.equal(got, want), float((got - want).abs().max())


@pytest.mark.parametrize("name,scale", [("MyEfficientLFNet", 4), ("DistgSSR", 2)])
def test_grid_against_oracle(name, scale):
    n, h0, w0 = 7, 32, 32
    net, sd = _load(name, scale)
    rs = np.random.RandomState(5)
    lr = rs.random_sample((n * h0, n * w0)).astype(np.float32)
    hr = rs.random_sample((n * h0 * scale, n * w0 * scale)).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr = scene.test_grid(net, torch.from_numpy(lr).to(DEV), torch.from_numpy(hr), n, A, scale)
    want = oracle_grid(name, lr, sd, n, A, scale, 32, 16, h0, w0)
    p_or, s_or, _, _ = lf_oracle.cal_metrics(hr, want, n)
    assert float(np.abs(sr.cpu().numpy() - want).max()) <= 1e-3
    assert abs(psnr - p_or) <= 0.01 and abs(ssim - s_or) <= 1e-3


# ---- test.py / inference.py ------------------------------------------------------------------------------------------------
def test_test_py_full_grid(tmp_path):
    import train
    from types import SimpleNamespace
    from utils.utils_datasets import _batch1, read_views
    name, scale = "MyEfficientLFNet", 4
    data = tmp_path / "data"
    _write_grid(str(data / "Set" / "a9"), _grid(9, 9, 64, 80, seed=1), "png")
    _write_grid(str(data / "Set" / "b9"), _grid(9, 9, 64, 64, seed=2), "png")
    scenes = ["a9", "b9"]
    net, sd = _load(name, scale)
    ckpt = tmp_path / "ck.pth"
    torch.save({"state_dict": sd}, ckpt)
    out, log = _entry(tmp_path, "run", "test.py", ["--model_name", name, "--angRes", "5", "--scale_factor", str(scale),
                                                   "--path_pre_pth", str(ckpt), "--path_for_test", str(data) + "/",
                                                   "--full_grid", "1"])
    prepared = [lfutils.prepare_views(read_views(str(data / "Set" / s), A, full_grid=True), 9, scale, "hr") for s in scenes]
    psnr, ssim = [], []
    for lr, hr, _ in prepared:
        with torch.no_grad():
            p, s, _ = scene.test_grid(net, lr, hr, 9, A, scale)
        psnr.append(p)
        ssim.append(s)
    line = [ln for ln in out.splitlines() if ln.startswith("Test on Set")]
    assert line == ["Test on Set, psnr/ssim is %.3f/%.4f" % (np.mean(psnr), np.mean(ssim))], out
    rows = [r for r in _eval_values(list(log.rglob("evaluation.*"))) if r[0] == "Set" and r[1] in scenes]
    np.testing.assert_allclose([r[2:] for r in rows], [[float("%.6f" % p), float("%.6f" % s)] for p, s in zip(psnr, ssim)],
                               rtol=1e-9)
    for s in scenes:
        assert len(list(log.rglob("TEST/Set/%s/View_*_*.bmp" % s))) == 81
    # train.test on an in-memory loader of the same tensors gives the same numbers
    loader = [_batch1(lr[None], hr[None], cb, A, A, s, 9) for (lr, hr, cb), s in zip(prepared, scenes)]
    args = SimpleNamespace(scale_factor=scale, patch_size_for_test=32, stride_for_test=16, minibatch=64, self_ensemble=0,
                           angRes_in=A, angRes_out=A, full_grid=1, ang_stride=0)
    with torch.no_grad():
        p2, s2, names = train.test(loader, DEV, net, args)
    assert names == scenes
    np.testing.assert_allclose([p2, s2], [psnr, ssim], rtol=1e-9)


@pytest.mark.parametrize("ens", [0, 1])
def test_inference_py_full_grid(tmp_path, ens):
    from train import _write_views
    from utils.utils_datasets import read_views
    name, scale = "DistgSSR", 2
    data = tmp_path / "data"
    _write_grid(str(data / "Set" / "p"), _grid(9, 9, 32, 40, seed=5), "png")
    _write_grid(str(data / "Set" / "q"), _grid(9, 7, 36, 32, seed=6), "bmp")
    net, sd = _load(name, scale)
    ckpt = tmp_path / "ck.pth"
    torch.save({"state_dict": sd}, ckpt)
    _, log = _entry(tmp_path, "run", "inference.py", [
        "--model_name", name, "--angRes", "5", "--scale_factor", str(scale), "--path_pre_pth", str(ckpt),
        "--path_for_test", str(data) + "/", "--self_ensemble", str(ens), "--full_grid", "1"])
    test_dir = next(log.rglob("TEST"))
    for s, n in (("p", 9), ("q", 7)):
        lr, _, cb = lfutils.prepare_views(read_views(str(data / "Set" / s), A, full_grid=True), n, scale, "lr")
        with torch.no_grad():
            sr = scene.super_resolve_grid(net, lr, n, A, scale, self_ensemble=bool(ens))
        ref = tmp_path / "ref"
        ref.mkdir(exist_ok=True)
        _write_views(ref, s, sr, cb, n)
        files = sorted(os.listdir(test_dir / "Set" / s))
        assert files == sorted("View_%d_%d.bmp" % (i, j) for i in range(n) for j in range(n))
        for f in files:
            assert (test_dir / "Set" / s / f).read_bytes() == (ref / s / f).read_bytes(), (s, f)


def test_test_py_full_grid_two_gpus(tmp_path):
    """3 scenes on 2 ranks: scenes 0 / 1 are one full round, scene 2 is the tail, whose windows are row-sharded"""
    _need_two()
    data = tmp_path / "data"
    for i in range(3):
        _write_grid(str(data / "Set" / ("s%d" % i)), _grid(7, 7, 128, 128, seed=20 + i), "png")
    ckpt = tmp_path / "MyEfficientLFNet_x4.pth"
    torch.save({"state_dict": weights.make_state_dict("MyEfficientLFNet", 4, 1234)}, ckpt)
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--path_pre_pth", str(ckpt),
             "--path_for_test", str(data) + "/", "--full_grid", "1"]
    out1, writes1, bmps1, ev1 = _run(tmp_path, "single", "test.py", flags, 1)
    out2, writes2, bmps2, ev2 = _run(tmp_path, "multi", "test.py", flags, 2)
    assert len(bmps1) == 3 * 49 and set(bmps2) == set(bmps1)
    bad = [k for k in bmps1 if bmps1[k] != bmps2[k]]
    assert not bad, bad[:5]
    assert sorted(writes2) == sorted(writes1) == sorted(bmps1)          # every view written once, by one rank
    for key in ("Test on ", "The mean psnr"):
        l1 = [line for line in out1.splitlines() if line.startswith(key)]
        l2 = [line for line in out2.splitlines() if line.startswith(key)]
        assert len(l1) == len(l2) == 1, (l1, l2)                        # printed by rank 0 only
        np.testing.assert_allclose(_numbers(l2[0]), _numbers(l1[0]), rtol=1e-9)
    v1, v2 = _eval_values(ev1), _eval_values(ev2)
    assert [v[:2] for v in v1] == [v[:2] for v in v2] and len(v1) == 3 + 2
    np.testing.assert_allclose([v[2:] for v in v2], [v[2:] for v in v1], rtol=1e-9)
