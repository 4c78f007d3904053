"""Angular window tiling on rectangular grids on the B200: the four `_uv` kernels (lfsr_window_accumulate_uv,
lfsr_metric_sums_uv, lfsr_rgb_to_ycbcr_mosaic_uv, lfsr_ycbcr_to_rgb8_uv) against their torch / numpy statements and
against the square entry points, scene.super_resolve_grid / test_grid on N_u x N_v grids against per-window
super_resolve_scene plus a torch merge and against the CPU oracle, and test.py / inference.py with --grid_views (one GPU
and torchrun on two)."""
import ctypes
import os

import numpy as np
import pytest
import torch

import lfsr_b200
from lfsr_b200 import lfutils, scene
from oracle import lf_oracle, weights
import view_oracle
from test_grid_rect_cpu import oracle_rect_grid, rect_pairs
from test_multi_gpu_eval_gpu import _eval_values, _need_two, _numbers, _run
from test_view_input_cpu import _grid, _write_grid
from test_view_input_gpu import _entry

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A = 5
_UV = [(3, 5), (5, 9), (9, 5)]


def torch_merge_uv(wins, nu, nv, ang, stride=None):
    """the definition in torch fp32 on the device: per view the windows that contain it in window order, summed with `+`,
    divided by their count (as a tensor: a Python scalar divisor may become a multiply by its reciprocal)"""
    h, w = wins[0].shape[0] // ang, wins[0].shape[1] // ang
    out = torch.empty((nu, h, nv, w), dtype=torch.float32, device=wins[0].device)
    pairs = rect_pairs(nu, nv, ang, stride)
    for u in range(nu):
        for v in range(nv):
            parts = [wk.view(ang, h, ang, w)[u - ou, :, v - ov, :] for wk, (ou, ov) in zip(wins, pairs)
                     if ou <= u < ou + ang and ov <= v < ov + ang]
            acc = parts[0].clone()
            for p in parts[1:]:
                acc = acc + p
            out[u, :, v, :] = acc if len(parts) == 1 else acc / torch.full_like(acc, float(len(parts)))
    return out.view(nu * h, nv * w)


# ---- kernels --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nu,nv", _UV)
@pytest.mark.parametrize("h,w", [(8, 12), (7, 9)])                 # float4 path, scalar path
def test_window_accumulate_uv_bit_exact(nu, nv, h, w):
    ops = lfsr_b200.kernels.default_ops()
    g = torch.Generator(device=DEV).manual_seed(nu * 100 + nv * 10 + w)
    for ang in (a for a in (3, 5) if a <= min(nu, nv)):
        for t in [None] + list(range(1, ang)):
            plan = scene.window_plan((nu, nv), ang, t)
            wins = [torch.rand((ang * h, ang * w), generator=g, device=DEV) * 4 - 2 for _ in plan]
            grid = torch.full((nu * h, nv * w), float("nan"), device=DEV)     # every pixel is stored before it is read
            for (ou, ov, modes), wk in zip(plan, wins):
                ops.window_accumulate_uv(wk, grid, ang, nu, nv, h, w, ou, ov, modes)
            want = torch_merge_uv(wins, nu, nv, ang, t)
            assert torch.equal(grid, want), (ang, t, float((grid - want).abs().max()))


@pytest.mark.parametrize("n,h,w", [(7, 8, 12), (9, 7, 9)])
def test_window_accumulate_uv_equal_sizes_is_the_square_entry(n, h, w):
    ops = lfsr_b200.kernels.default_ops()
    g = torch.Generator(device=DEV).manual_seed(n)
    plan = scene.window_plan(n, A, 2)
    wins = [torch.rand((A * h, A * w), generator=g, device=DEV) for _ in plan]
    g1 = torch.full((n * h, n * w), float("nan"), device=DEV)
    g2 = g1.clone()
    N = lfsr_b200.kernels.N
    stream = torch.cuda.current_stream(DEV).cuda_stream
    for (ou, ov, modes), wk in zip(plan, wins):
        m = (ctypes.c_int32 * (A * A))(*modes)                  # the square C entry point itself
        N.check(ops.lib.lfsr_window_accumulate(wk.data_ptr(), g1.data_ptr(), A, n, h, w, ou, ov, m, stream),
                "lfsr_window_accumulate")
        ops.window_accumulate_uv(wk, g2, A, n, n, h, w, ou, ov, modes)
    assert torch.equal(g1, g2)


def test_window_accumulate_uv_rejects_bad_input():
    ops = lfsr_b200.kernels.default_ops()
    LfsrError = lfsr_b200.kernels.N.LfsrError
    win = torch.zeros((3 * 4, 3 * 4), device=DEV)
    grid = torch.zeros((5 * 4, 7 * 4), device=DEV)
    ok = [0] * 9
    ops.window_accumulate_uv(win, grid, 3, 5, 7, 4, 4, 2, 4, ok)
    # per-axis mode bound: min(3, 5 - 3 + 1) * min(3, 7 - 3 + 1) = 9
    ops.window_accumulate_uv(win, grid, 3, 5, 7, 4, 4, 0, 0, [9] * 9)
    for args, words in [((3, 5, 7, 4, 4, 3, 0, ok), "outside"), ((3, 5, 7, 4, 4, 0, 5, ok), "outside"),
                        ((3, 5, 2, 4, 4, 0, 0, ok), "smaller"), ((3, 2, 7, 4, 4, 0, 0, ok), "smaller"),
                        ((3, 5, 7, 4, 4, 0, 0, [0] * 8 + [10]), "bad mode"),
                        ((3, 5, 7, 4, 4, 0, 0, [0] * 8 + [-1]), "bad mode")]:
        with pytest.raises(LfsrError, match=words):
            ops.window_accumulate_uv(win, grid, *args)
    torch.cuda.synchronize()


def _metric_inputs(au, av, hv, wv, seed):
    rs = np.random.RandomState(seed)
    la = torch.from_numpy(rs.random_sample((au * hv, av * wv)).astype(np.float32)).to(DEV)
    ou = (la + 0.03 * torch.randn_like(la)).clamp_(0, 1)
    return la, ou


@pytest.mark.parametrize("au,av", _UV)
def test_metric_sums_uv(au, av):
    """per view the sums of a launch over that view alone (fp64 atomics: equal up to the summation order) and the
    oracle's SSIM; view order row-major over the ang_u x ang_v mosaic"""
    ops = lfsr_b200.kernels.default_ops()
    hv, wv = 24, 40
    la, ou = _metric_inputs(au, av, hv, wv, au * 10 + av)
    acc = torch.zeros(2 * au * av, dtype=torch.float64, device=DEV)
    ops.metric_sums_uv(la, ou, au, av, hv, wv, acc)
    got = acc.view(au, av, 2).cpu().numpy()
    L, O = la.view(au, hv, av, wv), ou.view(au, hv, av, wv)
    for u in range(au):
        for v in range(av):
            one = torch.zeros(2, dtype=torch.float64, device=DEV)
            ops.metric_sums(L[u, :, v, :].contiguous(), O[u, :, v, :].contiguous(), 1, hv, wv, one)
            np.testing.assert_allclose(got[u, v], one.cpu().numpy(), rtol=1e-12, atol=0)
    a, b = la.cpu().numpy().reshape(au, hv, av, wv), ou.cpu().numpy().reshape(au, hv, av, wv)
    ssim = np.array([[lf_oracle.ssim_view(a[u, :, v, :], b[u, :, v, :]) for v in range(av)] for u in range(au)])
    assert np.abs(got[..., 1] / ((hv - 10) * (wv - 10)) - ssim).max() <= 1e-5
    se = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).sum(axis=(1, 3))
    np.testing.assert_allclose(got[..., 0], se, rtol=1e-12)


def test_metric_sums_uv_equal_sizes_is_the_square_entry():
    ops = lfsr_b200.kernels.default_ops()
    la, ou = _metric_inputs(5, 5, 32, 32, 1)
    a1 = torch.zeros(50, dtype=torch.float64, device=DEV)
    a2 = torch.zeros(50, dtype=torch.float64, device=DEV)
    ops.metric_sums(la, ou, 5, 32, 32, a1)
    ops.metric_sums_uv(la, ou, 5, 5, 32, 32, a2)
    assert torch.allclose(a1, a2, rtol=1e-12, atol=0)


@pytest.mark.parametrize("au,av", _UV)
@pytest.mark.parametrize("dtype", ["u8", "f64"])
def test_rgb_to_ycbcr_mosaic_uv_bit_exact(au, av, dtype):
    h, w = 7, 11
    rs = np.random.RandomState(au * 10 + av)
    if dtype == "u8":
        v = rs.randint(0, 256, (au, av, h, w, 3)).astype(np.uint8)
        v.reshape(-1, 3)[:256, 0] = np.arange(256)
        x = v.astype(np.float64) / 255.0
    else:
        v = x = rs.random_sample((au, av, h, w, 3))
    want = view_oracle.rgb2ycbcr(x)
    want_y = view_oracle._views_to_sai(want[..., 0]).astype("single")
    want_c = np.ascontiguousarray(view_oracle._views_to_sai(want[..., 1:3]).transpose(2, 0, 1)).astype("single")
    t = torch.from_numpy(v).to(DEV)
    y, c = lfutils.rgb_to_ycbcr_mosaic(t, (au, av))
    assert y.shape == (au * h, av * w) and c.shape == (2, au * h, av * w)
    assert np.array_equal(y.cpu().numpy(), want_y) and np.array_equal(c.cpu().numpy(), want_c)
    y, c = lfutils.rgb_to_ycbcr_mosaic(t.reshape(au * av, h, w, 3), (au, av), y=False)
    assert y is None and np.array_equal(c.cpu().numpy(), want_c)


@pytest.mark.parametrize("dtype", ["u8", "f64"])
def test_rgb_to_ycbcr_mosaic_uv_equal_sizes_is_the_square_entry(dtype):
    rs = np.random.RandomState(4)
    v = rs.randint(0, 256, (5, 5, 9, 12, 3)).astype(np.uint8) if dtype == "u8" else rs.random_sample((5, 5, 9, 12, 3))
    t = torch.from_numpy(v).to(DEV)
    y1, c1 = lfutils.rgb_to_ycbcr_mosaic(t, 5)
    y2, c2 = lfutils.rgb_to_ycbcr_mosaic(t, (5, 5))
    assert torch.equal(y1, y2) and torch.equal(c1, c2)


def _rgb8_views_uv(y, c, au, av):
    """lf_oracle.sai_to_rgb8_views for an ang_u x ang_v mosaic"""
    ycbcr = np.concatenate([y[None], c], 0).transpose(1, 2, 0)
    rgb = (lf_oracle.ycbcr2rgb(ycbcr).clip(0, 1) * 255).astype("uint8")
    H, W, _ = rgb.shape
    return np.ascontiguousarray(rgb.reshape(au, H // au, av, W // av, 3).transpose(0, 2, 1, 3, 4))


@pytest.mark.parametrize("au,av", _UV)
def test_ycbcr_to_rgb8_uv_bit_exact(au, av):
    h, w = 9, 13
    rs = np.random.RandomState(au + 7 * av)
    y = rs.uniform(-0.05, 1.05, (au * h, av * w)).astype(np.float32)
    c = rs.uniform(0.2, 0.8, (2, au * h, av * w)).astype(np.float32)
    got = lfutils.sai_to_rgb8_views(torch.from_numpy(y).to(DEV), torch.from_numpy(c).to(DEV), (au, av))
    assert got.shape == (au, av, h, w, 3)
    assert np.array_equal(got.cpu().numpy(), _rgb8_views_uv(y, c, au, av))


def test_ycbcr_to_rgb8_uv_equal_sizes_is_the_square_entry():
    rs = np.random.RandomState(8)
    y = torch.from_numpy(rs.uniform(-0.05, 1.05, (5 * 9, 5 * 12)).astype(np.float32)).to(DEV)
    c = torch.from_numpy(rs.uniform(0.2, 0.8, (2, 5 * 9, 5 * 12)).astype(np.float32)).to(DEV)
    assert torch.equal(lfutils.sai_to_rgb8_views(y, c, 5), lfutils.sai_to_rgb8_views(y, c, (5, 5)))


# ---- scene driver ---------------------------------------------------------------------------------------------------------
def _load(name, scale):
    net = lfsr_b200.load_net(name, A, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    return net.to(DEV), sd


@pytest.mark.parametrize("t,ens", [(None, False), (2, False), (None, True)])
def test_rect_grid_equals_torch_composition(t, ens):
    nu, nv, scale, h0, w0 = 9, 13, 4, 32, 32
    net, _ = _load("MyEfficientLFNet", scale)
    lr = torch.from_numpy(np.random.RandomState(2).random_sample((nu * h0, nv * w0)).astype(np.float32)).to(DEV)
    views = lr.view(nu, h0, nv, w0)
    with torch.no_grad():
        got = scene.super_resolve_grid(net, lr, (nu, nv), A, scale, ang_stride=t, self_ensemble=ens)
        wins = [scene.super_resolve_scene(net, views[ou:ou + A, :, ov:ov + A, :].reshape(A * h0, A * w0), A, scale,
                                          self_ensemble=ens).clone() for ou, ov in rect_pairs(nu, nv, A, t)]
    assert len(wins) == (2 * 3 if t is None else 3 * 5)
    want = torch_merge_uv(wins, nu, nv, A, t)
    torch.cuda.synchronize()
    assert got.shape == (nu * h0 * scale, nv * w0 * scale)
    assert torch.equal(got, want), float((got - want).abs().max())


def test_square_pair_is_the_int():
    n, scale, h0, w0 = 7, 4, 32, 32
    net, _ = _load("MyEfficientLFNet", scale)
    rs = np.random.RandomState(3)
    lr = torch.from_numpy(rs.random_sample((n * h0, n * w0)).astype(np.float32)).to(DEV)
    hr = torch.from_numpy(rs.random_sample((n * h0 * scale, n * w0 * scale)).astype(np.float32)).to(DEV)
    with torch.no_grad():
        s1 = scene.super_resolve_grid(net, lr, n, A, scale, ang_stride=2)
        s2 = scene.super_resolve_grid(net, lr, (n, n), A, scale, ang_stride=2)
        p1, q1, t1 = scene.test_grid(net, lr, hr, n, A, scale)
        p2, q2, t2 = scene.test_grid(net, lr, hr, (n, n), A, scale)
    torch.cuda.synchronize()
    assert torch.equal(s1, s2) and torch.equal(t1, t2)
    np.testing.assert_allclose([p2, q2], [p1, q1], rtol=1e-9)          # fp64 atomics: equal up to summation order


@pytest.mark.parametrize("name,scale", [("MyEfficientLFNet", 4), ("DistgSSR", 2)])
def test_rect_grid_against_oracle(name, scale):
    nu, nv, h0, w0 = 7, 9, 32, 32
    net, sd = _load(name, scale)
    rs = np.random.RandomState(5)
    lr = rs.random_sample((nu * h0, nv * w0)).astype(np.float32)
    hr = rs.random_sample((nu * h0 * scale, nv * w0 * scale)).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr = scene.test_grid(net, torch.from_numpy(lr).to(DEV), torch.from_numpy(hr), (nu, nv), A, scale)
    want = oracle_rect_grid(name, lr, sd, nu, nv, A, scale, 32, 16, h0, w0)
    la, ou = hr.reshape(nu, h0 * scale, nv, w0 * scale), want.reshape(nu, h0 * scale, nv, w0 * scale)
    pv = np.array([[lf_oracle.psnr_view(la[u, :, v, :], ou[u, :, v, :]) for v in range(nv)] for u in range(nu)], np.float32)
    sv = np.array([[lf_oracle.ssim_view(la[u, :, v, :], ou[u, :, v, :]) for v in range(nv)] for u in range(nu)], np.float32)
    assert float(np.abs(sr.cpu().numpy() - want).max()) <= 1e-3
    assert abs(psnr - pv.sum() / (pv > 0).sum()) <= 0.01 and abs(ssim - sv.sum() / (sv > 0).sum()) <= 1e-3


# ---- test.py / inference.py ------------------------------------------------------------------------------------------------
_DATASETS = [("all", (9, 13), (9, 13)), ("5x7", (9, 9), (5, 7))]


@pytest.mark.parametrize("grid_views,shape,views", _DATASETS)
def test_test_py_grid_views(tmp_path, grid_views, shape, views):
    import train
    from types import SimpleNamespace
    from utils.utils_datasets import _batch1, parse_grid_views, read_views
    name, scale = "MyEfficientLFNet", 4
    data = tmp_path / "data"
    _write_grid(str(data / "Set" / "a"), _grid(*shape, 64, 80, seed=1), "png")
    _write_grid(str(data / "Set" / "b"), _grid(*shape, 64, 64, seed=2), "png")
    scenes = ["a", "b"]
    net, sd = _load(name, scale)
    ckpt = tmp_path / "ck.pth"
    torch.save({"state_dict": sd}, ckpt)
    out, log = _entry(tmp_path, "run", "test.py", ["--model_name", name, "--angRes", "5", "--scale_factor", str(scale),
                                                   "--path_pre_pth", str(ckpt), "--path_for_test", str(data) + "/",
                                                   "--full_grid", "1", "--grid_views", grid_views])
    grid = parse_grid_views(grid_views, True)
    prepared = [lfutils.prepare_views(read_views(str(data / "Set" / s), A, full_grid=True, grid=grid), views, scale, "hr")
                for s in scenes]
    psnr, ssim = [], []
    for lr, hr, _ in prepared:
        with torch.no_grad():
            p, s, _ = scene.test_grid(net, lr, hr, views, A, scale)
        psnr.append(p)
        ssim.append(s)
    line = [ln for ln in out.splitlines() if ln.startswith("Test on Set")]
    assert line == ["Test on Set, psnr/ssim is %.3f/%.4f" % (np.mean(psnr), np.mean(ssim))], out
    rows = [r for r in _eval_values(list(log.rglob("evaluation.*"))) if r[0] == "Set" and r[1] in scenes]
    np.testing.assert_allclose([r[2:] for r in rows], [[float("%.6f" % p), float("%.6f" % s)] for p, s in zip(psnr, ssim)],
                               rtol=1e-9)
    for s in scenes:
        files = sorted(os.path.basename(str(f)) for f in log.rglob("TEST/Set/%s/View_*_*.bmp" % s))
        assert files == sorted("View_%d_%d.bmp" % (i, j) for i in range(views[0]) for j in range(views[1]))
    loader = [_batch1(lr[None], hr[None], cb, A, A, s, views) for (lr, hr, cb), s in zip(prepared, scenes)]
    args = SimpleNamespace(scale_factor=scale, patch_size_for_test=32, stride_for_test=16, minibatch=64, self_ensemble=0,
                           angRes_in=A, angRes_out=A, full_grid=1, ang_stride=0, grid_views=grid_views)
    with torch.no_grad():
        p2, s2, names = train.test(loader, DEV, net, args)
    assert names == scenes
    np.testing.assert_allclose([p2, s2], [psnr, ssim], rtol=1e-9)


@pytest.mark.parametrize("grid_views,shape,views", _DATASETS)
@pytest.mark.parametrize("ens", [0, 1])
def test_inference_py_grid_views(tmp_path, grid_views, shape, views, ens):
    from train import _write_views
    from utils.utils_datasets import parse_grid_views, read_views
    name, scale = "DistgSSR", 2
    data = tmp_path / "data"
    _write_grid(str(data / "Set" / "p"), _grid(*shape, 32, 40, seed=5), "png")
    _write_grid(str(data / "Set" / "q"), _grid(*shape, 36, 32, seed=6), "bmp")
    net, sd = _load(name, scale)
    ckpt = tmp_path / "ck.pth"
    torch.save({"state_dict": sd}, ckpt)
    _, log = _entry(tmp_path, "run", "inference.py", [
        "--model_name", name, "--angRes", "5", "--scale_factor", str(scale), "--path_pre_pth", str(ckpt),
        "--path_for_test", str(data) + "/", "--self_ensemble", str(ens), "--full_grid", "1", "--grid_views", grid_views])
    test_dir = next(log.rglob("TEST"))
    grid = parse_grid_views(grid_views, True)
    for s in ("p", "q"):
        lr, _, cb = lfutils.prepare_views(read_views(str(data / "Set" / s), A, full_grid=True, grid=grid), views, scale,
                                          "lr")
        with torch.no_grad():
            sr = scene.super_resolve_grid(net, lr, views, A, scale, self_ensemble=bool(ens))
        ref = tmp_path / "ref"
        ref.mkdir(exist_ok=True)
        _write_views(ref, s, sr, cb, views)
        files = sorted(os.listdir(test_dir / "Set" / s))
        assert files == sorted("View_%d_%d.bmp" % (i, j) for i in range(views[0]) for j in range(views[1]))
        for f in files:
            assert (test_dir / "Set" / s / f).read_bytes() == (ref / s / f).read_bytes(), (s, f)


def test_test_py_grid_views_two_gpus(tmp_path):
    """3 scenes of 7 x 9 views on 2 ranks: scenes 0 / 1 are one full round, scene 2 is the tail, whose windows are
    row-sharded"""
    _need_two()
    data = tmp_path / "data"
    for i in range(3):
        _write_grid(str(data / "Set" / ("s%d" % i)), _grid(7, 9, 128, 128, seed=30 + i), "png")
    ckpt = tmp_path / "MyEfficientLFNet_x4.pth"
    torch.save({"state_dict": weights.make_state_dict("MyEfficientLFNet", 4, 1234)}, ckpt)
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--path_pre_pth", str(ckpt),
             "--path_for_test", str(data) + "/", "--full_grid", "1", "--grid_views", "all"]
    out1, writes1, bmps1, ev1 = _run(tmp_path, "single", "test.py", flags, 1)
    out2, writes2, bmps2, ev2 = _run(tmp_path, "multi", "test.py", flags, 2)
    assert len(bmps1) == 3 * 63 and set(bmps2) == set(bmps1)
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
