"""Light fields stored as view images on the B200: lfsr_rgb_to_ycbcr_mosaic and the batched view resampling bit-exact
against their statements, lfutils.prepare_views against the numpy oracle, and test.py / inference.py (one GPU and
torchrun on two) on datasets of View_u_v.png|bmp folders."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import lfsr_b200
from lfsr_b200 import lfutils
from oracle import lf_oracle, nets as onets, weights
import view_oracle
from test_multi_gpu_eval_gpu import _compare, _eval_values, _need_two, _run
from test_view_input_cpu import _grid, _write_grid

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
A = 5


def _sai(v):
    return view_oracle._views_to_sai(v)


# ---- kernels --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ang,h,w", [(3, 7, 11), (5, 13, 9), (5, 16, 24)])
@pytest.mark.parametrize("dtype", ["u8", "f64"])
def test_rgb_to_ycbcr_mosaic_bit_exact(ang, h, w, dtype):
    rs = np.random.RandomState(ang * 100 + h)
    if dtype == "u8":
        v = rs.randint(0, 256, (ang, ang, h, w, 3)).astype(np.uint8)
        v.reshape(-1, 3)[:256, 0] = np.arange(256)                          # every uint8 value once
        x = v.astype(np.float64) / 255.0
    else:
        v = x = rs.random_sample((ang, ang, h, w, 3))
    want = view_oracle.rgb2ycbcr(x)
    want_y = _sai(want[..., 0]).astype("single")
    want_c = np.ascontiguousarray(_sai(want[..., 1:3]).transpose(2, 0, 1)).astype("single")
    t = torch.from_numpy(v).to(DEV)
    y, c = lfutils.rgb_to_ycbcr_mosaic(t, ang)
    assert np.array_equal(y.cpu().numpy(), want_y) and np.array_equal(c.cpu().numpy(), want_c)
    y, c = lfutils.rgb_to_ycbcr_mosaic(t, ang, cbcr=False)
    assert c is None and np.array_equal(y.cpu().numpy(), want_y)
    y, c = lfutils.rgb_to_ycbcr_mosaic(t.reshape(ang * ang, h, w, 3), ang, y=False)
    assert y is None and np.array_equal(c.cpu().numpy(), want_c)


@pytest.mark.parametrize("scale,h,w", [(0.5, 32, 24), (0.25, 48, 36), (2.0, 13, 9), (4.0, 7, 11), (0.5, 13, 17)])
def test_imresize_views_equals_per_view_imresize(scale, h, w):
    v = torch.from_numpy(np.random.RandomState(5).random_sample((3, 4, h, w, 3))).to(DEV)
    got = lfutils.imresize_views(v, scale)
    want = torch.stack([torch.stack([lfutils.imresize(v[i, j], scale) for j in range(4)]) for i in range(3)])
    assert got.shape == want.shape and torch.equal(got, want)


def _composition(rgb8, scale, kind):
    """prepare_views spelled out with per-view lfutils.imresize and the colour kernel."""
    x8 = torch.from_numpy(np.ascontiguousarray(lfutils.central_views(rgb8, A, scale))).to(DEV)
    x = torch.from_numpy(np.arange(256) / 255.0).to(DEV)[x8.long()]
    per_view = lambda t, s: torch.stack([torch.stack([lfutils.imresize(t[i, j], s) for j in range(A)]) for i in range(A)])
    if kind == "hr":
        hr = lfutils.rgb_to_ycbcr_mosaic(x8, A, cbcr=False)[0]
        lr_rgb = per_view(x, 1.0 / scale)
        lr = lfutils.rgb_to_ycbcr_mosaic(lr_rgb, A, cbcr=False)[0]
    else:
        hr, lr_rgb = None, x
        lr = lfutils.rgb_to_ycbcr_mosaic(x8, A, cbcr=False)[0]
    return lr, hr, lfutils.rgb_to_ycbcr_mosaic(per_view(lr_rgb, float(scale)), A, y=False)[1]


@pytest.mark.parametrize("kind", ["hr", "lr"])
@pytest.mark.parametrize("U,H,W,scale", [(7, 34, 26, 4), (5, 30, 41, 2)])
def test_prepare_views_against_oracle(kind, U, H, W, scale):
    g = _grid(U, U, H, W, seed=H)
    got = lfutils.prepare_views(g, A, scale, kind)
    want = view_oracle.prepare_views(g, A, scale, kind)
    comp = _composition(g, scale, kind)
    for a, b, c in zip(got, want, comp):
        if b is None:
            assert a is None and c is None
            continue
        assert a.is_cuda and a.dtype == torch.float32
        np.testing.assert_array_max_ulp(a.cpu().numpy(), b, maxulp=1)
        assert torch.equal(a, c)


# ---- test.py / inference.py ------------------------------------------------------------------------------------------------
def _dataset(root):
    """3 scenes: a 9x9 PNG grid, a 5x5 BMP grid and non-square 96x80 views, smooth seeded content."""
    _write_grid(os.path.join(root, "Set", "a_png9"), _grid(9, 9, 64, 64, seed=1), "png")
    _write_grid(os.path.join(root, "Set", "b_bmp5"), _grid(5, 5, 80, 64, seed=2), "bmp")
    _write_grid(os.path.join(root, "Set", "c_wide"), _grid(5, 5, 96, 80, seed=3), "png")
    return ["a_png9", "b_bmp5", "c_wide"]


def _load(name, scale):
    net = lfsr_b200.load_net(name, A, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    return net.to(DEV), sd


def _entry(tmp_path, tag, script, flags):
    log = tmp_path / tag
    p = subprocess.run([sys.executable, script] + flags + ["--path_log", str(log) + "/"], cwd=ROOT, capture_output=True,
                       text=True, timeout=1200)
    assert p.returncode == 0, p.stderr[-4000:]
    return p.stdout, log


@pytest.mark.parametrize("name,scale", [("MyEfficientLFNet", 4), ("DistgSSR", 2)])
def test_test_py_on_view_images(tmp_path, name, scale):
    import train
    from types import SimpleNamespace
    from utils.utils_datasets import _batch1, read_views
    data = tmp_path / "data"
    scenes = _dataset(str(data))
    net, sd = _load(name, scale)
    ckpt = tmp_path / ("%s_x%d.pth" % (name, scale))
    torch.save({"state_dict": sd}, ckpt)
    out, log = _entry(tmp_path, "run", "test.py", ["--model_name", name, "--angRes", "5", "--scale_factor", str(scale),
                                                   "--path_pre_pth", str(ckpt), "--path_for_test", str(data) + "/"])
    # the same scenes through train.test from an in-memory loader of prepare_views outputs
    prepared = [lfutils.prepare_views(read_views(str(data / "Set" / s), A), A, scale, "hr") for s in scenes]
    loader = [_batch1(lr[None], hr[None], cb, A, A, s) for (lr, hr, cb), s in zip(prepared, scenes)]
    args = SimpleNamespace(scale_factor=scale, patch_size_for_test=32, stride_for_test=16, minibatch=64, self_ensemble=0,
                           angRes_out=A)
    with torch.no_grad():
        psnr, ssim, names = train.test(loader, DEV, net, args)
    assert names == scenes
    line = [ln for ln in out.splitlines() if ln.startswith("Test on Set")]
    assert line == ["Test on Set, psnr/ssim is %.3f/%.4f" % (np.mean(psnr), np.mean(ssim))], out
    rows = [r for r in _eval_values(list(log.rglob("evaluation.*"))) if r[0] == "Set" and r[1] in scenes]
    assert [r[1] for r in rows] == scenes
    np.testing.assert_allclose([r[2:] for r in rows], [[float("%.6f" % p), float("%.6f" % s)] for p, s in zip(psnr, ssim)],
                               rtol=1e-9)
    for s in scenes:
        assert len(list(log.rglob("TEST/Set/%s/View_*_*.bmp" % s))) == A * A
    # against the CPU oracle pipeline: oracle preparation -> oracle network -> oracle metrics
    P, S = 32, 16
    for k, s in enumerate(scenes):
        lr, hr, _ = view_oracle.prepare_views(read_views(str(data / "Set" / s), A), A, scale, "hr")
        np.testing.assert_array_max_ulp(prepared[k][0].cpu().numpy(), lr, maxulp=1)
        sub = lf_oracle.lfdivide(lr, A, P, S)
        nu, nv = sub.shape[:2]
        y = onets.forward(name, torch.from_numpy(sub.reshape(nu * nv, 1, A * P, A * P)), sd, A, scale).numpy()
        h, w = hr.shape[0] // A, hr.shape[1] // A
        want = lf_oracle.to_sai(lf_oracle.lfintegrate(y.reshape(nu, nv, A * P * scale, A * P * scale), A, P * scale,
                                                      S * scale, h, w))
        p_or, s_or, _, _ = lf_oracle.cal_metrics(hr, want, A)
        with torch.no_grad():
            _, _, sr = lfsr_b200.scene.test_scene(net, prepared[k][0], prepared[k][1], A, scale)
        assert float(np.abs(sr.cpu().numpy() - want).max()) <= 1e-3
        assert abs(psnr[k] - p_or) <= 0.01 and abs(ssim[k] - s_or) <= 1e-3


@pytest.mark.parametrize("ens", [0, 1])
def test_inference_py_on_lr_view_images(tmp_path, ens):
    from train import _write_views
    from utils.utils_datasets import read_views
    name, scale = "DistgSSR", 2
    data = tmp_path / "data"
    _write_grid(str(data / "Set" / "p"), _grid(7, 7, 32, 40, seed=5), "png")
    _write_grid(str(data / "Set" / "q"), _grid(5, 5, 36, 32, seed=6), "bmp")
    net, sd = _load(name, scale)
    ckpt = tmp_path / "ck.pth"
    torch.save({"state_dict": sd}, ckpt)
    out, log = _entry(tmp_path, "run", "inference.py", [
        "--model_name", name, "--angRes", "5", "--scale_factor", str(scale), "--path_pre_pth", str(ckpt),
        "--path_for_test", str(data) + "/", "--self_ensemble", str(ens)])
    test_dir = next(log.rglob("TEST"))
    for s in ("p", "q"):
        lr, _, cb = lfutils.prepare_views(read_views(str(data / "Set" / s), A), A, scale, "lr")
        with torch.no_grad():
            sr = lfsr_b200.scene.super_resolve_scene(net, lr, A, scale, self_ensemble=bool(ens))
        ref = tmp_path / "ref"
        ref.mkdir(exist_ok=True)
        _write_views(ref, s, sr, cb, A)
        files = sorted(os.listdir(test_dir / "Set" / s))
        assert files == sorted("View_%d_%d.bmp" % (i, j) for i in range(A) for j in range(A))
        for f in files:
            assert (test_dir / "Set" / s / f).read_bytes() == (ref / s / f).read_bytes(), (s, f)
        back = read_views(str(test_dir / "Set" / s), A)
        inp = lfutils.central_views(read_views(str(data / "Set" / s), A), A, scale)
        assert back.shape == (A, A, inp.shape[2] * scale, inp.shape[3] * scale, 3)


def test_test_py_views_two_gpus(tmp_path):
    _need_two()
    data = tmp_path / "data"
    _dataset(str(data))
    ckpt = tmp_path / "MyEfficientLFNet_x4.pth"
    torch.save({"state_dict": weights.make_state_dict("MyEfficientLFNet", 4, 1234)}, ckpt)
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--path_pre_pth", str(ckpt),
             "--path_for_test", str(data) + "/"]
    _compare(_run(tmp_path, "single", "test.py", flags, 1), _run(tmp_path, "multi", "test.py", flags, 2), 3, True)
