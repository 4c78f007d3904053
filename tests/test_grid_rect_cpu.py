"""Angular window tiling on rectangular N_u x N_v grids and chosen central sub-grids (--grid_views) without a GPU: the
plan against the definition, the merge rule in numpy, the scene driver on the torch statements of
lfsr_window_accumulate_uv / lfsr_metric_sums_uv against the oracle composition, and the loader, its errors and the
routing of train.test."""
import itertools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import lf_oracle
import view_oracle
from test_grid_tiling_cpu import GridRefOps, _net, oracle_scene
from test_view_input_cpu import _grid, _write_grid

from lfsr_b200 import scene


# ---- the definition, in numpy -----------------------------------------------------------------------------------------
def rect_pairs(nu, nv, ang, stride=None):
    return [(ou, ov) for ou in scene.window_origins(nu, ang, stride) for ov in scene.window_origins(nv, ang, stride)]


def rect_merge_oracle(wins, nu, nv, ang, stride=None):
    """SR window mosaics [(A h), (A w)] in window order -> the N_u x N_v mosaic: per view (((W_k1 + W_k2) + ...) + W_kc)
    / c over the windows that contain it, in float32; c = 1 is a plain copy."""
    h, w = wins[0].shape[0] // ang, wins[0].shape[1] // ang
    out = np.empty((nu, h, nv, w), np.float32)
    pairs = rect_pairs(nu, nv, ang, stride)
    for u in range(nu):
        for v in range(nv):
            parts = [np.asarray(wk, np.float32).reshape(ang, h, ang, w)[u - ou, :, v - ov, :]
                     for wk, (ou, ov) in zip(wins, pairs) if ou <= u < ou + ang and ov <= v < ov + ang]
            acc = parts[0].copy()
            for p in parts[1:]:
                acc = acc + p
            out[u, :, v, :] = acc if len(parts) == 1 else acc / np.float32(len(parts))
    return out.reshape(nu * h, nv * w)


class RectRefOps(GridRefOps):
    """GridRefOps plus the torch statements of lfsr_window_accumulate_uv and lfsr_metric_sums_uv"""

    def window_accumulate_uv(self, win, grid, ang, n_u, n_v, h, w, o_u, o_v, modes):
        g, wv = grid.view(n_u, h, n_v, w), win.view(ang, h, ang, w)
        for a1 in range(ang):
            for a2 in range(ang):
                m, dst, v = modes[a1 * ang + a2], g[o_u + a1, :, o_v + a2, :], wv[a1, :, a2, :]
                if m == 0:
                    dst.copy_(v)
                elif m == 1:
                    dst.copy_(dst + v)
                else:
                    dst.copy_((dst + v) / torch.full_like(v, float(m)))

    def metric_sums_uv(self, label, out, ang_u, ang_v, h, w, acc):
        acc.copy_(acc + torch.from_numpy(metric_sums_oracle(label.numpy(), out.numpy(), ang_u, ang_v)).to(acc.device))


def metric_sums_oracle(label, out, nu, nv):
    """per view (row-major) {sum of squared errors, SSIM map sum over the interior}, flattened like lfsr_metric_sums_uv"""
    H, W = label.shape
    h, w = H // nu, W // nv
    la, ou = label.reshape(nu, h, nv, w), out.reshape(nu, h, nv, w)
    res = np.zeros((nu, nv, 2))
    for u in range(nu):
        for v in range(nv):
            a, b = la[u, :, v, :], ou[u, :, v, :]
            res[u, v, 0] = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).sum()
            res[u, v, 1] = lf_oracle.ssim_view(a, b) * (h - 10) * (w - 10)
    return res.reshape(-1)


def oracle_rect_grid(name, lr, sd, nu, nv, A, scale, patch, stride, h0, w0, ang_stride=None):
    """each window through the oracle pipeline, then the merge oracle"""
    views = lr.reshape(nu, h0, nv, w0)
    wins = [oracle_scene(name, np.ascontiguousarray(views[ou:ou + A, :, ov:ov + A, :]).reshape(A * h0, A * w0), sd, A,
                         scale, patch, stride, h0, w0) for ou, ov in rect_pairs(nu, nv, A, ang_stride)]
    return rect_merge_oracle(wins, nu, nv, A, ang_stride)


# ---- the plan ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ang", [2, 3, 5])
def test_window_plan_rectangular(ang):
    """every (N_u, N_v) with N <= 14: the plan is the row-major product of the per-axis origins, covers every view, stores
    on a view's first window, divides by c = c_u * c_v on its last; N_u = N_v is exactly the square plan"""
    for nu, nv in itertools.product(range(ang, 15), repeat=2):
        for t in [None] + list(range(1, ang)):
            plan = scene.window_plan((nu, nv), ang, t)
            assert [p[:2] for p in plan] == rect_pairs(nu, nv, ang, t)
            count = np.zeros((nu, nv), int)
            for ou, ov, _ in plan:
                count[ou:ou + ang, ov:ov + ang] += 1
            cu = np.bincount([o + a for o in scene.window_origins(nu, ang, t) for a in range(ang)], minlength=nu)
            cv = np.bincount([o + a for o in scene.window_origins(nv, ang, t) for a in range(ang)], minlength=nv)
            assert count.min() >= 1 and np.array_equal(count, np.outer(cu, cv))
            seen = np.zeros((nu, nv), int)
            last_mode = np.zeros((nu, nv), int)
            for ou, ov, modes in plan:
                for a1 in range(ang):
                    for a2 in range(ang):
                        u, v, m = ou + a1, ov + a2, modes[a1 * ang + a2]
                        seen[u, v] += 1
                        c = count[u, v]
                        assert m == (0 if seen[u, v] == 1 else (c if seen[u, v] == c else 1))
                        last_mode[u, v] = m
            assert np.array_equal(seen, count)
            # the last window's mode equals the view's count (a view of one window is stored, mode 0)
            assert np.array_equal(np.where(count == 1, 0, count), last_mode)
            if nu == nv:
                assert plan == scene.window_plan(nu, ang, t)


def test_window_plan_examples():
    assert len(scene.window_plan((9, 13), 5)) == 2 * 3
    assert len(scene.window_plan((9, 13), 5, 2)) == 3 * 5
    assert [p[:2] for p in scene.window_plan((5, 9), 5)] == [(0, 0), (0, 4)]
    with pytest.raises(ValueError):
        scene.window_plan((4, 9), 5)


# ---- the merge ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nu,nv,ang,t", [(9, 13, 5, None), (9, 13, 5, 2), (5, 9, 5, None), (9, 6, 3, 1), (7, 11, 5, 3)])
def test_rect_merge_oracle_is_the_per_view_mean(nu, nv, ang, t):
    h, w = 3, 4
    rs = np.random.RandomState(nu * 100 + nv)
    pairs = rect_pairs(nu, nv, ang, t)
    wins = [rs.randint(0, 100, (ang * h, ang * w)).astype(np.float32) for _ in pairs]
    got = rect_merge_oracle(wins, nu, nv, ang, t).reshape(nu, h, nv, w)
    total = np.zeros((nu, h, nv, w), np.int64)
    count = np.zeros((nu, nv), np.int64)
    for wk, (ou, ov) in zip(wins, pairs):
        total[ou:ou + ang, :, ov:ov + ang, :] += wk.astype(np.int64).reshape(ang, h, ang, w)
        count[ou:ou + ang, ov:ov + ang] += 1
    c = count[:, None, :, None]
    assert np.array_equal(got, total.astype(np.float32) / c.astype(np.float32))   # exact integer sums: one rounding


@pytest.mark.parametrize("nu,nv,ang,t", [(9, 13, 5, None), (9, 13, 5, 2), (6, 9, 3, 1)])
def test_torch_statement_with_rect_plan_equals_merge_oracle(nu, nv, ang, t):
    h, w = 3, 5
    rs = np.random.RandomState(9)
    wins = [rs.random_sample((ang * h, ang * w)).astype(np.float32) for _ in rect_pairs(nu, nv, ang, t)]
    grid = torch.full((nu * h, nv * w), float("nan"))
    for (ou, ov, modes), wk in zip(scene.window_plan((nu, nv), ang, t), wins):
        RectRefOps().window_accumulate_uv(torch.from_numpy(wk), grid, ang, nu, nv, h, w, ou, ov, modes)
    assert np.array_equal(grid.numpy(), rect_merge_oracle(wins, nu, nv, ang, t))


# ---- the scene driver on the torch backend --------------------------------------------------------------------------------
@pytest.mark.parametrize("nu,nv,t", [(5, 9, None), (9, 6, None), (7, 11, 2)])
def test_super_resolve_rect_grid_matches_oracle_composition(nu, nv, t):
    name, scale, A, P, S, h0, w0 = "MyEfficientLFNet", 4, 5, 8, 4, 8, 12
    ops = RectRefOps()
    net, sd = _net(name, A, scale, ops)
    lr = np.random.RandomState(nu * nv).random_sample((nu * h0, nv * w0)).astype(np.float32)
    with torch.no_grad():
        sr = scene.super_resolve_grid(net, torch.from_numpy(lr), (nu, nv), A, scale, P, S, minibatch=16, ops=ops,
                                      ang_stride=t)
    want = oracle_rect_grid(name, lr, sd, nu, nv, A, scale, P, S, h0, w0, t)
    assert sr.shape == want.shape == (nu * h0 * scale, nv * w0 * scale)
    assert np.abs(sr.numpy() - want).max() <= 2e-5


def test_rect_test_grid_metrics_match_oracle():
    """test_grid on a 7 x 11 grid: metrics_from_sums over the N_u * N_v views equals the oracle's per-view mean"""
    name, scale, A, P, S, h0, w0, nu, nv = "DistgSSR", 2, 5, 8, 4, 10, 8, 7, 11
    ops = RectRefOps()
    net, sd = _net(name, A, scale, ops)
    lr = np.random.RandomState(21).random_sample((nu * h0, nv * w0)).astype(np.float32)
    hr = np.random.RandomState(22).random_sample((nu * h0 * scale, nv * w0 * scale)).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr = scene.test_grid(net, torch.from_numpy(lr), torch.from_numpy(hr), (nu, nv), A, scale, P, S,
                                         minibatch=16, ops=ops)
    out = sr.numpy()
    la, ou = hr.reshape(nu, h0 * scale, nv, w0 * scale), out.reshape(nu, h0 * scale, nv, w0 * scale)
    pv = np.array([[lf_oracle.psnr_view(la[u, :, v, :], ou[u, :, v, :]) for v in range(nv)] for u in range(nu)], np.float32)
    sv = np.array([[lf_oracle.ssim_view(la[u, :, v, :], ou[u, :, v, :]) for v in range(nv)] for u in range(nu)], np.float32)
    # cal_metrics' rule (utils/utils.py:127-132): the sum over all views divided by the number of views with value > 0
    assert abs(psnr - pv.sum() / (pv > 0).sum()) <= 1e-3 and abs(ssim - sv.sum() / (sv > 0).sum()) <= 1e-4
    # metrics_from_sums on the oracle's sums of the same mosaics
    p2, s2 = scene.metrics_from_sums(metric_sums_oracle(hr, out, nu, nv), (nu, nv), h0 * scale, w0 * scale)
    assert (p2, s2) == (psnr, ssim)


def test_square_pair_is_the_int():
    name, scale, A, P, S, h0, w0, n = "DistgSSR", 2, 5, 8, 4, 10, 10, 7
    ops = RectRefOps()
    net, _ = _net(name, A, scale, ops)
    lr = torch.from_numpy(np.random.RandomState(3).random_sample((n * h0, n * w0)).astype(np.float32))
    hr = torch.from_numpy(np.random.RandomState(4).random_sample((n * h0 * scale, n * w0 * scale)).astype(np.float32))
    with torch.no_grad():
        p1, s1, sr1 = scene.test_grid(net, lr, hr, n, A, scale, P, S, minibatch=24, ops=ops, ang_stride=2)
        p2, s2, sr2 = scene.test_grid(net, lr, hr, (n, n), A, scale, P, S, minibatch=24, ops=ops, ang_stride=2)
    assert torch.equal(sr1, sr2) and (p1, s1) == (p2, s2)


def test_rect_grid_rejects_mismatched_mosaic():
    ops = RectRefOps()
    net, _ = _net("DistgSSR", 5, 2, ops)
    with pytest.raises(ValueError, match="9x13 grid"):
        scene.super_resolve_grid(net, torch.zeros(9 * 8 + 1, 13 * 8), (9, 13), 5, 2, 8, 4, ops=ops)


# ---- loader -----------------------------------------------------------------------------------------------------------------
def _args(path, **kw):
    a = dict(angRes_in=5, angRes_out=5, scale_factor=4, path_for_test=str(path), data_name="ALL", synthetic=0,
             synthetic_size=8, patch_size_for_test=8, stride_for_test=4, minibatch=4, self_ensemble=0, full_grid=1,
             ang_stride=0, grid_views="")
    a.update(kw)
    return SimpleNamespace(**a)


def _oracle_prepare_uv(rgb8, ang, scale, kind):
    """view_oracle.prepare_views for an int or a (U, V) angular size"""
    au, av = (ang, ang) if isinstance(ang, int) else ang
    U, V, H, W, _ = rgb8.shape
    u0, v0 = (U - au) // 2, (V - av) // 2
    x = rgb8[u0:u0 + au, v0:v0 + av, :H - H % scale, :W - W % scale].astype(np.float64) / 255.0
    per_view = lambda f, v: np.stack([np.stack([f(v[i, j]) for j in range(av)]) for i in range(au)])
    sai = view_oracle._views_to_sai
    if kind == "hr":
        hr_y = sai(view_oracle.rgb2ycbcr(x)[..., 0]).astype("single")
        lr_rgb = per_view(lambda im: lf_oracle.imresize(im, scalar_scale=1 / scale), x)
    else:
        hr_y, lr_rgb = None, x
    lr_y = sai(view_oracle.rgb2ycbcr(lr_rgb)[..., 0]).astype("single")
    sr_rgb = per_view(lambda im: lf_oracle.imresize(im, scalar_scale=scale), lr_rgb)
    cbcr = np.ascontiguousarray(sai(view_oracle.rgb2ycbcr(sr_rgb)[..., 1:3]).transpose(2, 0, 1)).astype("single")
    return torch.from_numpy(lr_y), None if hr_y is None else torch.from_numpy(hr_y), torch.from_numpy(cbcr)


def test_oracle_prepare_uv_is_the_square_oracle():
    g = _grid(7, 7, 16, 12, seed=1)
    for a, b in zip(_oracle_prepare_uv(g, 5, 4, "hr"), view_oracle.prepare_views(g, 5, 4, "hr")):
        assert np.array_equal(a.numpy(), b)


@pytest.mark.parametrize("U,V", [(9, 13), (15, 15)])
@pytest.mark.parametrize("grid,nu,nv", [("all", None, None), ((7, 9), 7, 9), ((9, 9), 9, 9)])
def test_read_views_grid(tmp_path, U, V, grid, nu, nv):
    from utils.utils_datasets import read_views
    g = _grid(U, V, 6, 5, seed=U * V)
    _write_grid(str(tmp_path / "s"), g, "png")
    nu, nv = (U, V) if grid == "all" else (nu, nv)
    got = read_views(str(tmp_path / "s"), 5, full_grid=True, grid=grid)
    u0, v0 = (U - nu) // 2, (V - nv) // 2
    assert got.shape == (nu, nv, 6, 5, 3)
    assert np.array_equal(got, g[u0:u0 + nu, v0:v0 + nv])
    # the (u, v) written into each view's top-left pixel: the central views, in order
    assert [tuple(got[i, j, 0, 0, :2]) for i in range(nu) for j in range(nv)] == \
        [(u0 + i, v0 + j) for i in range(nu) for j in range(nv)]
    m = min(U, V)
    assert read_views(str(tmp_path / "s"), 5, full_grid=True).shape[:2] == (m, m)      # the default is unchanged


def test_parse_grid_views():
    from utils.utils_datasets import parse_grid_views
    assert parse_grid_views("", True) is None and parse_grid_views("", False) is None
    assert parse_grid_views("all", True) == "all"
    assert parse_grid_views("9x13", True) == (9, 13)
    for bad in ("9", "9x", "x9", "9x13x2", "9X13", "a", "0x9", "9x-1", "9 x 13", "All"):
        with pytest.raises(ValueError, match="--grid_views"):
            parse_grid_views(bad, True)
    for value in ("all", "7x9"):
        with pytest.raises(ValueError, match="--grid_views.*--full_grid 1"):
            parse_grid_views(value, False)


def test_grid_views_errors(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare_uv)
    _write_grid(str(tmp_path / "Set" / "a"), _grid(9, 13, 16, 12), "png")
    scene_dir = str(tmp_path / "Set" / "a")
    # malformed value, and --grid_views without --full_grid 1
    with pytest.raises(ValueError, match="--grid_views"):
        D.MultiTestSetDataLoader(_args(tmp_path, grid_views="9by13"), views="hr")
    with pytest.raises(ValueError, match="--grid_views.*--full_grid 1"):
        D.MultiTestSetDataLoader(_args(tmp_path, grid_views="all", full_grid=0), views="hr")
    with pytest.raises(ValueError, match="--full_grid 1"):
        D.read_views(scene_dir, 5, grid="all")
    # smaller than A, larger than the scene's grid: the error names the flag and the scene folder
    for grid in ((4, 9), (9, 3), (11, 9), (9, 15)):
        with pytest.raises(ValueError, match="--grid_views") as e:
            D.read_views(scene_dir, 5, full_grid=True, grid=grid)
        assert scene_dir in str(e.value)
    for value in ("4x9", "9x15"):
        _, loaders, _ = D.MultiTestSetDataLoader(_args(tmp_path, grid_views=value), views="hr")
        with pytest.raises(ValueError, match="--grid_views") as e:
            loaders[0][0]
        assert scene_dir in str(e.value)


def test_grid_views_loader_data_info(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare_uv)
    _write_grid(str(tmp_path / "Set" / "a"), _grid(9, 13, 16, 12), "bmp")
    _write_grid(str(tmp_path / "Set" / "b"), _grid(9, 9, 16, 12), "png")
    lr, hr, cb, info, name = D.MultiTestSetDataLoader(_args(tmp_path, grid_views="all"), views="hr")[1][0][0]
    assert name == ["a"] and [int(x) for x in info] == [5, 5, 9, 13]
    assert lr.shape == (1, 1, 9 * 4, 13 * 3) and hr.shape == (1, 1, 9 * 16, 13 * 12) and cb.shape == (1, 2, 9 * 16, 13 * 12)
    want = _oracle_prepare_uv(_grid(9, 13, 16, 12), (9, 13), 4, "hr")
    assert torch.equal(lr[0, 0], want[0]) and torch.equal(hr[0, 0], want[1]) and torch.equal(cb[0], want[2])
    lr, _, _, info, _ = D.MultiTestSetDataLoader(_args(tmp_path, grid_views="5x7"), views="lr")[1][0][1]
    assert [int(x) for x in info] == [5, 5, 5, 7] and lr.shape == (1, 1, 5 * 16, 7 * 12)
    # the default keeps [A, A, N] with N = min(U, V)
    lr, _, _, info, _ = D.MultiTestSetDataLoader(_args(tmp_path), views="hr")[1][0][0]
    assert [int(x) for x in info] == [5, 5, 9] and lr.shape == (1, 1, 9 * 4, 9 * 3)


def test_grid_size():
    import train
    assert train.grid_size([torch.tensor([5]), torch.tensor([5]), torch.tensor([9])]) == (9, 9)
    assert train.grid_size([torch.tensor([5]), torch.tensor([5]), torch.tensor([9]), torch.tensor([13])]) == (9, 13)
    assert train.grid_size([5, 5, 7, 11]) == (7, 11)
    with pytest.raises(ValueError):
        train.grid_size([torch.tensor([5]), torch.tensor([5])])


def test_train_test_routes_rect_scenes(tmp_path, monkeypatch):
    """train.test with --grid_views on the torch backend: per scene, test_grid over the prepared N_u x N_v tensors"""
    import train
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare_uv)
    _write_grid(str(tmp_path / "Set" / "a"), _grid(5, 7, 32, 32, seed=3), "png")
    _write_grid(str(tmp_path / "Set" / "b"), _grid(7, 5, 32, 32, seed=4), "png")
    ops = RectRefOps()
    net, _ = _net("LF_InterNet", 5, 4, ops)
    args = _args(tmp_path, data_name="Set", ang_stride=2, grid_views="all")
    _, loaders, _ = D.MultiTestSetDataLoader(args, views="hr")
    calls = []
    real = scene.test_grid
    monkeypatch.setattr(scene, "test_grid", lambda *a, **k: calls.append(a[3]) or real(*a, **k))
    with torch.no_grad():
        psnr, ssim, names = train.test(loaders[0], "cpu", net, args)
    assert names == ["a", "b"] and calls == [(5, 7), (7, 5)]
    monkeypatch.setattr(scene, "test_grid", real)
    with torch.no_grad():
        for k, batch in enumerate(loaders[0]):
            lr, hr, _, info, _ = batch
            p, s, _ = scene.test_grid(net, lr, hr, (int(info[2]), int(info[3])), 5, 4, 8, 4, 4, ang_stride=2)
            assert (p, s) == (psnr[k], ssim[k])
