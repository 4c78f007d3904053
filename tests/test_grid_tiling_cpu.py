"""Angular window tiling (include/lfsr.h, "Angular window tiling") without a GPU: the window origins, the merge rule in
numpy against a direct per-view mean, the scene driver's plan on the torch statement of lfsr_window_accumulate against
the numpy composition over the oracle forward, and the full-grid loader and its errors."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from opref import RefOps
from oracle import lf_oracle, nets as onets, weights
from test_view_input_cpu import _grid, _oracle_prepare, _write_grid

import lfsr_b200
from lfsr_b200 import scene


# ---- the definition, in numpy -----------------------------------------------------------------------------------------
def window_pairs(n, ang, stride=None):
    o = scene.window_origins(n, ang, stride)
    return [(ou, ov) for ou in o for ov in o]


def merge_oracle(wins, n, ang, stride=None):
    """SR window mosaics [(A h), (A w)] in window order -> the N x N mosaic: per view (((W_k1 + W_k2) + ...) + W_kc) / c
    over the windows that contain it, in float32; c = 1 is a plain copy."""
    h, w = wins[0].shape[0] // ang, wins[0].shape[1] // ang
    out = np.empty((n, h, n, w), np.float32)
    pairs = window_pairs(n, ang, stride)
    for u in range(n):
        for v in range(n):
            parts = [np.asarray(wk, np.float32).reshape(ang, h, ang, w)[u - ou, :, v - ov, :]
                     for wk, (ou, ov) in zip(wins, pairs) if ou <= u < ou + ang and ov <= v < ov + ang]
            acc = parts[0].copy()
            for p in parts[1:]:
                acc = acc + p
            out[u, :, v, :] = acc if len(parts) == 1 else acc / np.float32(len(parts))
    return out.reshape(n * h, n * w)


class GridRefOps(RefOps):
    """RefOps plus the torch statement of lfsr_window_accumulate (fp32 `+`, and `/` by a tensor)"""

    def window_accumulate(self, win, grid, ang, n, h, w, o_u, o_v, modes):
        g, wv = grid.view(n, h, n, w), win.view(ang, h, ang, w)
        for a1 in range(ang):
            for a2 in range(ang):
                m, dst, v = modes[a1 * ang + a2], g[o_u + a1, :, o_v + a2, :], wv[a1, :, a2, :]
                if m == 0:
                    dst.copy_(v)
                elif m == 1:
                    dst.copy_(dst + v)
                else:
                    dst.copy_((dst + v) / torch.full_like(v, float(m)))


def oracle_scene(name, lr, sd, A, scale, patch, stride, h0, w0):
    sub = lf_oracle.lfdivide(lr, A, patch, stride)
    nu, nv = sub.shape[:2]
    L = A * patch
    y = onets.forward(name, torch.from_numpy(sub.reshape(nu * nv, 1, L, L)), sd, A, scale).numpy()
    y = y.reshape(nu, nv, L * scale, L * scale)
    return lf_oracle.to_sai(lf_oracle.lfintegrate(y, A, patch * scale, stride * scale, h0 * scale, w0 * scale))


def oracle_grid(name, lr, sd, n, A, scale, patch, stride, h0, w0, ang_stride=None):
    """each window through the oracle pipeline, then the merge oracle"""
    views = lr.reshape(n, h0, n, w0)
    wins = [oracle_scene(name, np.ascontiguousarray(views[ou:ou + A, :, ov:ov + A, :]).reshape(A * h0, A * w0), sd, A,
                         scale, patch, stride, h0, w0) for ou, ov in window_pairs(n, A, ang_stride)]
    return merge_oracle(wins, n, A, ang_stride)


# ---- window origins -------------------------------------------------------------------------------------------------------
def test_window_origins_properties():
    for ang in (2, 3, 5):
        for n in range(ang, 18):
            strides = [None] + (list(range(1, ang)) if n > ang else [None])
            for t in strides:
                o = scene.window_origins(n, ang, t)
                assert o[0] == 0 and o[-1] == n - ang
                assert all(b > a for a, b in zip(o, o[1:]))
                assert all(b - a <= (t or ang - 1) for a, b in zip(o, o[1:]))
                assert {x for a in o for x in range(a, a + ang)} == set(range(n))
                if n == ang:
                    assert o == [0]
                # the definition: 0, t, 2t, ... while < N - A, then N - A
                step = t or ang - 1
                assert o == ([k * step for k in range(n) if k * step < n - ang] + [n - ang] if n > ang else [0])


def test_window_origins_examples_and_errors():
    assert scene.window_origins(9, 5) == [0, 4] and len(window_pairs(9, 5)) == 4
    assert scene.window_origins(14, 5) == [0, 4, 8, 9] and len(window_pairs(14, 5)) == 16
    assert scene.window_origins(7, 5, 2) == [0, 2]
    assert scene.window_origins(5, 5, 3) == [0]
    for n, ang, t in ((4, 5, None), (9, 5, 5), (9, 5, -1), (6, 1, None)):
        with pytest.raises(ValueError):
            scene.window_origins(n, ang, t)


def test_window_plan_modes():
    """first window over a view stores, the last divides by the view's count, the ones between add"""
    for n, ang, t in ((9, 5, None), (14, 5, None), (9, 5, 2), (7, 3, 1), (5, 5, None)):
        plan = scene.window_plan(n, ang, t)
        assert [p[:2] for p in plan] == window_pairs(n, ang, t)
        seen = np.zeros((n, n), int)
        count = np.zeros((n, n), int)
        for ou, ov, _ in plan:
            count[ou:ou + ang, ov:ov + ang] += 1
        for ou, ov, modes in plan:
            for a1 in range(ang):
                for a2 in range(ang):
                    u, v, m = ou + a1, ov + a2, modes[a1 * ang + a2]
                    seen[u, v] += 1
                    c = count[u, v]
                    assert m == (0 if seen[u, v] == 1 else (c if seen[u, v] == c else 1))
        assert (seen == count).all() and count.min() >= 1


# ---- the merge ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,ang,t", [(9, 5, None), (9, 5, 2), (14, 5, None), (7, 3, 1), (5, 5, None)])
def test_merge_oracle_is_the_per_view_mean(n, ang, t):
    h, w = 3, 4
    rs = np.random.RandomState(n * 10 + ang)
    pairs = window_pairs(n, ang, t)
    wins = [rs.randint(0, 100, (ang * h, ang * w)).astype(np.float32) for _ in pairs]
    got = merge_oracle(wins, n, ang, t).reshape(n, h, n, w)
    total = np.zeros((n, h, n, w), np.int64)
    count = np.zeros((n, n), np.int64)
    for wk, (ou, ov) in zip(wins, pairs):
        total[ou:ou + ang, :, ov:ov + ang, :] += wk.astype(np.int64).reshape(ang, h, ang, w)
        count[ou:ou + ang, ov:ov + ang] += 1
    c = count[:, None, :, None]
    want = total.astype(np.float32) / c.astype(np.float32)         # integer sums are exact in fp32: one rounding
    assert np.array_equal(got, want)
    assert np.allclose(got, total / c, rtol=1e-6, atol=0)


@pytest.mark.parametrize("n,ang,t", [(9, 5, None), (9, 5, 2), (7, 3, 1)])
def test_torch_statement_with_plan_equals_merge_oracle(n, ang, t):
    """window_plan's modes through the torch statement of the kernel give the definition's bits on random floats"""
    h, w = 3, 5
    rs = np.random.RandomState(7)
    pairs = window_pairs(n, ang, t)
    wins = [rs.random_sample((ang * h, ang * w)).astype(np.float32) for _ in pairs]
    grid = torch.full((n * h, n * w), float("nan"))
    for (ou, ov, modes), wk in zip(scene.window_plan(n, ang, t), wins):
        GridRefOps().window_accumulate(torch.from_numpy(wk), grid, ang, n, h, w, ou, ov, modes)
    assert np.array_equal(grid.numpy(), merge_oracle(wins, n, ang, t))


# ---- the scene driver on the torch backend --------------------------------------------------------------------------------
def _net(name, A, scale, ops):
    sd = weights.make_state_dict(name, scale, 1234)
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(sd, strict=True)
    net.set_backend(ops)
    return net, sd


def test_super_resolve_grid_matches_oracle_composition():
    name, scale, A, n, t, P, S, h0, w0 = "MyEfficientLFNet", 4, 5, 7, 2, 8, 4, 12, 8
    ops = GridRefOps()
    net, sd = _net(name, A, scale, ops)
    lr = np.random.RandomState(11).random_sample((n * h0, n * w0)).astype(np.float32)
    assert len(scene.window_plan(n, A, t)) == 4
    with torch.no_grad():
        sr = scene.super_resolve_grid(net, torch.from_numpy(lr), n, A, scale, P, S, minibatch=16, ops=ops, ang_stride=t)
    want = oracle_grid(name, lr, sd, n, A, scale, P, S, h0, w0, t)
    assert sr.shape == want.shape and np.abs(sr.numpy() - want).max() <= 2e-5
    # test_grid: the metrics over all N^2 views against the oracle's
    hr = np.random.RandomState(12).random_sample(want.shape).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr2 = scene.test_grid(net, torch.from_numpy(lr), torch.from_numpy(hr), n, A, scale, P, S, minibatch=16,
                                          ops=ops, ang_stride=t)
    assert torch.equal(sr2, sr)
    p_or, s_or, _, _ = lf_oracle.cal_metrics(hr, want, n)
    assert abs(psnr - p_or) <= 1e-3 and abs(ssim - s_or) <= 1e-4


def test_single_window_grid_is_the_scene():
    name, scale, A, P, S, h0, w0 = "DistgSSR", 2, 5, 8, 4, 10, 10
    ops = GridRefOps()
    net, _ = _net(name, A, scale, ops)
    lr = torch.from_numpy(np.random.RandomState(3).random_sample((A * h0, A * w0)).astype(np.float32))
    hr = torch.from_numpy(np.random.RandomState(4).random_sample((A * h0 * scale, A * w0 * scale)).astype(np.float32))
    with torch.no_grad():
        p1, s1, sr1 = scene.test_scene(net, lr, hr, A, scale, P, S, minibatch=24, ops=ops)
        sr1 = sr1.clone()
        p2, s2, sr2 = scene.test_grid(net, lr, hr, A, A, scale, P, S, minibatch=24, ops=ops)
    assert torch.equal(sr1, sr2) and p1 == p2 and s1 == s2


# ---- loader -----------------------------------------------------------------------------------------------------------------
def _args(path, **kw):
    a = dict(angRes_in=5, angRes_out=5, scale_factor=4, path_for_test=str(path), data_name="ALL", synthetic=0,
             synthetic_size=8, patch_size_for_test=8, stride_for_test=4, minibatch=4, self_ensemble=0, full_grid=1,
             ang_stride=0)
    a.update(kw)
    return SimpleNamespace(**a)


@pytest.mark.parametrize("U,V,n,u0,v0", [(9, 9, 9, 0, 0), (9, 7, 7, 1, 0), (6, 8, 6, 0, 1), (5, 5, 5, 0, 0)])
def test_read_views_full_grid(tmp_path, U, V, n, u0, v0):
    from utils.utils_datasets import read_views
    g = _grid(U, V, 6, 5, seed=U * V)
    _write_grid(str(tmp_path / "s"), g, "png")
    got = read_views(str(tmp_path / "s"), 5, full_grid=True)
    assert got.shape == (n, n, 6, 5, 3)
    assert np.array_equal(got, g[u0:u0 + n, v0:v0 + n])
    assert read_views(str(tmp_path / "s"), 5).shape == (5, 5, 6, 5, 3)          # the default is unchanged


def test_full_grid_smaller_than_window_raises(tmp_path):
    from utils.utils_datasets import read_views
    _write_grid(str(tmp_path / "small"), _grid(9, 4, 8, 8), "png")
    with pytest.raises(ValueError, match="9x4 grid"):
        read_views(str(tmp_path / "small"), 5, full_grid=True)


def test_full_grid_loader_yields_grid_and_window_size(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare)
    _write_grid(str(tmp_path / "Set" / "a"), _grid(9, 7, 16, 12), "bmp")
    _write_grid(str(tmp_path / "Set" / "b"), _grid(5, 5, 16, 12), "png")
    names, loaders, n = D.MultiTestSetDataLoader(_args(tmp_path), views="hr")
    assert names == ["Set"] and n == 2
    lr, hr, cb, info, name = loaders[0][0]
    assert name == ["a"] and [int(x) for x in info] == [5, 5, 7]
    assert lr.shape == (1, 1, 7 * 4, 7 * 3) and hr.shape == (1, 1, 7 * 16, 7 * 12) and cb.shape == (1, 2, 7 * 16, 7 * 12)
    assert [int(x) for x in loaders[0][1][3]] == [5, 5, 5]
    lr, hr, cb, info, _ = D.MultiTestSetDataLoader(_args(tmp_path), views="lr")[1][0][0]
    assert lr.shape == (1, 1, 7 * 16, 7 * 12) and hr.numel() == 0 and cb.shape == (1, 2, 7 * 64, 7 * 48)
    # --full_grid 0 keeps the central A x A and the two-entry data_info
    lr, _, _, info, _ = D.MultiTestSetDataLoader(_args(tmp_path, full_grid=0), views="hr")[1][0][0]
    assert len(info) == 2 and lr.shape == (1, 1, 5 * 4, 5 * 3)


def test_full_grid_needs_view_images(tmp_path):
    from utils.utils_datasets import MultiTestSetDataLoader
    with pytest.raises(ValueError, match="--full_grid 1.*synthetic"):
        MultiTestSetDataLoader(_args(tmp_path, synthetic=2), views="hr")
    (tmp_path / "SR_5x5_4x" / "Set").mkdir(parents=True)
    with pytest.raises(ValueError, match="--full_grid 1.*h5"):
        MultiTestSetDataLoader(_args(tmp_path), views="hr")
    assert MultiTestSetDataLoader(_args(tmp_path, synthetic=2, full_grid=0), views="hr")[2] == 2


def test_train_test_routes_full_grid_scenes(tmp_path, monkeypatch):
    """train.test with --full_grid 1 on the torch backend: per scene, test_grid over the prepared N x N tensors"""
    import train
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare)
    _write_grid(str(tmp_path / "Set" / "a"), _grid(7, 7, 32, 32, seed=3), "png")
    _write_grid(str(tmp_path / "Set" / "b"), _grid(5, 5, 32, 32, seed=4), "png")
    ops = GridRefOps()
    net, _ = _net("LF_InterNet", 5, 4, ops)
    args = _args(tmp_path, data_name="Set", ang_stride=2)
    _, loaders, _ = D.MultiTestSetDataLoader(args, views="hr")
    with torch.no_grad():
        psnr, ssim, names = train.test(loaders[0], "cpu", net, args)
        assert names == ["a", "b"]
        for k, batch in enumerate(loaders[0]):
            lr, hr, _, info, _ = batch
            p, s, _ = scene.test_grid(net, lr, hr, int(info[2]), 5, 4, 8, 4, 4, ang_stride=2)
            assert (p, s) == (psnr[k], ssim[k])
