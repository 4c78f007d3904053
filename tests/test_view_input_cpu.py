"""Light fields stored as view images (utils_datasets.ViewsTestSet) without a GPU: the oracle's statement of the
preparation recipe (include/lfsr.h, "View preparation"), the reader and its errors, the loader choice of
MultiTestSetDataLoader, and the dataset split at world 2 over gloo with the device preparation replaced by the oracle."""
import os
import pickle
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from PIL import Image

from oracle import lf_oracle
import view_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dropin_utils(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["test"])          # utils.utils parses the command line at import (option.py)
    import utils.utils as U
    return U


def _args(path, A=5, scale=4, data_name="ALL", **kw):
    a = dict(angRes_in=A, angRes_out=A, scale_factor=scale, path_for_test=str(path), data_name=data_name, synthetic=0,
             synthetic_size=8, patch_size_for_test=8, stride_for_test=4, minibatch=4, self_ensemble=0)
    a.update(kw)
    return SimpleNamespace(**a)


def _grid(U, V, H, W, seed=0):
    """uint8 [U, V, H, W, 3] of smooth seeded content with (u, v) in the top-left pixel's R and G."""
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    g = np.empty((U, V, H, W, 3), np.uint8)
    for u in range(U):
        for v in range(V):
            for c in range(3):
                f = rs.uniform(1, 3, 2)
                g[u, v, :, :, c] = np.round(127.5 + 100 * np.sin(f[0] * yy * 3 + u * 0.1) * np.cos(f[1] * xx * 3 + v * 0.1))
            g[u, v, 0, 0, :2] = (u, v)
    return g


def _write_grid(scene_dir, grid, ext):
    from lfsr_b200 import lfutils
    os.makedirs(scene_dir, exist_ok=True)
    for u in range(grid.shape[0]):
        for v in range(grid.shape[1]):
            fn = os.path.join(scene_dir, "View_%d_%d.%s" % (u, v, ext))
            if ext == "bmp":
                lfutils.write_bmp(fn, grid[u, v])
            else:
                Image.fromarray(grid[u, v]).save(fn)


def _oracle_prepare(rgb8, ang, scale, kind):
    lr, hr, cbcr = view_oracle.prepare_views(rgb8, ang, scale, kind)
    return torch.from_numpy(lr), None if hr is None else torch.from_numpy(hr), torch.from_numpy(cbcr)


# ---- colour conversion ----------------------------------------------------------------------------------------------------
def test_rgb2ycbcr_term_by_term_matches_dropin_and_inverts(monkeypatch):
    U = _dropin_utils(monkeypatch)
    x = np.random.RandomState(1).random_sample((37, 29, 3))
    x[0, 0], x[0, 1] = 0.0, 1.0
    got = view_oracle.rgb2ycbcr(x)
    assert np.abs(got - U.rgb2ycbcr(x)).max() <= 1e-14
    assert np.abs(lf_oracle.ycbcr2rgb(got) - x).max() <= 1e-12
    # the numbers the device kernel must reproduce: uint8 / 255.0 in fp64, then the term-by-term sums
    k = np.arange(256, dtype=np.float64) / 255.0
    x8 = np.stack([k, k[::-1], np.roll(k, 7)], -1)[None]
    want_y = (((65.481 * x8[..., 0] + 128.553 * x8[..., 1]) + 24.966 * x8[..., 2]) + 16.0) / 255.0
    assert np.array_equal(view_oracle.rgb2ycbcr(x8)[..., 0], want_y)


# ---- oracle preparation -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale,H,W", [(2, 22, 30), (4, 34, 26)])
def test_prepare_views_shapes(scale, H, W):
    A = 5
    g = _grid(7, 7, H, W)
    Hc, Wc = H - H % scale, W - W % scale
    lr, hr, cb = view_oracle.prepare_views(g, A, scale, "hr")
    assert lr.shape == (A * Hc // scale, A * Wc // scale) and hr.shape == (A * Hc, A * Wc) and cb.shape == (2, A * Hc, A * Wc)
    assert lr.dtype == hr.dtype == cb.dtype == np.float32
    lr, hr, cb = view_oracle.prepare_views(g, A, scale, "lr")
    assert hr is None and lr.shape == (A * Hc, A * Wc) and cb.shape == (2, A * Hc * scale, A * Wc * scale)


def test_constant_views_give_equal_lr_and_hr_y():
    g = np.full((5, 5, 16, 24, 3), (200, 31, 77), np.uint8)
    lr, hr, cb, lr_rgb = view_oracle.prepare_views(g, 5, 4, "hr", with_lr_rgb=True)
    y_hr = view_oracle.rgb2ycbcr(g[0, 0].astype(np.float64) / 255.0)[..., 0]
    y_lr = view_oracle.rgb2ycbcr(lr_rgb)[..., 0]
    assert np.abs(y_lr - y_hr[0, 0]).max() <= 1e-12 and np.ptp(y_hr) == 0
    assert np.abs(lr - hr[0, 0]).max() <= 1e-6 and np.ptp(hr) == 0


def test_lr_kind_on_fp64_lr_views_reproduces_hr_kind():
    g = _grid(5, 5, 32, 48, seed=4)
    lr, hr, cb, lr_rgb = view_oracle.prepare_views(g, 5, 4, "hr", with_lr_rgb=True)
    assert lr_rgb.dtype == np.float64 and lr_rgb.shape == (5, 5, 8, 12, 3)
    lr2, hr2, cb2 = view_oracle.prepare_views(lr_rgb, 5, 4, "lr")
    assert hr2 is None and np.array_equal(lr2, lr) and np.array_equal(cb2, cb)


# ---- reader ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ext", ["bmp", "png"])
def test_views_read_back_exactly(tmp_path, ext):
    from utils.utils_datasets import read_views
    g = _grid(5, 5, 13, 17, seed=2)
    _write_grid(str(tmp_path / "s"), g, ext)
    assert np.array_equal(read_views(str(tmp_path / "s"), 5), g)


@pytest.mark.parametrize("n,first", [(7, 1), (9, 2)])
def test_central_views_are_read(tmp_path, n, first):
    from utils.utils_datasets import read_views
    g = _grid(n, n, 6, 6)
    _write_grid(str(tmp_path / "s"), g, "png")
    got = read_views(str(tmp_path / "s"), 5)
    assert got.shape == (5, 5, 6, 6, 3)
    for i in range(5):
        for j in range(5):
            assert tuple(got[i, j, 0, 0, :2]) == (first + i, first + j)


def test_loader_crops_to_multiples_of_scale(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare)
    _write_grid(str(tmp_path / "Set" / "scene"), _grid(5, 5, 35, 42), "bmp")
    names, loaders, n = D.MultiTestSetDataLoader(_args(tmp_path, scale=4), views="hr")
    assert names == ["Set"] and n == 1
    lr, hr, cb, info, name = loaders[0][0]
    assert name == ["scene"] and int(info[0][0]) == 5
    assert lr.shape == (1, 1, 5 * 8, 5 * 10) and hr.shape == (1, 1, 5 * 32, 5 * 40) and cb.shape == (1, 2, 5 * 32, 5 * 40)
    names, loaders, n = D.MultiTestSetDataLoader(_args(tmp_path, scale=4), views="lr")
    lr, hr, cb, _, _ = loaders[0][0]
    assert lr.shape == (1, 1, 5 * 32, 5 * 40) and hr.numel() == 0 and cb.shape == (1, 2, 5 * 128, 5 * 160)


def _bad(tmp_path, case):
    d = tmp_path / case
    g = _grid(5, 5, 8, 8)
    _write_grid(str(d), g, "png")
    target = d / "View_2_3.png"
    if case == "missing":
        target.unlink()
    elif case == "size":
        Image.fromarray(np.zeros((8, 9, 3), np.uint8)).save(target)
    elif case == "L":
        Image.fromarray(g[2, 3, :, :, 0]).save(target)
    elif case == "RGBA":
        Image.fromarray(np.concatenate([g[2, 3], g[2, 3, :, :, :1]], -1)).save(target)
    elif case == "P":
        Image.fromarray(g[2, 3]).convert("P").save(target)
    elif case == "16bit":
        import struct
        import zlib
        a = g[2, 3].astype(">u2") * 257
        chunk = lambda t, b: struct.pack(">I", len(b)) + t + b + struct.pack(">I", zlib.crc32(t + b) & 0xFFFFFFFF)
        raw = b"".join(b"\x00" + a[i].tobytes() for i in range(a.shape[0]))
        target.write_bytes(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 8, 8, 16, 2, 0, 0, 0))
                           + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b""))
    return str(d), "View_2_3"


@pytest.mark.parametrize("case,words", [("missing", "missing"), ("size", "9x8"), ("L", "mode L"), ("RGBA", "mode RGBA"),
                                        ("P", "mode P"), ("16bit", "16-bit")])
def test_bad_views_raise_naming_the_file(tmp_path, case, words):
    from utils.utils_datasets import read_views
    d, fn = _bad(tmp_path, case)
    with pytest.raises(ValueError) as e:
        read_views(d, 5)
    assert fn in str(e.value) and words in str(e.value), str(e.value)


def test_grid_smaller_than_angres_raises(tmp_path):
    from utils.utils_datasets import read_views
    _write_grid(str(tmp_path / "small"), _grid(5, 4, 8, 8), "png")
    with pytest.raises(ValueError, match="small.*5x4 grid"):
        read_views(str(tmp_path / "small"), 5)


# ---- loader choice --------------------------------------------------------------------------------------------------------
def test_h5_layout_still_takes_precedence(tmp_path):
    from utils.utils_datasets import MultiTestSetDataLoader
    _write_grid(str(tmp_path / "Set" / "scene"), _grid(5, 5, 8, 8), "png")
    (tmp_path / "SR_5x5_4x" / "Set").mkdir(parents=True)
    try:
        import h5py  # noqa: F401
    except ImportError:
        with pytest.raises(RuntimeError, match="h5py"):
            MultiTestSetDataLoader(_args(tmp_path), views="hr")
    else:
        names, loaders, n = MultiTestSetDataLoader(_args(tmp_path), views="hr")
        assert names == ["Set"] and n == 0 and type(loaders[0]).__name__ == "H5TestSet"


def test_synthetic_still_wins_and_no_data_names_both_layouts(tmp_path):
    from utils.utils_datasets import MultiTestSetDataLoader, SyntheticTestSet
    _write_grid(str(tmp_path / "Set" / "scene"), _grid(5, 5, 8, 8), "png")
    names, loaders, n = MultiTestSetDataLoader(_args(tmp_path, synthetic=2), views="hr")
    assert names == ["Synthetic"] and n == 2 and isinstance(loaders[0], SyntheticTestSet)
    with pytest.raises(FileNotFoundError) as e:
        MultiTestSetDataLoader(_args(tmp_path / "empty"), views="lr")
    assert "SR_5x5_4x" in str(e.value) and "View_u_v" in str(e.value)


def test_single_dataset_and_all(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare)
    for ds, scenes in (("B", ["z", "a"]), ("A", ["m"])):
        for s in scenes:
            _write_grid(str(tmp_path / ds / s), _grid(5, 5, 8, 8), "png")
    (tmp_path / "notes").mkdir()
    names, loaders, n = D.MultiTestSetDataLoader(_args(tmp_path), views="hr")
    assert names == ["A", "B"] and n == 3
    assert [b[4][0] for b in loaders[1]] == ["a", "z"]
    names, loaders, n = D.MultiTestSetDataLoader(_args(tmp_path, data_name="B"), views="hr")
    assert names == ["B"] and n == 2 and len(loaders[0]) == 2


# ---- world 2 over gloo ----------------------------------------------------------------------------------------------------
def _net(scale):
    import lfsr_b200
    from opref import RefOps
    from oracle import weights
    net = lfsr_b200.load_net("LF_InterNet", 5, scale).eval()
    net.load_state_dict(weights.make_state_dict("LF_InterNet", scale, 1234))
    net.set_backend(RefOps())
    return net


def _run_split(data_root):
    """train.test over the views dataset with the oracle preparation; returns (results, scene folders read)."""
    import train
    import utils.utils_datasets as D
    reads = []
    read, prepare = D.read_views, D.prepare_views

    def counting(scene_dir, ang):
        reads.append(os.path.basename(scene_dir))
        return read(scene_dir, ang)

    D.read_views, D.prepare_views = counting, _oracle_prepare
    try:
        names, loaders, _ = D.MultiTestSetDataLoader(_args(data_root, data_name="Set"), views="hr")
        return train.test(loaders[0], "cpu", _net(4), _args(data_root)), reads
    finally:
        D.read_views, D.prepare_views = read, prepare


def _worker(rank, world, port, out_dir, data_root):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    res, reads = _run_split(data_root)
    with open(os.path.join(out_dir, f"rank{rank}.pkl"), "wb") as f:
        pickle.dump((res, reads), f)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(900)
def test_two_rank_split_decodes_only_own_scenes(tmp_path):
    data = tmp_path / "data"
    for i in range(3):
        _write_grid(str(data / "Set" / ("scene_%d" % i)), _grid(5, 5, 32, 32, seed=10 + i), "bmp")
    out = tmp_path / "out"
    out.mkdir()
    port = 29500 + ((os.getpid() + 900) % 2000)
    mp.spawn(_worker, args=(2, port, str(out), str(data)), nprocs=2, join=True)
    got = [pickle.load(open(out / f"rank{r}.pkl", "rb")) for r in range(2)]
    threads = torch.get_num_threads()
    torch.set_num_threads(2)
    try:
        want, reads = _run_split(str(data))
    finally:
        torch.set_num_threads(threads)
    assert reads == ["scene_0", "scene_1", "scene_2"]
    for r in range(2):
        (psnr, ssim, names), reads = got[r]
        assert names == want[2]
        assert reads == ["scene_%d" % r, "scene_2"]           # scene 0 / 1: one full round; scene 2: the tail
        assert psnr[:2] == want[0][:2] and ssim[:2] == want[1][:2]
        assert np.abs(np.subtract(psnr[2:], want[0][2:])).max() <= 1e-4
