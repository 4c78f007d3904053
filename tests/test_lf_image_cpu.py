"""Light fields stored as one image (include/lfsr.h, "Image light fields": SAI mosaic or lenslet) without a GPU: a numpy
statement of both layouts, the reader and its errors, the --input_layout / --input_grid options, and ImageTestSet against
ViewsTestSet on the same light fields with the device preparation replaced by the numpy oracle, also split over two
ranks (gloo)."""
import os
import pickle
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from PIL import Image

from oracle import nets as onets
from test_grid_rect_cpu import _oracle_prepare_uv
from test_view_input_cpu import _args, _grid, _net, _write_grid

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the layouts, in numpy ----------------------------------------------------------------------------------------------------
def views_to_image(g, layout):
    """uint8 views [U, V, H, W, 3] -> the mosaic [(U H), (V W), 3] or lenslet [(H U), (W V), 3] image"""
    U, V, H, W, _ = g.shape
    if layout == "mosaic":
        return np.ascontiguousarray(g.transpose(0, 2, 1, 3, 4)).reshape(U * H, V * W, 3)
    return np.ascontiguousarray(g.transpose(2, 0, 3, 1, 4)).reshape(H * U, W * V, 3)


def image_to_views(img, layout, U, V):
    """the inverse of views_to_image"""
    rows, cols = img.shape[:2]
    H, W = rows // U, cols // V
    if layout == "mosaic":
        return np.ascontiguousarray(img.reshape(U, H, V, W, 3).transpose(0, 2, 1, 3, 4))
    return np.ascontiguousarray(img.reshape(H, U, W, V, 3).transpose(1, 3, 0, 2, 4))


def _oracle_prepare_image(img8, layout, grid, ang, scale, kind):
    return _oracle_prepare_uv(image_to_views(np.asarray(img8), layout, *grid), ang, scale, kind)


def write_image(path, g, layout):
    from lfsr_b200 import lfutils
    os.makedirs(os.path.dirname(path), exist_ok=True)
    img = views_to_image(g, layout)
    if path.lower().endswith(".bmp"):
        lfutils.write_bmp(path, img)
    else:
        Image.fromarray(img).save(path)


@pytest.mark.parametrize("U,V", [(1, 5), (5, 9), (9, 14), (14, 1), (14, 5), (9, 9)])
@pytest.mark.parametrize("layout", ["mosaic", "lenslet"])
def test_layout_definition_and_round_trip(U, V, layout):
    H, W = 7, 5
    g = np.random.RandomState(U * 31 + V).randint(0, 256, (U, V, H, W, 3)).astype(np.uint8)
    img = views_to_image(g, layout)
    assert img.shape == (U * H, V * W, 3)
    for u, v, h, w in [(0, 0, 0, 0), (U - 1, V - 1, H - 1, W - 1), (U // 2, V - 1, 3, 1), (U - 1, 0, H - 1, 2)]:
        px = img[u * H + h, v * W + w] if layout == "mosaic" else img[h * U + u, w * V + v]
        assert np.array_equal(px, g[u, v, h, w])
    assert np.array_equal(image_to_views(img, layout, U, V), g)


@pytest.mark.parametrize("A", [1, 5, 9, 14])
def test_lenslet_is_sai2macpi(A):
    H, W = 5, 7
    g = np.random.RandomState(A).randint(0, 256, (A, A, H, W, 3)).astype(np.uint8)
    sai = torch.from_numpy(views_to_image(g, "mosaic").transpose(2, 0, 1)[None].copy())
    want = onets.sai2macpi(sai, A)[0].permute(1, 2, 0).numpy()
    assert np.array_equal(views_to_image(g, "lenslet"), want)


# ---- reader ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ext", ["png", "bmp"])
@pytest.mark.parametrize("layout", ["mosaic", "lenslet"])
def test_read_lf_image_round_trips(tmp_path, ext, layout):
    from utils.utils_datasets import read_lf_image
    g = _grid(9, 5, 13, 11, seed=3)
    fn = str(tmp_path / ("s." + ext))
    write_image(fn, g, layout)
    img = read_lf_image(fn, layout, (9, 5))
    assert img.dtype == np.uint8 and img.shape == (9 * 13, 5 * 11, 3)
    assert np.array_equal(image_to_views(img, layout, 9, 5), g)


def _png16(path, h, w):
    import struct
    import zlib
    a = np.random.RandomState(0).randint(0, 65536, (h, w, 3)).astype(">u2")
    chunk = lambda t, b: struct.pack(">I", len(b)) + t + b + struct.pack(">I", zlib.crc32(t + b) & 0xFFFFFFFF)
    raw = b"".join(b"\x00" + a[i].tobytes() for i in range(h))
    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 16, 2, 0, 0, 0))
                + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b""))


@pytest.mark.parametrize("case,words", [("size", "multiple of 5"), ("16bit", "16-bit"), ("L", "mode L"),
                                        ("RGBA", "mode RGBA")])
def test_read_lf_image_errors_name_the_file(tmp_path, case, words):
    from utils.utils_datasets import read_lf_image
    fn = str(tmp_path / "bad_scene.png")
    img = views_to_image(_grid(5, 5, 8, 8), "lenslet")
    if case == "size":
        Image.fromarray(img[:, :-1]).save(fn)
    elif case == "16bit":
        _png16(fn, 40, 40)
    elif case == "L":
        Image.fromarray(img[..., 0]).save(fn)
    else:
        Image.fromarray(np.concatenate([img, img[..., :1]], -1)).save(fn)
    with pytest.raises(ValueError) as e:
        read_lf_image(fn, "lenslet", (5, 5))
    assert "bad_scene.png" in str(e.value) and words in str(e.value), str(e.value)


def test_pillow_limit_is_lifted_for_the_call_only(tmp_path, monkeypatch):
    from utils.utils_datasets import read_lf_image
    g = _grid(5, 5, 8, 12)
    fn = str(tmp_path / "big.png")
    write_image(fn, g, "mosaic")
    monkeypatch.setattr(Image, "MAX_IMAGE_PIXELS", 100)
    with pytest.raises(Image.DecompressionBombError):          # 2400 px: over twice the patched limit
        Image.open(fn)
    assert np.array_equal(image_to_views(read_lf_image(fn, "mosaic", (5, 5)), "mosaic", 5, 5), g)
    assert Image.MAX_IMAGE_PIXELS == 100
    with pytest.raises(ValueError):
        read_lf_image(fn, "mosaic", (7, 5))
    assert Image.MAX_IMAGE_PIXELS == 100


# ---- options and the loader's choice ----------------------------------------------------------------------------------------
def test_parse_input_grid():
    from utils.utils_datasets import parse_input_grid
    assert parse_input_grid("14x14", "lenslet") == (14, 14)
    assert parse_input_grid(" 9x13 ", "mosaic") == (9, 13)
    assert parse_input_grid("", "views") is None and parse_input_grid(None, "views") is None
    for bad in ("14", "14x", "x14", "0x5", "5x0", "14X14", "14x14x1", "a", "-1x5"):
        with pytest.raises(ValueError, match="--input_grid"):
            parse_input_grid(bad, "lenslet")
    with pytest.raises(ValueError, match="--input_layout lenslet needs --input_grid"):
        parse_input_grid("", "lenslet")
    with pytest.raises(ValueError, match="--input_grid.*--input_layout"):
        parse_input_grid("5x5", "views")
    with pytest.raises(ValueError, match="--input_layout"):
        parse_input_grid("5x5", "macpi")


def _img_args(path, layout, grid="9x7", **kw):
    return _args(path, input_layout=layout, input_grid=grid, **kw)


def test_loader_choice_and_errors(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_image", _oracle_prepare_image)
    write_image(str(tmp_path / "B" / "z.png"), _grid(5, 5, 8, 8), "lenslet")
    write_image(str(tmp_path / "B" / "a.bmp"), _grid(5, 5, 8, 8), "lenslet")
    write_image(str(tmp_path / "A" / "m.png"), _grid(5, 5, 8, 8), "lenslet")
    _write_grid(str(tmp_path / "V" / "scene"), _grid(5, 5, 8, 8), "png")     # a view folder is not an image dataset
    (tmp_path / "SR_5x5_4x" / "B").mkdir(parents=True)                        # nor is the h5 layout looked at
    names, loaders, n = D.MultiTestSetDataLoader(_img_args(tmp_path, "lenslet", "5x5"), views="hr")
    assert names == ["A", "B"] and n == 3 and all(isinstance(d, D.ImageTestSet) for d in loaders)
    assert loaders[1].scenes == ["a", "z"] and [b[4][0] for b in loaders[1]] == ["a", "z"]
    names, loaders, n = D.MultiTestSetDataLoader(_img_args(tmp_path, "lenslet", "5x5", data_name="B"), views="lr")
    assert names == ["B"] and n == 2
    with pytest.raises(ValueError, match="--synthetic"):
        D.MultiTestSetDataLoader(_img_args(tmp_path, "mosaic", "5x5", synthetic=2), views="hr")
    with pytest.raises(ValueError, match="--input_grid"):
        D.MultiTestSetDataLoader(_img_args(tmp_path, "mosaic", ""), views="hr")
    with pytest.raises(ValueError, match="--input_grid"):
        D.MultiTestSetDataLoader(_img_args(tmp_path, "views", "5x5"), views="hr")
    with pytest.raises(FileNotFoundError, match="one image each"):
        D.MultiTestSetDataLoader(_img_args(tmp_path / "empty", "mosaic", "5x5"), views="hr")
    # duplicate stems
    write_image(str(tmp_path / "A" / "m.bmp"), _grid(5, 5, 8, 8), "lenslet")
    with pytest.raises(ValueError, match="m.*stored twice") as e:
        D.MultiTestSetDataLoader(_img_args(tmp_path, "lenslet", "5x5", data_name="A"), views="hr")
    assert str(tmp_path / "A") in str(e.value)


def test_scene_errors_name_the_file(tmp_path, monkeypatch):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_image", _oracle_prepare_image)
    fn = str(tmp_path / "Set" / "small.png")
    write_image(fn, _grid(5, 4, 8, 8), "mosaic")
    _, loaders, _ = D.MultiTestSetDataLoader(_img_args(tmp_path, "mosaic", "5x4"), views="hr")
    with pytest.raises(ValueError, match="smaller than angRes") as e:
        loaders[0][0]
    assert fn in str(e.value)
    _, loaders, _ = D.MultiTestSetDataLoader(_img_args(tmp_path, "mosaic", "3x4"), views="hr")
    with pytest.raises(ValueError, match="multiple of 3") as e:
        loaders[0][0]
    assert fn in str(e.value)
    fn = str(tmp_path / "Set2" / "big.bmp")
    write_image(fn, _grid(9, 7, 8, 8), "lenslet")
    for value in ("11x7", "9x9", "4x7"):
        _, loaders, _ = D.MultiTestSetDataLoader(_img_args(tmp_path, "lenslet", "9x7", data_name="Set2", full_grid=1,
                                                           grid_views=value), views="hr")
        with pytest.raises(ValueError, match="--grid_views") as e:
            loaders[0][0]
        assert fn in str(e.value)


# ---- ImageTestSet = ViewsTestSet ------------------------------------------------------------------------------------------------
_SELECTIONS = [dict(), dict(full_grid=1), dict(full_grid=1, grid_views="all"), dict(full_grid=1, grid_views="7x5")]


@pytest.mark.parametrize("layout", ["mosaic", "lenslet"])
@pytest.mark.parametrize("sel", _SELECTIONS)
@pytest.mark.parametrize("kind", ["hr", "lr"])
def test_image_set_equals_views_set(tmp_path, monkeypatch, layout, sel, kind):
    import utils.utils_datasets as D
    monkeypatch.setattr(D, "prepare_views", _oracle_prepare_uv)
    monkeypatch.setattr(D, "prepare_image", _oracle_prepare_image)
    grids = {"p": _grid(9, 7, 13, 11, seed=1), "q": _grid(9, 7, 10, 9, seed=2)}
    for s, g in grids.items():
        _write_grid(str(tmp_path / "views" / "Set" / s), g, "png")
        write_image(str(tmp_path / "image" / "Set" / (s + (".png" if s == "p" else ".bmp"))), g, layout)
    want_names, want_loaders, want_n = D.MultiTestSetDataLoader(_args(tmp_path / "views", scale=2, **sel), views=kind)
    names, loaders, n = D.MultiTestSetDataLoader(_img_args(tmp_path / "image", layout, scale=2, **sel), views=kind)
    assert names == want_names == ["Set"] and n == want_n == 2
    for got, want in zip(loaders[0], want_loaders[0]):
        assert got[4] == want[4]
        assert [int(x) for x in got[3]] == [int(x) for x in want[3]]
        for a, b in zip(got[:3], want[:3]):
            assert a.shape == b.shape and torch.equal(a, b)
    info = [int(x) for x in got[3]]
    assert info == {0: [5, 5], 1: [5, 5, 7], 2: [5, 5, 9, 7], 3: [5, 5, 7, 5]}[_SELECTIONS.index(sel)]


def test_save_layout_rejects_images_over_4gib(tmp_path):
    import pathlib
    import train
    huge = torch.zeros(1, 1).expand(5 * 8192, 5 * 8192)                      # 40960^2 RGB: 4.7 GiB as a BMP
    for layout in ("mosaic", "lenslet"):
        with pytest.raises(ValueError, match="BMP"):
            train._write_views(pathlib.Path(tmp_path), "s", huge, huge, 5, layout)
    assert not os.listdir(tmp_path)


# ---- world 2 over gloo ------------------------------------------------------------------------------------------------------------
def _run_split(data_root):
    """train.test over a lenslet dataset with the oracle preparation; returns (results, image files decoded)."""
    import train
    import utils.utils_datasets as D
    reads = []
    read, prepare = D.read_lf_image, D.prepare_image

    def counting(path, layout, grid):
        reads.append(os.path.basename(path))
        return read(path, layout, grid)

    D.read_lf_image, D.prepare_image = counting, _oracle_prepare_image
    try:
        args = _img_args(data_root, "lenslet", "5x5", data_name="Set")
        names, loaders, _ = D.MultiTestSetDataLoader(args, views="hr")
        return train.test(loaders[0], "cpu", _net(4), args), reads
    finally:
        D.read_lf_image, D.prepare_image = read, prepare


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
        write_image(str(data / "Set" / ("scene_%d.png" % i)), _grid(5, 5, 32, 32, seed=10 + i), "lenslet")
    out = tmp_path / "out"
    out.mkdir()
    port = 29500 + ((os.getpid() + 1300) % 2000)
    mp.spawn(_worker, args=(2, port, str(out), str(data)), nprocs=2, join=True)
    got = [pickle.load(open(out / f"rank{r}.pkl", "rb")) for r in range(2)]
    threads = torch.get_num_threads()
    torch.set_num_threads(2)
    try:
        want, reads = _run_split(str(data))
    finally:
        torch.set_num_threads(threads)
    assert reads == ["scene_0.png", "scene_1.png", "scene_2.png"]
    for r in range(2):
        (psnr, ssim, names), reads = got[r]
        assert names == want[2] == ["scene_0", "scene_1", "scene_2"]
        assert reads == ["scene_%d.png" % r, "scene_2.png"]     # scene 0 / 1: one full round; scene 2: the tail
        assert psnr[:2] == want[0][:2] and ssim[:2] == want[1][:2]
        assert np.abs(np.subtract(psnr[2:], want[0][2:])).max() <= 1e-4
