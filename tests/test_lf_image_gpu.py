"""Light fields stored as one image on the B200: lfsr_image_to_views_u8 and lfsr_ycbcr_to_rgb8_layout against numpy,
prepare_image against prepare_views and the oracle, and test.py / inference.py on mosaic and lenslet datasets against
the same light fields stored as View_u_v folders (one GPU, and torchrun on two)."""
import os

import numpy as np
import pytest
import torch
from PIL import Image

import lfsr_b200
from lfsr_b200 import lfutils
from oracle import weights
import view_oracle
from test_grid_rect_gpu import _rgb8_views_uv
from test_lf_image_cpu import image_to_views, views_to_image, write_image
from test_multi_gpu_eval_gpu import _compare, _eval_values, _need_two, _run
from test_view_input_cpu import _grid, _write_grid
from test_view_input_gpu import _entry

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A = 5
N = lfsr_b200._native
_CODE = {"mosaic": N.LAYOUT_MOSAIC, "lenslet": N.LAYOUT_LENSLET}


def _gather(img, layout, U, V, u0, v0, nu, nv, hc, wc):
    rows, cols = img.shape[:2]
    out = torch.full((nu, nv, hc, wc, 3), 7, dtype=torch.uint8, device=DEV)
    st = N.load().lfsr_image_to_views_u8(img.data_ptr(), layout, U, V, rows // U, cols // V, u0, v0, nu, nv, hc, wc,
                                         out.data_ptr(), torch.cuda.current_stream(DEV).cuda_stream)
    return st, out


# ---- kernels ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["mosaic", "lenslet"])
@pytest.mark.parametrize("U,V,H,W", [(9, 13, 23, 17), (14, 14, 15, 21)])
@pytest.mark.parametrize("s", [2, 3, 4])
def test_image_to_views_bit_exact(layout, U, V, H, W, s):
    g = np.random.RandomState(U * V + H + s).randint(0, 256, (U, V, H, W, 3)).astype(np.uint8)
    img = torch.from_numpy(views_to_image(g, layout)).to(DEV)
    hc, wc = H - H % s, W - W % s
    # central A x A, central 9 x 9, the whole grid, and off-centre selections touching each border
    for u0, v0, nu, nv in [((U - A) // 2, (V - A) // 2, A, A), ((U - 9) // 2, (V - 9) // 2, 9, 9), (0, 0, U, V),
                           (0, V - 3, 4, 3), (U - 2, 1, 2, 5), (3, 2, 1, 1)]:
        st, out = _gather(img, _CODE[layout], U, V, u0, v0, nu, nv, hc, wc)
        assert st == 0, N.load().lfsr_last_error()
        assert np.array_equal(out.cpu().numpy(), g[u0:u0 + nu, v0:v0 + nv, :hc, :wc]), (u0, v0, nu, nv)


def test_image_to_views_rejects_bad_geometry():
    U, V, H, W = 5, 7, 6, 8
    img = torch.zeros((U * H, V * W, 3), dtype=torch.uint8, device=DEV)
    lib = N.load()
    assert _gather(img, 2, U, V, 0, 0, U, V, H, W)[0] == 0
    for layout, u0, v0, nu, nv, hc, wc in [(0, 0, 0, 1, 1, 6, 8), (3, 0, 0, 1, 1, 6, 8), (-1, 0, 0, 1, 1, 6, 8),
                                           (1, 1, 0, 5, 1, 6, 8), (2, 0, 3, 1, 5, 6, 8), (1, -1, 0, 1, 1, 6, 8),
                                           (2, 0, 0, 0, 1, 6, 8), (1, 0, 0, 1, 1, 7, 8), (2, 0, 0, 1, 1, 6, 9),
                                           (1, 0, 0, 1, 1, 0, 8)]:
        out = torch.zeros((1,), dtype=torch.uint8, device=DEV)
        st = lib.lfsr_image_to_views_u8(img.data_ptr(), layout, U, V, H, W, u0, v0, nu, nv, hc, wc, out.data_ptr(),
                                        torch.cuda.current_stream(DEV).cuda_stream)
        assert st == -1, (layout, u0, v0, nu, nv, hc, wc)
    # an image side of 2^31 pixels or more (no memory is touched: the call is rejected first)
    assert lib.lfsr_image_to_views_u8(img.data_ptr(), 1, 2, 2, 1 << 30, 8, 0, 0, 1, 1, 1, 1, img.data_ptr(), None) == -1
    assert lib.lfsr_image_to_views_u8(img.data_ptr(), 2, 3, 3, 8, (1 << 31) // 3 + 1, 0, 0, 1, 1, 1, 1, img.data_ptr(),
                                      None) == -1
    torch.cuda.synchronize()


def _colour(au, av, h, w):
    rs = np.random.RandomState(au * 10 + av)
    y = torch.from_numpy(rs.uniform(-0.05, 1.05, (au * h, av * w)).astype(np.float32)).to(DEV)
    c = torch.from_numpy(rs.uniform(0.2, 0.8, (2, au * h, av * w)).astype(np.float32)).to(DEV)
    return y, c


@pytest.mark.parametrize("au,av,h,w", [(5, 5, 9, 13), (9, 13, 7, 11), (14, 14, 6, 5)])
def test_ycbcr_to_rgb8_layouts(au, av, h, w):
    y, c = _colour(au, av, h, w)
    views = lfutils.sai_to_rgb8(y, c, (au, av), "views")
    assert torch.equal(views, lfutils.sai_to_rgb8_views(y, c, (au, av)))          # layout 0 = lfsr_ycbcr_to_rgb8_uv
    g = views.cpu().numpy()
    assert np.array_equal(g, _rgb8_views_uv(y.cpu().numpy(), c.cpu().numpy(), au, av))
    for layout in ("mosaic", "lenslet"):
        img = lfutils.sai_to_rgb8(y, c, (au, av), layout)
        assert img.shape == (au * h, av * w, 3)
        assert np.array_equal(img.cpu().numpy(), views_to_image(g, layout)), layout
    if au == av:
        assert torch.equal(lfutils.sai_to_rgb8(y, c, au, "lenslet"), lfutils.sai_to_rgb8(y, c, (au, au), "lenslet"))


def test_ycbcr_to_rgb8_layout_rejects_unknown_layout():
    y, c = _colour(5, 5, 4, 4)
    out = torch.empty((5 * 4 * 5 * 4 * 3,), dtype=torch.uint8, device=DEV)
    inv255 = np.zeros(9)
    off = np.zeros(3)
    for layout in (-1, 3):
        st = N.load().lfsr_ycbcr_to_rgb8_layout(y.data_ptr(), c[0].data_ptr(), c[1].data_ptr(), out.data_ptr(), 5, 5, 4,
                                                4, layout, inv255.ctypes.data, off.ctypes.data, None)
        assert st == -1
    with pytest.raises(ValueError, match="layout"):
        lfutils.sai_to_rgb8(y, c, 5, "macpi")


# ---- preparation --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["hr", "lr"])
@pytest.mark.parametrize("layout", ["mosaic", "lenslet"])
@pytest.mark.parametrize("U,V,H,W,scale", [(7, 7, 34, 26, 4), (5, 9, 30, 41, 2)])
def test_prepare_image_equals_prepare_views(kind, layout, U, V, H, W, scale):
    g = _grid(U, V, H, W, seed=H + V)
    img = views_to_image(g, layout)
    got = lfutils.prepare_image(img, layout, (U, V), A, scale, kind)
    want = lfutils.prepare_views(g, A, scale, kind)
    u0, v0 = (U - A) // 2, (V - A) // 2           # view_oracle takes a square grid: give it the central A x A itself
    oracle = view_oracle.prepare_views(g[u0:u0 + A, v0:v0 + A], A, scale, kind)
    for a, b, c in zip(got, want, oracle):
        if b is None:
            assert a is None and c is None
            continue
        assert a.is_cuda and a.dtype == torch.float32 and torch.equal(a, b)
        np.testing.assert_array_max_ulp(a.cpu().numpy(), c, maxulp=1)
    # a rectangular selection goes through the same gather
    lr1, _, cb1 = lfutils.prepare_image(img, layout, (U, V), (5, 5 if V < 7 else 7), scale, "lr")
    lr2, _, cb2 = lfutils.prepare_views(g, (5, 5 if V < 7 else 7), scale, "lr")
    assert torch.equal(lr1, lr2) and torch.equal(cb1, cb2)


# ---- test.py / inference.py --------------------------------------------------------------------------------------------------
def _datasets(root, grids, layouts):
    """the same light fields as View_u_v folders under <root>/views and as one image per scene under <root>/<layout>"""
    for k, (s, g) in enumerate(grids.items()):
        _write_grid(os.path.join(root, "views", "Set", s), g, "png" if k % 2 == 0 else "bmp")
        for layout in layouts:
            write_image(os.path.join(root, layout, "Set", s + (".bmp" if k % 2 == 0 else ".png")), g, layout)


def _ckpt(tmp_path, name, scale):
    ckpt = tmp_path / ("%s_x%d.pth" % (name, scale))
    torch.save({"state_dict": weights.make_state_dict(name, scale, 1234)}, ckpt)
    return ckpt


def _bmps(log):
    test_dir = next(log.rglob("TEST"))
    return {os.path.relpath(str(b), test_dir): b.read_bytes() for b in test_dir.rglob("*.bmp")}


@pytest.mark.parametrize("name,scale", [("MyEfficientLFNet", 4), ("DistgSSR", 2)])
def test_test_py_on_image_datasets(tmp_path, name, scale):
    """three 9x9 light fields (view sizes 64x48, 80x64, 48x48) as View_u_v folders, lenslet images and mosaic images:
    the same printed metrics, evaluation.xls and BMPs"""
    grids = {"a": _grid(9, 9, 64, 48, seed=1), "b": _grid(9, 9, 80, 64, seed=2), "c": _grid(9, 9, 48, 48, seed=3)}
    data = tmp_path / "data"
    _datasets(str(data), grids, ("lenslet", "mosaic"))
    ckpt = _ckpt(tmp_path, name, scale)
    flags = ["--model_name", name, "--angRes", "5", "--scale_factor", str(scale), "--path_pre_pth", str(ckpt)]
    want_out, want_log = _entry(tmp_path, "views", "test.py", flags + ["--path_for_test", str(data / "views") + "/"])
    want_bmps = _bmps(want_log)
    assert len(want_bmps) == 3 * A * A
    want_eval = _eval_values(list(want_log.rglob("evaluation.*")))
    assert len(want_eval) == 3 + 2
    for layout in ("lenslet", "mosaic"):
        out, log = _entry(tmp_path, layout, "test.py", flags + ["--path_for_test", str(data / layout) + "/",
                                                                "--input_layout", layout, "--input_grid", "9x9"])
        for key in ("Test on ", "The mean psnr"):
            got = [ln for ln in out.splitlines() if ln.startswith(key)]
            want = [ln for ln in want_out.splitlines() if ln.startswith(key)]
            assert got == want and len(got) == 1, (layout, got, want)
        assert _eval_values(list(log.rglob("evaluation.*"))) == want_eval, layout
        assert _bmps(log) == want_bmps, layout


def _readback(path):
    with Image.open(path) as im:
        return np.asarray(im.convert("RGB"))


@pytest.mark.parametrize("grid,extra,sr_grid", [((7, 7), [], (A, A)),
                                                ((14, 14), ["--full_grid", "1", "--grid_views", "9x9"], (9, 9)),
                                                ((7, 7), ["--self_ensemble", "1"], (A, A))])
def test_inference_py_save_layouts(tmp_path, grid, extra, sr_grid):
    name, scale = "DistgSSR", 2
    data = tmp_path / "data"
    scenes = {"p": _grid(*grid, 32, 40, seed=5), "q": _grid(*grid, 36, 32, seed=6)}
    for k, (s, g) in enumerate(scenes.items()):
        write_image(str(data / "Set" / (s + (".png" if k == 0 else ".bmp"))), g, "lenslet")
    ckpt = _ckpt(tmp_path, name, scale)
    flags = ["--model_name", name, "--angRes", "5", "--scale_factor", str(scale), "--path_pre_pth", str(ckpt),
             "--path_for_test", str(data) + "/", "--input_layout", "lenslet", "--input_grid", "%dx%d" % grid] + extra
    _, log = _entry(tmp_path, "views", "inference.py", flags)
    ref = next(log.rglob("TEST")) / "Set"
    for layout in ("lenslet", "mosaic"):
        _, log = _entry(tmp_path, layout, "inference.py", flags + ["--save_layout", layout])
        out = next(log.rglob("TEST")) / "Set"
        assert sorted(os.listdir(out)) == ["p.bmp", "q.bmp"]
        for s in scenes:
            nu, nv = sr_grid
            views = np.stack([np.stack([_readback(ref / s / ("View_%d_%d.bmp" % (i, j))) for j in range(nv)])
                              for i in range(nu)])
            assert len(os.listdir(ref / s)) == nu * nv
            got = _readback(out / (s + ".bmp"))
            assert got.shape == (nu * views.shape[2], nv * views.shape[3], 3)
            assert np.array_equal(got, views_to_image(views, layout)), (layout, s)
            assert np.array_equal(image_to_views(got, layout, nu, nv), views)


def test_test_py_lenslet_two_gpus(tmp_path):
    _need_two()
    data = tmp_path / "data"
    for i in range(3):
        write_image(str(data / "Set" / ("s%d.png" % i)), _grid(7, 7, 64, 64, seed=40 + i), "lenslet")
    ckpt = _ckpt(tmp_path, "MyEfficientLFNet", 4)
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--path_pre_pth", str(ckpt),
             "--path_for_test", str(data) + "/", "--input_layout", "lenslet", "--input_grid", "7x7"]
    _compare(_run(tmp_path, "single", "test.py", flags, 1), _run(tmp_path, "multi", "test.py", flags, 2), 3, True)
