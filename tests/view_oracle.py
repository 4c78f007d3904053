"""Test infrastructure, not product code: the light-field preparation of include/lfsr.h ("View preparation") in numpy,
next to the oracle of oracle/lf_oracle.py (whose MATLAB-style imresize it uses). It restates BasicLFSR's data generators
(Generate_Data_for_Test.py, Generate_Data_for_inference.py) as DESIGN.md row f-7 records them; those scripts are not in
this tree, so parity with them is unpinned."""
import numpy as np

from oracle import lf_oracle


def rgb2ycbcr(x: np.ndarray) -> np.ndarray:
    """BasicLFSR's rgb2ycbcr as its data generators use it: fp64, term by term, left to right, then / 255. A term's sign
    is folded into its constant (a - k*b == a + (-k)*b exactly), which gives the same numbers as the written form."""
    x = x.astype(np.float64)
    r, g, b = x[..., 0], x[..., 1], x[..., 2]
    y = np.zeros(x.shape, dtype=np.float64)
    y[..., 0] = 65.481 * r + 128.553 * g + 24.966 * b + 16.0
    y[..., 1] = -37.797 * r - 74.203 * g + 112.0 * b + 128.0
    y[..., 2] = 112.0 * r - 93.786 * g - 18.214 * b + 128.0
    return y / 255.0


def _views_to_sai(v: np.ndarray) -> np.ndarray:
    """[a1, a2, h, w, ...] -> [(a1 h), (a2 w), ...]."""
    a1, a2, h, w = v.shape[:4]
    return np.ascontiguousarray(v.swapaxes(1, 2)).reshape(a1 * h, a2 * w, *v.shape[4:])


def prepare_views(views: np.ndarray, ang: int, scale: int, kind: str = "hr", with_lr_rgb: bool = False):
    """the light-field preparation of include/lfsr.h ("View preparation"; BasicLFSR's Generate_Data_for_Test.py and
    Generate_Data_for_inference.py as DESIGN.md row f-7 records them): views [U, V, H, W, 3], uint8 (divided by 255.0)
    or fp64 in [0, 1] -> (Lr_SAI_y, Hr_SAI_y or None, Sr_SAI_cbcr [2, ...]) as fp32 SAI mosaics. with_lr_rgb also
    returns the fp64 LR views [A, A, h, w, 3] (kind "hr": imresize(x, 1/scale); kind "lr": x)."""
    U, V, H, W, _ = views.shape
    u0, v0 = (U - ang) // 2, (V - ang) // 2
    x = views[u0:u0 + ang, v0:v0 + ang, :H - H % scale, :W - W % scale]
    x = x.astype(np.float64) / 255.0 if x.dtype == np.uint8 else x.astype(np.float64)
    per_view = lambda f, v: np.stack([np.stack([f(v[i, j]) for j in range(ang)]) for i in range(ang)])
    if kind == "hr":
        hr_y = _views_to_sai(rgb2ycbcr(x)[..., 0]).astype("single")
        lr_rgb = per_view(lambda im: lf_oracle.imresize(im, scalar_scale=1 / scale), x)
    else:
        hr_y, lr_rgb = None, x
    lr_y = _views_to_sai(rgb2ycbcr(lr_rgb)[..., 0]).astype("single")
    sr_rgb = per_view(lambda im: lf_oracle.imresize(im, scalar_scale=scale), lr_rgb)
    sr_cbcr = np.ascontiguousarray(_views_to_sai(rgb2ycbcr(sr_rgb)[..., 1:3]).transpose(2, 0, 1)).astype("single")
    return (lr_y, hr_y, sr_cbcr, lr_rgb) if with_lr_rgb else (lr_y, hr_y, sr_cbcr)
