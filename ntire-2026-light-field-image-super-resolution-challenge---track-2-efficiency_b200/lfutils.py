"""Device-side mirrors of the reference's patch-pipeline functions (utils/utils.py:91-178).

Same names, argument meaning and return layouts as the reference so `train.test()` /
`inference.test()` run unchanged; the arithmetic runs in liblfsr_b200 kernels on the GPU. Tensors
that arrive on the host (the reference keeps `subLFout`, `Hr_SAI_y` on the CPU, train.py:303,322)
are staged to the current CUDA device and the result is returned on the caller's device. There is
no CPU implementation behind these functions.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N
from . import kernels as K


def _device_for(t: torch.Tensor, ops=None) -> torch.device:
    if t.is_cuda:
        return t.device
    if ops is not None and getattr(ops, "name", "cuda") != "cuda":
        return t.device          # an injected test backend (tests/opref.RefOps) works where the tensors live
    if not torch.cuda.is_available():
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    return torch.device("cuda", torch.cuda.current_device())


def divide_geometry(h0: int, w0: int, patch_size: int, stride: int):
    bdr = (patch_size - stride) // 2
    return bdr, (h0 + bdr * 2 - 1) // stride, (w0 + bdr * 2 - 1) // stride


def check_divide_geometry(h0: int, w0: int, patch_size: int, stride: int) -> None:
    """The reference's LFdivide only works when its unfold yields exactly the numU x numV patches its rearrange expects
    (utils/utils.py:152-166): ImageExtend pads bdr above and bdr + stride - 1 below out of ONE mirrored copy of the view
    (at most n rows), unfold then gives (ext - patch) // stride + 1 windows. In practice: patch == 2 * stride and views no
    smaller than ~patch / 2. Everything else raises inside the reference (einops shape error); same here, up front."""
    bdr = (patch_size - stride) // 2
    for n, what in ((h0, "height"), (w0, "width")):
        ext = n + bdr + min(bdr + stride - 1, n)
        windows = (ext - patch_size) // stride + 1 if ext >= patch_size else 0
        want = (n + 2 * bdr - 1) // stride
        if n <= 0 or bdr > n or windows < 1 or windows != want:
            raise ValueError(f"LFdivide: view {what} {n} cannot be tiled with patch {patch_size} / stride {stride} "
                             f"(the reference's unfold gives {windows} windows where it expects {want})")


def LFdivide(data: torch.Tensor, angRes: int, patch_size: int, stride: int, rows=None, ops=None) -> torch.Tensor:
    """data [(a1 h0), (a2 w0)] -> subLF [numU, numV, a1*P, a2*P]  (utils/utils.py:152-166).
    rows=(u0,u1) returns only that band of the patch grid (multi-GPU scene sharding)."""
    if data.dim() != 2:
        raise ValueError(f"LFdivide expects a 2-D SAI mosaic, got {tuple(data.shape)}")
    dev = _device_for(data, ops)
    ops = ops or K.default_ops()
    src = data.to(device=dev, dtype=torch.float32).contiguous()
    H, W = src.shape
    h0, w0 = H // angRes, W // angRes
    check_divide_geometry(h0, w0, patch_size, stride)
    _, num_u, num_v = divide_geometry(h0, w0, patch_size, stride)
    u0, u1 = (0, num_u) if rows is None else rows
    sub = torch.empty((u1 - u0, num_v, angRes * patch_size, angRes * patch_size), dtype=torch.float32, device=dev)
    ops.divide_rows(src, sub, angRes, h0, w0, patch_size, stride, u0, u1)
    return sub if data.is_cuda else sub.to(data.device)


def LFintegrate(subLF: torch.Tensor, angRes: int, pz: int, stride: int, h: int, w: int, ops=None) -> torch.Tensor:
    """subLF [n1, n2, a1*pz, a2*pz] (or 6-D n1 n2 a1 a2 pz pz) -> outLF [a1, a2, h, w]
    (utils/utils.py:169-178). The result is a view of the stitched SAI mosaic, so the reference's
    following 'a1 a2 h w -> 1 1 (a1 h) (a2 w)' rearrange (train.py:319) is a cheap copy."""
    dev = _device_for(subLF, ops)
    ops = ops or K.default_ops()
    sub = subLF.to(device=dev, dtype=torch.float32)
    if sub.dim() == 6:
        n1, n2, a1, a2, ph, pw = sub.shape
        sub = sub.permute(0, 1, 2, 4, 3, 5).reshape(n1, n2, a1 * ph, a2 * pw)
    if sub.dim() != 4:
        raise ValueError(f"LFintegrate expects a 4-D or 6-D tensor, got {tuple(subLF.shape)}")
    sub = sub.contiguous()
    n1, n2 = sub.shape[:2]
    # the reference slices [0:h, 0:w] out of the n1*stride x n2*stride stitched views (utils.py:176-178): with
    # non-overlapping patches the grid can be smaller than the scene and the slice returns what is covered
    h, w = min(h, n1 * stride), min(w, n2 * stride)
    mosaic = torch.empty((angRes * h, angRes * w), dtype=torch.float32, device=dev)
    ops.integrate_rows(sub, mosaic, angRes, pz, stride, h, w, n1, n2, 0, n1)
    out = mosaic.view(angRes, h, angRes, w).permute(0, 2, 1, 3)
    return out if subLF.is_cuda else out.to(subLF.device)


def metric_views(label_sai: torch.Tensor, out_sai: torch.Tensor, angRes: int, ops=None):
    """per-view PSNR / SSIM of two SAI mosaics [(a1 h), (a2 w)] -> float32 arrays [A, A]."""
    dev = _device_for(out_sai if out_sai.is_cuda else label_sai, ops)
    ops = ops or K.default_ops()
    if label_sai.dim() != 2 or tuple(label_sai.shape) != tuple(out_sai.shape):
        # the reference crops SR to the HR size before this point (train.py:316) and skimage raises on a mismatch
        raise ValueError(f"cal_metrics: label {tuple(label_sai.shape)} and output {tuple(out_sai.shape)} mosaics differ")
    la = label_sai.to(device=dev, dtype=torch.float32).contiguous()
    ou = out_sai.to(device=dev, dtype=torch.float32).contiguous()
    H, W = la.shape
    if H % angRes or W % angRes:
        raise ValueError(f"cal_metrics: mosaic {H}x{W} is not divisible by angRes={angRes}")
    h, w = H // angRes, W // angRes
    acc = torch.zeros(2 * angRes * angRes, dtype=torch.float64, device=dev)
    ops.metric_sums(la, ou, angRes, h, w, acc)
    a = acc.cpu().numpy().reshape(angRes, angRes, 2)
    mse = a[..., 0] / float(h * w)
    with np.errstate(divide="ignore"):
        psnr = (10.0 * np.log10(1.0 / mse)).astype(np.float32)
    ssim = (a[..., 1] / float((h - 10) * (w - 10))).astype(np.float32)
    return psnr, ssim


def cal_metrics(args, label: torch.Tensor, out: torch.Tensor, ops=None):
    """(PSNR_mean, SSIM_mean) over views with value > 0 (utils/utils.py:91-134, SR task)."""
    if getattr(args, "task", "SR") != "SR":
        raise N.LfsrError("cal_metrics: only the SR task is on the accelerated path")
    A = int(args.angRes_in)
    if label.dim() == 5:                       # [B, C, U, V?...] -> the reference permutes (0,1,3,2,4) and unsqueezes
        label = label.permute((0, 1, 3, 2, 4)).unsqueeze(0)
        out = out.permute((0, 1, 3, 2, 4)).unsqueeze(0)
    if label.dim() == 6:                       # B C U h V w -> mosaic
        B, C, U, h, V, w = label.shape
        label = label.reshape(B, C, U * h, V * w)
        out = out.reshape(B, C, U * h, V * w)
        A = U
    if label.dim() != 4:
        raise ValueError(f"cal_metrics: unsupported label shape {tuple(label.shape)}")
    B = label.shape[0]
    PSNR = np.zeros((B, A, A), dtype="float32")
    SSIM = np.zeros((B, A, A), dtype="float32")
    for b in range(B):
        PSNR[b], SSIM[b] = metric_views(label[b, 0], out[b, 0], A, ops)
    valid_psnr = np.sum(PSNR > 0)
    psnr_mean = PSNR.sum() / valid_psnr if valid_psnr > 0 else 0.0
    valid_ssim = np.sum(SSIM > 0)
    ssim_mean = SSIM.sum() / valid_ssim if valid_ssim > 0 else 0.0
    return psnr_mean, ssim_mean


# ---- MATLAB-style imresize (utils/imresize.py) ---------------------------------------------------------------------------
def _cubic(x):
    ax = np.abs(np.asarray(x, dtype=np.float64))
    ax2, ax3 = ax * ax, ax * ax * ax
    return (1.5 * ax3 - 2.5 * ax2 + 1) * (ax <= 1) + (-0.5 * ax3 + 2.5 * ax2 - 4 * ax + 2) * ((1 < ax) & (ax <= 2))


def _triangle(x):
    x = np.asarray(x, dtype=np.float64)
    return (x + 1) * ((x >= -1) & (x < 0)) + (1 - x) * ((x <= 1) & (x >= 0))


def resize_contributions(in_length: int, out_length: int, scale: float, method: str = "bicubic"):
    """Host side of one resampled dimension (utils/imresize.py:32-55): per output sample its <= ceil(4/min(scale,1)) + 2
    normalised kernel weights (Keys cubic A = -0.5 or triangle, stretched by 1/scale when shrinking = antialiasing) and
    the symmetric-border source indices. A few KB of fp64 / int32, recomputed per call like the reference does."""
    kernel = _cubic if method == "bicubic" else _triangle
    if scale < 1:
        h, kernel_width = (lambda t: scale * kernel(scale * t)), 4.0 / scale
    else:
        h, kernel_width = kernel, 4.0
    u = np.arange(1, out_length + 1, dtype=np.float64) / scale + 0.5 * (1 - 1 / scale)
    left = np.floor(u - kernel_width / 2)
    taps = int(np.ceil(kernel_width)) + 2
    ind = (left[:, None] + np.arange(taps) - 1).astype(np.int32)
    w = h(u[:, None] - ind - 1)
    w = w / w.sum(axis=1, keepdims=True)
    aux = np.concatenate((np.arange(in_length), np.arange(in_length - 1, -1, -1))).astype(np.int32)
    ind = aux[np.mod(ind, aux.size)]
    keep = np.nonzero(np.any(w, axis=0))[0]
    return np.ascontiguousarray(w[:, keep]), np.ascontiguousarray(ind[:, keep])


def imresize(I, scalar_scale=None, method="bicubic", output_shape=None, mode="vec"):
    """utils/imresize.py:104-145 on the GPU: same signature and return type (numpy in -> numpy out, torch in -> torch out
    on the caller's device); [H, W] or [H, W, C]; float inputs give float64, uint8 inputs are clipped and rounded
    half-to-even after each pass like the reference. The two separable passes run in lfsr_resample_f64 (fp64, tap-order
    sums); `mode` is accepted for compatibility ("org" and "vec" give the same numbers)."""
    if method not in ("bicubic", "bilinear"):
        raise ValueError(f"unidentified method {method!r}")
    if scalar_scale is None and output_shape is None:
        raise ValueError("scalar_scale OR output_shape should be defined")
    as_numpy = isinstance(I, np.ndarray)
    t = torch.from_numpy(np.ascontiguousarray(I)) if as_numpy else I
    if t.dim() not in (2, 3):
        raise ValueError(f"expected [H, W] or [H, W, C], got {tuple(t.shape)}")
    home = t.device
    dev = _device_for(t)
    if dev.type != "cuda":
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    is_u8 = t.dtype == torch.uint8
    H, W = t.shape[:2]
    if scalar_scale is not None:
        scale = [float(scalar_scale)] * 2
        out_size = [int(np.ceil(scale[0] * H)), int(np.ceil(scale[1] * W))]
    else:
        scale = [1.0 * output_shape[0] / H, 1.0 * output_shape[1] / W]
        out_size = [int(output_shape[0]), int(output_shape[1])]
    cur = t.to(dev).to(torch.float64)
    if cur.dim() == 2:
        cur = cur[:, :, None]
    cur = _resample_passes(cur[None], scale, out_size, method, is_u8)[0]
    if is_u8:
        cur = cur.to(torch.uint8)
    if t.dim() == 2:
        cur = cur[:, :, 0]
    cur = cur.to(home)
    return cur.numpy() if as_numpy else cur


def _resample_passes(cur: torch.Tensor, scale, out_size, method: str, is_u8: bool = False) -> torch.Tensor:
    """the two separable passes of imresize over a batch of images: fp64 [N, H, W, C] on the device -> [N, H', W', C].
    The dimension with the smaller scale goes first (rows first on a tie); one lfsr_resample_f64 launch per pass covers
    all N images: rows as [N][H][W*C], columns as [N*H'][W][C]. Each output sample is the same tap-order sum as for
    a single image, so the batch is bit-identical to N separate calls."""
    dev = cur.device
    lib = N.load()
    cur = cur.contiguous()
    stream = torch.cuda.current_stream(dev).cuda_stream
    for dim in np.argsort(np.array(scale)):
        dim = int(dim)
        w, ind = resize_contributions(cur.shape[dim + 1], out_size[dim], scale[dim], method)
        wd, idd = torch.from_numpy(w).to(dev), torch.from_numpy(ind).to(dev)
        shape = list(cur.shape)
        outer = shape[0] if dim == 0 else shape[0] * shape[1]
        inner = shape[2] * shape[3] if dim == 0 else shape[3]
        in_len = shape[dim + 1]
        shape[dim + 1] = out_size[dim]
        out = torch.empty(shape, dtype=torch.float64, device=dev)
        N.check(lib.lfsr_resample_f64(cur.data_ptr(), out.data_ptr(), wd.data_ptr(), idd.data_ptr(), outer, in_len, out_size[dim],
                                      inner, w.shape[1], stream), "lfsr_resample_f64")
        cur = out.clamp_(0, 255).round_() if is_u8 else out
    return cur


def imresize_views(views: torch.Tensor, scalar_scale: float, method: str = "bicubic") -> torch.Tensor:
    """imresize(view, scalar_scale) of every view of a light field at once: fp64 [..., H, W, C] on the device (the
    leading dimensions, e.g. the A x A views, are flattened) -> fp64 [..., ceil(s H), ceil(s W), C], bit-identical to
    calling imresize on each view (the float path; uint8 views go through imresize one by one)."""
    if not views.is_cuda:
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    if views.dtype != torch.float64 or views.dim() < 3:
        raise ValueError(f"imresize_views expects fp64 [..., H, W, C] views, got {tuple(views.shape)} {views.dtype}")
    lead, (H, W, C) = views.shape[:-3], views.shape[-3:]
    scale = [float(scalar_scale)] * 2
    out_size = [int(np.ceil(scale[0] * H)), int(np.ceil(scale[1] * W))]
    out = _resample_passes(views.reshape(-1, H, W, C), scale, out_size, method)
    return out.reshape(*lead, *out.shape[1:])


# ---- colour / BMP tail of test() (train.py:329-341) -------------------------------------------------------------------------
_BT601 = np.array([[65.481, 128.553, 24.966], [-37.797, -74.203, 112.0], [112.0, -93.786, -18.214]])


def ang_pair(angRes):
    """(a1, a2) of an angular size given as an int (a square grid) or as a (U, V) pair"""
    if isinstance(angRes, (tuple, list)):
        if len(angRes) != 2:
            raise ValueError(f"an angular size is an int or a (U, V) pair, got {angRes!r}")
        return int(angRes[0]), int(angRes[1])
    return int(angRes), int(angRes)


def sai_to_rgb8_views(sr_y: torch.Tensor, sr_cbcr: torch.Tensor, angRes) -> torch.Tensor:
    """Sr_SAI_y [.., (a1 h), (a2 w)] + Sr_SAI_cbcr [.., 2, (a1 h), (a2 w)] -> uint8 [a1, a2, h, w, 3] on the device:
    torch.cat + ycbcr2rgb (fp64) + clip(0,1)*255 + astype(uint8) + the view rearrange of train.py:332-335 in one kernel.
    angRes: a1 = a2 as an int, or the pair (a1, a2) of a rectangular grid."""
    y = sr_y.reshape(sr_y.shape[-2:])
    cbcr = sr_cbcr.reshape(2, *sr_cbcr.shape[-2:])
    if cbcr.shape[-2:] != y.shape:
        raise ValueError(f"Y {tuple(y.shape)} and CbCr {tuple(cbcr.shape)} mosaics differ in size")
    dev = _device_for(y)
    if dev.type != "cuda":
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    H, W = y.shape
    au, av = ang_pair(angRes)
    if H % au or W % av:
        raise ValueError(f"mosaic {H}x{W} is not divisible by angRes={angRes}")
    y = y.to(dev, torch.float32).contiguous()
    cbcr = cbcr.to(dev, torch.float32).contiguous()
    inv = np.linalg.inv(_BT601)                                   # exactly the reference's constants (utils/utils.py:192-198)
    offset = np.ascontiguousarray(np.matmul(inv, np.array([16, 128, 128])))
    inv255 = np.ascontiguousarray(inv * 255)
    out = torch.empty((au, av, H // au, W // av, 3), dtype=torch.uint8, device=dev)
    lib, stream = N.load(), torch.cuda.current_stream(dev).cuda_stream
    if not isinstance(angRes, (tuple, list)):
        N.check(lib.lfsr_ycbcr_to_rgb8(y.data_ptr(), cbcr[0].data_ptr(), cbcr[1].data_ptr(), out.data_ptr(), angRes,
                                       H // angRes, W // angRes, inv255.ctypes.data, offset.ctypes.data, stream),
                "lfsr_ycbcr_to_rgb8")
    else:
        N.check(lib.lfsr_ycbcr_to_rgb8_uv(y.data_ptr(), cbcr[0].data_ptr(), cbcr[1].data_ptr(), out.data_ptr(), au, av,
                                          H // au, W // av, inv255.ctypes.data, offset.ctypes.data, stream),
                "lfsr_ycbcr_to_rgb8_uv")
    return out


# ---- input side: RGB views -> the Lr_SAI_y / Hr_SAI_y / Sr_SAI_cbcr tensors of a test set (include/lfsr.h) ------------------
def rgb_to_ycbcr_mosaic(views: torch.Tensor, angRes, y: bool = True, cbcr: bool = True):
    """views [a1, a2, h, w, 3] (or [a1*a2, h, w, 3]) on the device, uint8 or fp64 in [0, 1] -> (Y mosaic [(a1 h), (a2 w)],
    CbCr mosaics [2, (a1 h), (a2 w)]) in fp32, BasicLFSR's term-by-term rgb2ycbcr in one kernel; an output that is not
    asked for is None. angRes: a1 = a2 as an int, or the pair (a1, a2)."""
    if not views.is_cuda:
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    if views.dtype not in (torch.uint8, torch.float64):
        raise ValueError(f"views must be uint8 or float64, got {views.dtype}")
    h, w, c = views.shape[-3:]
    au, av = ang_pair(angRes)
    if c != 3 or views.numel() != au * av * h * w * 3:
        raise ValueError(f"expected {au}x{av} RGB views, got {tuple(views.shape)}")
    if not (y or cbcr):
        raise ValueError("rgb_to_ycbcr_mosaic: ask for Y, CbCr or both")
    src = views.contiguous()
    dev = src.device
    oy = torch.empty((au * h, av * w), dtype=torch.float32, device=dev) if y else None
    oc = torch.empty((2, au * h, av * w), dtype=torch.float32, device=dev) if cbcr else None
    ptr = lambda t: None if t is None else t.data_ptr()
    outs = (src.data_ptr(), int(src.dtype == torch.uint8), ptr(oy), None if oc is None else oc[0].data_ptr(),
            None if oc is None else oc[1].data_ptr())
    stream = torch.cuda.current_stream(dev).cuda_stream
    if not isinstance(angRes, (tuple, list)):
        N.check(N.load().lfsr_rgb_to_ycbcr_mosaic(*outs, angRes, h, w, stream), "lfsr_rgb_to_ycbcr_mosaic")
    else:
        N.check(N.load().lfsr_rgb_to_ycbcr_mosaic_uv(*outs, au, av, h, w, stream), "lfsr_rgb_to_ycbcr_mosaic_uv")
    return oy, oc


def central_views(rgb8: np.ndarray, angRes, scale: int) -> np.ndarray:
    """the views the preparation uses, as a host view (no copy): the central angRes x angRes of a [U, V, H, W, 3] grid
    (or the central a1 x a2 for angRes = (a1, a2)), each cropped top-left to a multiple of `scale` in height and width."""
    a = np.asarray(rgb8)
    if a.ndim != 5 or a.shape[-1] != 3:
        raise ValueError(f"expected RGB views [U, V, H, W, 3], got {a.shape}")
    U, V, H, W, _ = a.shape
    au, av = ang_pair(angRes)
    if U < au or V < av:
        raise ValueError(f"a {U}x{V} grid of views has no central {au}x{av}")
    hc, wc = H - H % scale, W - W % scale
    if hc == 0 or wc == 0:
        raise ValueError(f"views of {H}x{W} are smaller than the scale factor {scale}")
    u0, v0 = (U - au) // 2, (V - av) // 2
    return a[u0:u0 + au, v0:v0 + av, :hc, :wc]


_U8_TO_UNIT = {}


def _unit(x8: torch.Tensor) -> torch.Tensor:
    """uint8 -> fp64 k / 255.0, exactly numpy's astype('double') / 255.0: a 256-entry table of correctly rounded quotients
    (a division by a scalar in torch may become a multiplication by its reciprocal)."""
    lut = _U8_TO_UNIT.get(x8.device)
    if lut is None:
        lut = _U8_TO_UNIT[x8.device] = torch.from_numpy(np.arange(256, dtype=np.float64) / 255.0).to(x8.device)
    return lut.index_select(0, x8.reshape(-1).to(torch.int32)).view(x8.shape)


def prepare_views(rgb8, angRes, scale: int, kind: str = "hr"):
    """RGB views of one scene -> (Lr_SAI_y, Hr_SAI_y or None, Sr_SAI_cbcr) as fp32 mosaics on the current CUDA device,
    by the recipe of include/lfsr.h. rgb8: host uint8 [U, V, H, W, 3]; angRes: the central angRes x angRes views, or the
    central a1 x a2 for a pair (a1, a2). kind="hr": the views are ground truth (test.py),
    the LR input is their bicubic x1/scale; kind="lr": the views are the LR input (inference.py) and there is no HR.
    The cropped central views cross PCIe once (3 bytes per pixel, from pinned memory); the rest runs on the device."""
    if kind not in ("hr", "lr"):
        raise ValueError(f"kind must be 'hr' or 'lr', got {kind!r}")
    a = np.asarray(rgb8)
    if a.dtype != np.uint8:
        raise ValueError(f"prepare_views takes uint8 views, got {a.dtype}")
    if not torch.cuda.is_available():
        raise N.LfsrError("lfsr_b200 needs a CUDA device (sm_100a); there is no CPU fallback for this path")
    dev = torch.device("cuda", torch.cuda.current_device())
    crop = central_views(a, angRes, scale)
    host = torch.empty(crop.shape, dtype=torch.uint8, pin_memory=True)
    host.numpy()[...] = crop
    x8 = host.to(dev, non_blocking=True)
    A = angRes
    if kind == "hr":
        hr_y, _ = rgb_to_ycbcr_mosaic(x8, A, cbcr=False)
        lr_rgb = imresize_views(_unit(x8), 1.0 / scale)
        lr_y, _ = rgb_to_ycbcr_mosaic(lr_rgb, A, cbcr=False)
    else:
        hr_y, lr_rgb = None, _unit(x8)
        lr_y, _ = rgb_to_ycbcr_mosaic(x8, A, cbcr=False)
    _, sr_cbcr = rgb_to_ycbcr_mosaic(imresize_views(lr_rgb, float(scale)), A, y=False)
    return lr_y, hr_y, sr_cbcr


def write_bmp(path, img) -> None:
    """[h, w, 3] uint8 RGB -> 24-bit uncompressed BMP, byte-identical to what imageio.imwrite (Pillow's BmpImagePlugin)
    produces for such an array: 14-byte file header, 40-byte BITMAPINFOHEADER (96 dpi = 3780 px/m), bottom-up BGR rows
    padded to 4 bytes."""
    import struct
    a = np.ascontiguousarray(img.cpu().numpy() if torch.is_tensor(img) else img)
    if a.ndim != 3 or a.shape[2] != 3 or a.dtype != np.uint8:
        raise ValueError(f"expected [h, w, 3] uint8, got {a.shape} {a.dtype}")
    h, w, _ = a.shape
    stride = (w * 3 + 3) & ~3
    rows = np.zeros((h, stride), dtype=np.uint8)
    rows[:, : w * 3] = a[::-1, :, ::-1].reshape(h, w * 3)
    image = h * stride
    with open(path, "wb") as f:
        f.write(b"BM" + struct.pack("<IHHI", 14 + 40 + image, 0, 0, 14 + 40))
        f.write(struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, 0, image, 3780, 3780, 0, 0))
        f.write(rows.tobytes())
