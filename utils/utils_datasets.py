"""Test-set loaders for the entry points (the reference's utils/utils_datasets.py:61-136 on the
inference path). Disk I/O is outside the accelerated path (SURVEY 2 #12): this module only has to
yield the same 5-tuples `(Lr_SAI_y[1,1,AH,AW], Hr_SAI_y, Sr_SAI_cbcr, [angRes_in, angRes_out], [name])`
the reference's DataLoader(batch_size=1) yields. Three sources, chosen by MultiTestSetDataLoader:
- `--synthetic N`: seeded scenes, so the whole entry point can run without any dataset;
- h5 files under <path_for_test>/SR_AxA_sx/<data_name>/ (BasicLFSR's prepared test sets; needs h5py);
- light fields stored as view images, <path_for_test>/<data_name>/<scene>/View_u_v.{png,bmp} with 0-based u, v (the
  layout inference.py writes). They are decoded with Pillow on the host and prepared on the GPU
  (lfsr_b200.lfutils.prepare_views: central A x A views, crop, rgb2ycbcr, bicubic LR / SR colour), so no offline
  generator step is needed: test.py reads them as ground truth, inference.py as LR input."""
import os
import re

import numpy as np
import torch


def _batch1(lr, hr, cbcr, ang_in, ang_out, name, grid=None):
    """grid: the N of a full-grid scene (--full_grid 1), carried as a third data_info entry next to the window size, or
    its (N_u, N_v) (--grid_views), carried as a third and a fourth"""
    grid = [] if grid is None else list(grid) if isinstance(grid, (tuple, list)) else [grid]
    info = [torch.tensor([ang_in]), torch.tensor([ang_out])] + [torch.tensor([g]) for g in grid]
    return (lr[None], hr[None], cbcr[None], info, [name])


class SyntheticTestSet:
    def __init__(self, args, n, size):
        self.args, self.n, self.size = args, n, size

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if not 0 <= i < self.n:
            raise IndexError(i)
        A, s, h = self.args.angRes_in, self.args.scale_factor, self.size
        rs = np.random.RandomState(1000 + i)
        lr = torch.from_numpy(rs.random_sample((1, A * h, A * h)).astype(np.float32))
        hr = torch.from_numpy(rs.random_sample((1, A * h * s, A * h * s)).astype(np.float32))
        cbcr = torch.full((2, A * h * s, A * h * s), 0.5)
        return _batch1(lr, hr, cbcr, A, self.args.angRes_out, "synthetic_%02d" % i)

    def __iter__(self):
        for i in range(self.n):
            yield self[i]


class H5TestSet:
    """one dataset directory <path_for_test>/SR_AxA_sx/<data_name>/*.h5 (utils_datasets.py:87-136)."""

    def __init__(self, args, data_name):
        try:
            import h5py  # noqa: F401
        except ImportError as e:
            raise RuntimeError("reading .h5 test sets needs h5py, which is not installed; use --synthetic N") from e
        self.args = args
        self.root = os.path.join(args.path_for_test, "SR_%dx%d_%dx" % (args.angRes_in, args.angRes_in, args.scale_factor),
                                 data_name)
        self.files = sorted(os.listdir(self.root))

    def __len__(self):
        return len(self.files)

    def __getitem__(self, i):
        """reads only the i-th file (a rank of a multi-GPU run opens just the scenes it runs)"""
        import h5py
        fn = self.files[i]
        with h5py.File(os.path.join(self.root, fn), "r") as hf:
            lr = np.array(hf.get("Lr_SAI_y")).T
            hr = np.array(hf.get("Hr_SAI_y")).T
            cb = np.array(hf.get("Sr_SAI_cbcr"), dtype="single")
        if cb.ndim == 3:
            cb = np.transpose(cb, (2, 1, 0))
        elif cb.ndim == 0 or cb.size == 0:
            cb = np.zeros((hr.shape[0], hr.shape[1], 2), np.float32)
        elif cb.ndim == 2:
            cb = cb[..., None]
        to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
        return _batch1(to_t(lr)[None], to_t(hr)[None], to_t(cb).permute(2, 0, 1).contiguous(), self.args.angRes_in,
                       self.args.angRes_out, fn.split(".")[0])

    def __iter__(self):
        for i in range(len(self.files)):
            yield self[i]


_VIEW_FILE = re.compile(r"View_(\d+)_(\d+)\.(png|bmp)$", re.IGNORECASE)


def _scene_dirs(path):
    """sub-directories of `path` that hold at least one View_u_v image, sorted by name."""
    if not os.path.isdir(path):
        return []
    out = []
    for d in sorted(os.listdir(path)):
        full = os.path.join(path, d)
        if os.path.isdir(full) and any(_VIEW_FILE.match(f) for f in os.listdir(full)):
            out.append(d)
    return out


def _check_rgb8(im, fn):
    """8-bit RGB only: Pillow also opens 48-bit PNGs as mode RGB, so look at the raw mode of the encoded data too."""
    if im.mode != "RGB":
        raise ValueError(f"{fn}: mode {im.mode} is not supported (8-bit RGB views only)")
    for tile in getattr(im, "tile", None) or []:
        args = tile[3] if len(tile) > 3 else None
        raw = args[0] if isinstance(args, tuple) and args else args
        if isinstance(raw, str) and (";16" in raw or ";15" in raw):
            raise ValueError(f"{fn}: 16-bit samples are not supported (8-bit RGB views only)")


def parse_grid_views(value, full_grid):
    """--grid_views -> None ('' : the central N x N, N = min(U, V)), "all" (the whole U x V grid) or (R, C) (the central
    R x C views, from "RxC"). Valid only with --full_grid 1. Raises ValueError naming the flag."""
    value = (value or "").strip()
    if not value:
        return None
    if not full_grid:
        raise ValueError(f"--grid_views {value!r} needs --full_grid 1")
    if value == "all":
        return "all"
    m = re.fullmatch(r"(\d+)x(\d+)", value)
    if not m or int(m.group(1)) < 1 or int(m.group(2)) < 1:
        raise ValueError(f"--grid_views {value!r}: expected '', 'all' or RxC with positive integers R and C (e.g. 9x13)")
    return int(m.group(1)), int(m.group(2))


def read_views(scene_dir, ang, full_grid=False, grid=None):
    """the central ang x ang views of one scene folder of View_u_v.{png,bmp} images -> uint8 [ang, ang, H, W, 3]; with
    full_grid, the central N x N views with N = min(U, V) of the U x V grid -> uint8 [N, N, H, W, 3] (angular window
    tiling, include/lfsr.h), or with grid = "all" the whole grid [U, V, H, W, 3] and with grid = (R, C) the central R x C
    views [R, C, H, W, 3] (--grid_views; A <= R <= U and A <= C <= V). Every view of the grid must be present, 8-bit RGB
    and of one size (headers only are read for the views outside the centre); only the chosen views are decoded. Raises
    ValueError naming the file and the problem."""
    from PIL import Image
    files = {}
    for f in sorted(os.listdir(scene_dir)):
        m = _VIEW_FILE.match(f)
        if m:
            key = (int(m.group(1)), int(m.group(2)))
            if key in files:
                raise ValueError(f"{os.path.join(scene_dir, f)}: view {key} is stored twice "
                                 f"(also {os.path.basename(files[key])})")
            files[key] = os.path.join(scene_dir, f)
    if not files:
        raise ValueError(f"{scene_dir}: no View_u_v.png or View_u_v.bmp images")
    U = max(u for u, _ in files) + 1
    V = max(v for _, v in files) + 1
    for u in range(U):
        for v in range(V):
            if (u, v) not in files:
                raise ValueError(f"{os.path.join(scene_dir, 'View_%d_%d.png|bmp' % (u, v))}: view is missing "
                                 f"from the {U}x{V} grid")
    if U < ang or V < ang:
        raise ValueError(f"{scene_dir}: a {U}x{V} grid of views is smaller than angRes {ang}x{ang}")
    if grid is not None and not full_grid:
        raise ValueError("--grid_views needs --full_grid 1")
    if grid is None:
        nu = nv = min(U, V) if full_grid else ang
    elif grid == "all":
        nu, nv = U, V
    else:
        nu, nv = (int(g) for g in grid)
        if not (ang <= nu <= U and ang <= nv <= V):
            raise ValueError(f"{scene_dir}: --grid_views {nu}x{nv} is not a sub-grid of the {U}x{V} grid of views of at "
                             f"least angRes {ang}x{ang}")
    size = None
    for (u, v), fn in sorted(files.items()):
        with Image.open(fn) as im:
            _check_rgb8(im, fn)
            if size is None:
                size, first = im.size, fn
            elif im.size != size:
                raise ValueError(f"{fn}: view is {im.size[0]}x{im.size[1]} (WxH) but {first} is {size[0]}x{size[1]}")
    u0, v0 = (U - nu) // 2, (V - nv) // 2
    out = np.empty((nu, nv, size[1], size[0], 3), dtype=np.uint8)
    for i in range(nu):
        for j in range(nv):
            with Image.open(files[(u0 + i, v0 + j)]) as im:
                out[i, j] = np.asarray(im)
    return out


def prepare_views(rgb8, ang, scale, kind):
    """the device preparation (a module attribute, so that tests on machines without a GPU can substitute the oracle)."""
    from lfsr_b200 import lfutils
    return lfutils.prepare_views(rgb8, ang, scale, kind)


class ViewsTestSet:
    """one dataset directory <path_for_test>/<data_name>/ of scene folders of View_u_v.{png,bmp} images. kind="hr":
    the views are ground truth (test.py: LR input = their bicubic x1/s); kind="lr": the views are the LR input
    (inference.py; Hr_SAI_y is an empty tensor). Yields the batch-1 5-tuple with the tensors on the current CUDA device;
    __getitem__ decodes only the scene asked for. full_grid: every view of the central N x N (N = min(U, V)) instead of
    the central A x A, for angular window tiling (scene.test_grid / super_resolve_grid); data_info is then
    [A, A, N]. grid ("all" or (R, C), parse_grid_views; full_grid only): the whole grid or its central R x C views
    instead, and data_info [A, A, N_u, N_v]."""

    def __init__(self, args, data_name, kind, full_grid=False, grid=None):
        if kind not in ("hr", "lr"):
            raise ValueError(f"kind must be 'hr' or 'lr', got {kind!r}")
        if grid is not None and not full_grid:
            raise ValueError("--grid_views needs --full_grid 1")
        self.args, self.kind, self.full_grid, self.grid = args, kind, bool(full_grid), grid
        self.root = os.path.join(args.path_for_test, data_name)
        self.scenes = _scene_dirs(self.root)

    def __len__(self):
        return len(self.scenes)

    def __getitem__(self, i):
        if not 0 <= i < len(self.scenes):
            raise IndexError(i)
        A, s = self.args.angRes_in, self.args.scale_factor
        if self.grid is not None:
            rgb8 = read_views(os.path.join(self.root, self.scenes[i]), A, full_grid=True, grid=self.grid)
            n = tuple(rgb8.shape[:2])
        elif self.full_grid:
            rgb8 = read_views(os.path.join(self.root, self.scenes[i]), A, full_grid=True)
            n = rgb8.shape[0]
        else:
            rgb8 = read_views(os.path.join(self.root, self.scenes[i]), A)
            n = A
        lr, hr, cbcr = prepare_views(rgb8, n, s, self.kind)
        if hr is None:
            hr = lr.new_empty((0, 0))
        return _batch1(lr[None], hr[None], cbcr, A, self.args.angRes_out, self.scenes[i],
                       n if self.full_grid else None)

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]


def MultiTestSetDataLoader(args, views=None):
    """(dataset names, loaders, total scenes). --synthetic N wins; then BasicLFSR's h5 layout
    <path_for_test>/SR_AxA_sx/<data_name>/*.h5 if that directory exists (or `views` is None); otherwise light fields
    stored as view images, <path_for_test>/<data_name>/<scene>/View_u_v.{png,bmp}, read as `views` = "hr" (ground
    truth, test.py) or "lr" (LR input, inference.py). --full_grid 1 (every view, angular window tiling) needs the view
    layout: synthetic scenes and h5 files hold only A x A views, so it raises ValueError with them. --grid_views (the
    whole grid or a central R x C of it, parse_grid_views) raises ValueError without --full_grid 1 or when malformed."""
    full_grid = bool(getattr(args, "full_grid", 0))
    grid = parse_grid_views(getattr(args, "grid_views", ""), full_grid)
    if full_grid and getattr(args, "synthetic", 0) > 0:
        raise ValueError("--full_grid 1 needs light fields stored as view images: --synthetic scenes have only "
                         f"{args.angRes_in}x{args.angRes_in} views")
    if getattr(args, "synthetic", 0) > 0:
        ds = SyntheticTestSet(args, args.synthetic, args.synthetic_size)
        return ["Synthetic"], [ds], len(ds)
    base = os.path.join(args.path_for_test, "SR_%dx%d_%dx" % (args.angRes_in, args.angRes_in, args.scale_factor))
    if views is None or os.path.isdir(base):
        if full_grid:
            raise ValueError(f"--full_grid 1 needs light fields stored as view images: the h5 test sets in {base} hold "
                             f"only {args.angRes_in}x{args.angRes_in} views")
        names = sorted(os.listdir(base)) if args.data_name == "ALL" else [args.data_name]
        loaders = [H5TestSet(args, n) for n in names]
        return names, loaders, sum(len(d) for d in loaders)
    root = args.path_for_test
    if args.data_name == "ALL":
        names = [d for d in sorted(os.listdir(root)) if _scene_dirs(os.path.join(root, d))] if os.path.isdir(root) else []
    else:
        names = [args.data_name]
    loaders = [ViewsTestSet(args, n, views, full_grid, grid) for n in names]
    n_scenes = sum(len(d) for d in loaders)
    if n_scenes == 0:
        raise FileNotFoundError(
            f"no test data under {root}: expected either h5 files in {base}/<data_name>/ or scene folders of "
            f"View_u_v.png|bmp images in {os.path.join(root, '<data_name>')}/<scene>/ (data_name {args.data_name})")
    return names, loaders, n_scenes
