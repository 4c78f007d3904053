"""Inference half of the reference's train.py: only `test()` (train.py:286-347), which test.py
imports (`from train import test`). Training (train.py:20-282) is outside this repository's scope.

`test()` keeps the reference's signature and return value but runs the patch loop on the device:
LFdivide -> batched forward (args.minibatch patches per call instead of minibatch_for_test = 1 with
a host round trip per patch) -> LFintegrate -> PSNR/SSIM -> YCbCr->RGB uint8 views, all on liblfsr_b200
kernels; one D2H copy of the uint8 views per scene feeds the BMP writer.

With torch.distributed initialised (test.py / inference.py under torchrun), a dataset is split across the ranks by
`scene.assign_scenes`: full rounds of scenes run one per rank, the remaining scenes are row-sharded over all ranks.

With --full_grid 1 every scene is the central N x N of a larger light field (data_info [A, A, N]), or with --grid_views
its whole U x V grid or central R x C (data_info [A, A, N_u, N_v]); it runs through `scene.test_grid`: overlapping A x A
windows (A = args.angRes_in), averaged where they overlap, N_u * N_v views written. With --save_layout mosaic|lenslet
each scene is written as one <scene>.bmp of its whole SR grid instead of View_i_j.bmp files."""
import torch

from lfsr_b200 import scene as _scene
from lfsr_b200 import lfutils as _lfutils


def _write_views(save_dir, name, sr_sai_y, cbcr, ang, layout="views"):
    """Colour tail of the reference's test() (train.py:329-341): cat(Y, CbCr) -> ycbcr2rgb -> clip*255 -> uint8 -> one
    View_i_j.bmp per view. The conversion runs on the device (lfsr_ycbcr_to_rgb8, bit-exact to the reference's fp64 numpy
    arithmetic) so only 1 byte per channel crosses PCIe; the BMP files are byte-identical to imageio.imwrite's.
    ang: an ang x ang grid of views, or (N_u, N_v) for N_u x N_v (i < N_u, j < N_v). layout (--save_layout) "mosaic" or
    "lenslet": one <save_dir>/<name>.bmp of the whole grid in that layout instead (include/lfsr.h, "Image light fields")."""
    if layout != "views":
        rows, cols = sr_sai_y.shape[-2:]
        if _lfutils.bmp_bytes(rows, cols) >= 1 << 32:
            raise ValueError(f"--save_layout {layout}: the {cols}x{rows} (WxH) image of scene {name} does not fit a BMP "
                             "file (4 GiB at most); use --save_layout views")
        _lfutils.write_bmp(str(save_dir.joinpath(name + ".bmp")),
                           _lfutils.sai_to_rgb8(sr_sai_y, cbcr, ang, layout).cpu().numpy())
        return
    d = save_dir.joinpath(name)
    d.mkdir(exist_ok=True)
    views = _lfutils.sai_to_rgb8_views(sr_sai_y, cbcr, ang).cpu().numpy()
    for i in range(views.shape[0]):
        for j in range(views.shape[1]):
            _lfutils.write_bmp(str(d) + "/View_%d_%d.bmp" % (i, j), views[i, j])


def dist_world():
    """(world, rank) of the default process group, (1, 0) without one."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def rank_scenes(loader, world, rank):
    """Yields (index, solo, owner, batch) for the scenes this rank runs, in dataset order. solo: a full-round scene this
    rank runs alone (pass world=1, rank=0 to the scene driver); otherwise a tail scene that every rank runs row-sharded.
    owner: this rank keeps the scene's result and writes its files. Loaders with __getitem__ read only these scenes; a
    loader that can only iterate is enumerated and filtered by index. With world > 1 every rank must call this for the
    same dataset: the ranks first agree on its length, since the tail's all-gathers need every rank."""
    if world == 1:
        for i, batch in enumerate(loader):
            yield i, True, True, batch
        return
    import torch.distributed as dist
    n = len(loader)
    counts = [None] * world
    dist.all_gather_object(counts, n)
    if len(set(counts)) != 1:
        raise RuntimeError(f"ranks disagree on the number of scenes of the dataset: {counts}")
    own, tail = _scene.assign_scenes(n, world, rank)
    mine = own + tail
    if hasattr(loader, "__getitem__"):
        items = ((i, loader[i]) for i in mine)
    else:
        keep = set(mine)
        items = ((i, b) for i, b in enumerate(loader) if i in keep)
    n_own = len(own)
    for k, (i, batch) in enumerate(items):
        solo = k < n_own
        yield i, solo, solo or i % world == rank, batch


def gather_in_order(rows, world):
    """every rank's (index, ...) rows, merged in index order on every rank."""
    if world == 1:
        return rows
    import torch.distributed as dist
    parts = [None] * world
    dist.all_gather_object(parts, rows)
    return sorted((r for p in parts for r in p), key=lambda r: r[0])


def grid_size(data_info):
    """(N_u, N_v) of a full-grid scene: data_info [A, A, N] (utils_datasets.ViewsTestSet with full_grid: N_u = N_v = N)
    or [A, A, N_u, N_v] (with --grid_views)."""
    if len(data_info) < 3:
        raise ValueError("--full_grid 1: the loader did not report the grid size of the scene")
    n = [int(x[0].item()) if torch.is_tensor(x) else int(x) for x in data_info[2:4]]
    return (n[0], n[0]) if len(n) == 1 else (n[0], n[1])


def test(test_loader, device, net, args, save_dir=None):
    net.eval()
    world, rank = dist_world()
    full_grid = bool(getattr(args, "full_grid", 0))
    rows = []
    for i, solo, owner, (Lr_SAI_y, Hr_SAI_y, Sr_SAI_cbcr, data_info, LF_name) in rank_scenes(test_loader, world, rank):
        ang = int(data_info[0][0].item()) if torch.is_tensor(data_info[0]) else int(data_info[0])
        # host tensors go in as they are: the scene driver stages them through pinned buffers on its copy stream
        lr, hr = Lr_SAI_y.squeeze(), Hr_SAI_y.squeeze()
        shard = dict(world=1, rank=0) if solo else {}
        with torch.no_grad():
            if full_grid:
                views = grid_size(data_info)
                psnr, ssim, sr = _scene.test_grid(net, lr, hr, views, args.angRes_in, args.scale_factor,
                                                  args.patch_size_for_test, args.stride_for_test,
                                                  getattr(args, "minibatch", 64),
                                                  ang_stride=getattr(args, "ang_stride", 0) or None,
                                                  self_ensemble=bool(getattr(args, "self_ensemble", 0)), **shard)
            else:
                views = args.angRes_out
                psnr, ssim, sr = _scene.test_scene(net, lr, hr, ang, args.scale_factor, args.patch_size_for_test,
                                                   args.stride_for_test, getattr(args, "minibatch", 64),
                                                   self_ensemble=bool(getattr(args, "self_ensemble", 0)), **shard)
        if owner:
            rows.append((i, psnr, ssim, LF_name[0]))
            if save_dir is not None:
                _write_views(save_dir, LF_name[0], sr, Sr_SAI_cbcr, views, getattr(args, "save_layout", "views"))
    rows = gather_in_order(rows, world)
    return [r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows]
