"""`python inference.py --model_name M --angRes 5 --scale_factor 4 --path_pre_pth X --path_for_test D
--data_name N` - the reference's inference entry point (inference.py:93-228): test.py without
metrics; writes View_i_j.bmp per scene. The reference's fvcore FLOP probe (:117-124) is optional
there (wrapped in try/except) and is not reproduced.

Under torchrun (WORLD_SIZE > 1) each dataset is split across the ranks like test.py's (train.rank_scenes); every
View_i_j.bmp is written once, by the rank that owns its scene, and only rank 0 prints. With --full_grid 1 every view of
the central N x N of each light field (with --grid_views: the whole U x V grid, or its central R x C) is super-resolved
with overlapping angRes x angRes windows (scene.super_resolve_grid) and N_u * N_v View_i_j.bmp are written. Light
fields stored as one mosaic or lenslet image each are read with --input_layout mosaic|lenslet --input_grid UxV; with
--save_layout mosaic|lenslet each scene's SR grid is written as one <scene>.bmp in that layout."""
import importlib

import torch

from utils.utils import create_dir
from utils.utils_datasets import MultiTestSetDataLoader
from lfsr_b200 import scene as _scene
from test import broadcast_weights, finish_distributed, init_distributed, load_checkpoint
from train import _write_views, dist_world, gather_in_order, grid_size, rank_scenes


def main(args):
    device, rank = init_distributed(args)
    try:
        run(args, device, rank)
    finally:
        finish_distributed()


def run(args, device, rank):
    log = print if rank == 0 else (lambda *a: None)
    _, _, result_dir = create_dir(args)
    result_dir = result_dir.joinpath("TEST")
    result_dir.mkdir(exist_ok=True)
    test_names, test_loaders, n_scenes = MultiTestSetDataLoader(args, views="lr")
    log("The number of test data is: %d" % n_scenes)
    MODEL = importlib.import_module("model." + args.task + "." + args.model_name)
    net = MODEL.get_model(args)
    if args.use_pre_ckpt == False:  # noqa: E712
        net.apply(MODEL.weights_init)
    else:
        load_checkpoint(net, args.path_pre_pth)
    net = net.to(device).eval()
    broadcast_weights(net)
    world, _ = dist_world()
    full_grid = bool(getattr(args, "full_grid", 0))
    with torch.no_grad():
        for name, loader in zip(test_names, test_loaders):
            save_dir = result_dir.joinpath(name)
            save_dir.mkdir(exist_ok=True)
            written = []
            for i, solo, owner, (Lr_SAI_y, _hr, cbcr, data_info, lf_name) in rank_scenes(loader, world, rank):
                ang = int(data_info[0][0].item())
                shard = dict(world=1, rank=0) if solo else {}
                if full_grid:
                    views = grid_size(data_info)
                    sr = _scene.super_resolve_grid(net, Lr_SAI_y.squeeze().to(device), views, args.angRes_in,
                                                   args.scale_factor, args.patch_size_for_test, args.stride_for_test,
                                                   args.minibatch, ang_stride=getattr(args, "ang_stride", 0) or None,
                                                   self_ensemble=bool(getattr(args, "self_ensemble", 0)), **shard)
                else:
                    views = args.angRes_out
                    sr = _scene.super_resolve_scene(net, Lr_SAI_y.squeeze().to(device), ang, args.scale_factor,
                                                    args.patch_size_for_test, args.stride_for_test, args.minibatch,
                                                    self_ensemble=bool(getattr(args, "self_ensemble", 0)), **shard)
                if owner:
                    _write_views(save_dir, lf_name[0], sr, cbcr, views, getattr(args, "save_layout", "views"))
                    written.append((i, lf_name[0]))
                    if world == 1:
                        print("scene %s -> %s" % (lf_name[0], save_dir))
            if world > 1:
                for _, n in gather_in_order(written, world):
                    log("scene %s -> %s" % (n, save_dir))


if __name__ == "__main__":
    from option import args
    main(args)
