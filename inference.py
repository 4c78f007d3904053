"""`python inference.py --model_name M --angRes 5 --scale_factor 4 --path_pre_pth X --path_for_test D
--data_name N` - the reference's inference entry point (inference.py:93-228): test.py without
metrics; writes View_i_j.bmp per scene. The reference's fvcore FLOP probe (:117-124) is optional
there (wrapped in try/except) and is not reproduced."""
import importlib

import torch

from utils.utils import create_dir
from utils.utils_datasets import MultiTestSetDataLoader
from lfsr_b200 import scene as _scene
from test import load_checkpoint
from train import _write_views


def main(args):
    _, _, result_dir = create_dir(args)
    result_dir = result_dir.joinpath("TEST")
    result_dir.mkdir(exist_ok=True)
    device = torch.device(args.device)
    if "cuda" in args.device:
        torch.cuda.set_device(device)
    test_names, test_loaders, n_scenes = MultiTestSetDataLoader(args)
    print("The number of test data is: %d" % n_scenes)
    MODEL = importlib.import_module("model." + args.task + "." + args.model_name)
    net = MODEL.get_model(args)
    if args.use_pre_ckpt == False:  # noqa: E712
        net.apply(MODEL.weights_init)
    else:
        load_checkpoint(net, args.path_pre_pth)
    net = net.to(device).eval()
    with torch.no_grad():
        for name, loader in zip(test_names, test_loaders):
            save_dir = result_dir.joinpath(name)
            save_dir.mkdir(exist_ok=True)
            for Lr_SAI_y, _hr, cbcr, data_info, lf_name in loader:
                ang = int(data_info[0][0].item())
                sr = _scene.super_resolve_scene(net, Lr_SAI_y.squeeze().to(device), ang, args.scale_factor,
                                                args.patch_size_for_test, args.stride_for_test, args.minibatch,
                                                self_ensemble=bool(getattr(args, "self_ensemble", 0)))
                _write_views(save_dir, lf_name[0], sr, cbcr, args.angRes_out)
                print("scene %s -> %s" % (lf_name[0], save_dir))


if __name__ == "__main__":
    from option import args
    main(args)
