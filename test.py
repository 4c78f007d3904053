"""`python test.py --model_name M --angRes 5 --scale_factor 4 [--use_pre_ckpt '' | --path_pre_pth X]`
- the reference's evaluation entry point (test.py:10-101) on the B200-native path: same flags, same
plugin discovery (model.SR.<name>.get_model), same checkpoint convention ('module.'-prefixed keys
first, plain keys second), same result layout log/SR_AxA_sx/<data>/<model>/results/TEST/.

Under torchrun (WORLD_SIZE > 1, one process per GPU) each dataset is split across the ranks (train.test): the results
and files are the ones a single-GPU run gives, and only rank 0 prints and writes evaluation.xls."""
import importlib
import os
from collections import OrderedDict

import numpy as np
import torch
import torch.distributed as dist

from utils.utils import ExcelFile, create_dir
from utils.utils_datasets import MultiTestSetDataLoader
from train import test


def load_checkpoint(net, path):
    ckpt = torch.load(path, map_location="cpu")
    sd = ckpt["state_dict"] if "state_dict" in ckpt else ckpt
    for prefix in ("module.", ""):
        try:
            net.load_state_dict(OrderedDict((prefix + k, v) for k, v in sd.items()))
            return
        except RuntimeError:
            continue
    net.load_state_dict(OrderedDict((k[len("module."):] if k.startswith("module.") else k, v) for k, v in sd.items()))


def init_distributed(args):
    """(device, rank). Under torchrun (WORLD_SIZE > 1): cuda:$LOCAL_RANK and an NCCL process group bound to it, which
    train.test / inference.py split each dataset over. Otherwise --device and no group."""
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        device = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=device)
        return device, dist.get_rank()
    device = torch.device(args.device)
    if "cuda" in args.device:
        torch.cuda.set_device(device)
    return device, 0


def broadcast_weights(net):
    """every parameter and buffer from rank 0, so that all ranks run the same network whatever initialised it."""
    if dist.is_initialized():
        with torch.no_grad():
            for t in list(net.parameters()) + list(net.buffers()):
                dist.broadcast(t, 0)


def finish_distributed():
    if dist.is_initialized():
        dist.destroy_process_group()


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
    test_names, test_loaders, n_scenes = MultiTestSetDataLoader(args)
    log("The number of test data is: %d" % n_scenes)
    MODEL = importlib.import_module("model." + args.task + "." + args.model_name)
    net = MODEL.get_model(args)
    if args.use_pre_ckpt == False:  # noqa: E712  (type=bool flag: only '' is False)
        net.apply(MODEL.weights_init)
    else:
        load_checkpoint(net, args.path_pre_pth)
        log("Use pretrain model!")
    net = net.to(device)
    broadcast_weights(net)
    log(args)
    excel = ExcelFile()
    psnr_sets, ssim_sets = [], []
    with torch.no_grad():
        for name, loader in zip(test_names, test_loaders):
            save_dir = result_dir.joinpath(name)
            save_dir.mkdir(exist_ok=True)
            psnr, ssim, lf_names = test(loader, device, net, args, save_dir)
            excel.write_sheet(name, lf_names, psnr, ssim)
            psnr_sets.append(float(np.mean(psnr)))
            ssim_sets.append(float(np.mean(ssim)))
            log("Test on %s, psnr/ssim is %.3f/%.4f" % (name, psnr_sets[-1], ssim_sets[-1]))
    excel.add_sheet("ALL", "Average", float(np.mean(psnr_sets)), float(np.mean(ssim_sets)))
    log("The mean psnr on testsets is %.5f, mean ssim is %.5f" % (np.mean(psnr_sets), np.mean(ssim_sets)))
    if rank == 0:
        excel.xlsx_file.save(str(result_dir) + "/evaluation.xls")


if __name__ == "__main__":
    from option import args
    main(args)
