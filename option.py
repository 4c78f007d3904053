"""Command-line options of the inference entry points; flag names, types and defaults follow the
reference's option.py:4-34 (including its `type=bool` quirk: any non-empty string is True, so the
random-init path needs --use_pre_ckpt ''), parsed at import time like the reference because
utils/utils.py and the entry points do `from option import args`.
Additive flags (not in the reference): --synthetic, --synthetic_size, --minibatch, --self_ensemble, --full_grid,
--ang_stride, --grid_views, --input_layout, --input_grid, --save_layout."""
import argparse

_FLAGS = [
    # name, kwargs
    ("--task", dict(type=str, default="SR", help="SR (RE is outside the accelerated path)")),
    ("--angRes", dict(type=int, default=5, help="angular resolution")),
    ("--scale_factor", dict(type=int, default=2, help="4, 2")),
    ("--model_name", dict(type=str, default="LFT", help="model name (model/SR/<name>.py)")),
    ("--use_pre_ckpt", dict(type=bool, default=True, help="load --path_pre_pth; '' = random init")),
    ("--path_pre_pth", dict(type=str, default="./pth/", help="checkpoint path")),
    ("--data_name", dict(type=str, default="ALL", help="EPFL, HCI_new, HCI_old, INRIA_Lytro, Stanford_Gantry, ALL")),
    ("--path_for_train", dict(type=str, default="./data_for_training/")),
    ("--path_for_test", dict(type=str, default="./data_for_test/")),
    ("--path_log", dict(type=str, default="./log/")),
    ("--batch_size", dict(type=int, default=4)),
    ("--lr", dict(type=float, default=2e-4)),
    ("--decay_rate", dict(type=float, default=0)),
    ("--n_steps", dict(type=int, default=15)),
    ("--gamma", dict(type=float, default=0.5)),
    ("--epoch", dict(type=int, default=51)),
    ("--device", dict(type=str, default="cuda:0")),
    ("--num_workers", dict(type=int, default=2)),
    ("--local_rank", dict(dest="local_rank", type=int, default=0)),
    ("--use_masked_pretrain", dict(type=bool, default=True)),
    ("--mask_ratio", dict(type=float, default=0.3)),
    # additive
    ("--synthetic", dict(type=int, default=0, help="run on N seeded synthetic scenes instead of h5 files")),
    ("--synthetic_size", dict(type=int, default=64, help="view height/width of the synthetic LR scenes")),
    ("--minibatch", dict(type=int, default=64, help="patches per forward on the device path")),
    ("--self_ensemble", dict(type=int, default=0, help="1: x8 flip/transpose self-ensemble per patch (8x the forwards)")),
    ("--full_grid", dict(type=int, default=0, help="1: super-resolve every view of the central N x N (N = min(U, V)) of "
                         "view-image light fields with overlapping angRes x angRes windows, averaged where they overlap")),
    ("--ang_stride", dict(type=int, default=0, help="angular stride of the --full_grid windows, 1..angRes-1 "
                          "(0: angRes - 1, the fewest windows)")),
    ("--grid_views", dict(type=str, default="", help="with --full_grid 1: which views to super-resolve; '' the central "
                          "N x N (N = min(U, V)), 'all' the whole U x V grid, RxC (e.g. 9x13) the central R x C")),
    ("--input_layout", dict(type=str, default="views", choices=["views", "mosaic", "lenslet"],
                            help="how the test light fields are stored: views = <scene>/View_u_v.png|bmp folders, "
                            "mosaic = one sub-aperture image array <scene>.png|bmp, lenslet = one macro-pixel image")),
    ("--input_grid", dict(type=str, default="", help="UxV views of each mosaic / lenslet image (e.g. 14x14); "
                          "required with --input_layout mosaic|lenslet")),
    ("--save_layout", dict(type=str, default="views", choices=["views", "mosaic", "lenslet"],
                           help="how SR results are written: views = <scene>/View_u_v.bmp, mosaic / lenslet = one "
                           "<scene>.bmp of the whole SR grid")),
]

parser = argparse.ArgumentParser()
for _name, _kw in _FLAGS:
    parser.add_argument(_name, **_kw)
args = parser.parse_args()

if args.task == "SR":
    args.angRes_in = args.angRes
    args.angRes_out = args.angRes
    args.patch_size_for_test = 32
    args.stride_for_test = 16
    args.minibatch_for_test = 1      # reference value; the device driver batches args.minibatch patches itself
del args.angRes
