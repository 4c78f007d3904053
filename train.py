"""Inference half of the reference's train.py: only `test()` (train.py:286-347), which test.py
imports (`from train import test`). Training (train.py:20-282) is outside this repository's scope.

`test()` keeps the reference's signature and return value but runs the patch loop on the device:
LFdivide -> batched forward (args.minibatch patches per call instead of minibatch_for_test = 1 with
a host round trip per patch) -> LFintegrate -> PSNR/SSIM -> YCbCr->RGB uint8 views, all on liblfsr_b200
kernels; one D2H copy of the uint8 views per scene feeds the BMP writer."""
import torch

from lfsr_b200 import scene as _scene
from lfsr_b200 import lfutils as _lfutils


def _write_views(save_dir, name, sr_sai_y, cbcr, ang):
    """Colour tail of the reference's test() (train.py:329-341): cat(Y, CbCr) -> ycbcr2rgb -> clip*255 -> uint8 -> one
    View_i_j.bmp per view. The conversion runs on the device (lfsr_ycbcr_to_rgb8, bit-exact to the reference's fp64 numpy
    arithmetic) so only 1 byte per channel crosses PCIe; the BMP files are byte-identical to imageio.imwrite's."""
    d = save_dir.joinpath(name)
    d.mkdir(exist_ok=True)
    views = _lfutils.sai_to_rgb8_views(sr_sai_y, cbcr, ang).cpu().numpy()
    for i in range(ang):
        for j in range(ang):
            _lfutils.write_bmp(str(d) + "/View_%d_%d.bmp" % (i, j), views[i, j])


def test(test_loader, device, net, args, save_dir=None):
    names, psnrs, ssims = [], [], []
    net.eval()
    for Lr_SAI_y, Hr_SAI_y, Sr_SAI_cbcr, data_info, LF_name in test_loader:
        ang = int(data_info[0][0].item()) if torch.is_tensor(data_info[0]) else int(data_info[0])
        # host tensors go in as they are: the scene driver stages them through pinned buffers on its copy stream
        lr, hr = Lr_SAI_y.squeeze(), Hr_SAI_y.squeeze()
        with torch.no_grad():
            psnr, ssim, sr = _scene.test_scene(net, lr, hr, ang, args.scale_factor, args.patch_size_for_test,
                                               args.stride_for_test, getattr(args, "minibatch", 64),
                                               self_ensemble=bool(getattr(args, "self_ensemble", 0)))
        psnrs.append(psnr)
        ssims.append(ssim)
        names.append(LF_name[0])
        if save_dir is not None:
            _write_views(save_dir, LF_name[0], sr, Sr_SAI_cbcr, args.angRes_out)
    return psnrs, ssims, names
