"""Shared host logic of the drop-in `get_model(args)` modules.

Every network keeps the reference's parameter tree (same state_dict keys and shapes, so reference
``.pth`` files load and ``net.apply(weights_init)`` works) but never calls those leaf modules: the
forward packs the weights once per weight version (BatchNorm folded, RepConv branches merged,
tap-major layouts) and enqueues the sm_100a kernels of liblfsr_b200 on torch's current stream.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch
import torch.nn as nn

from .. import _native as N
from .. import kernels as K


#: LFSR_FP16_OPS=0 keeps every tensor-core layer on fp32 activations / TF32 operands (comparison, debugging). Default: layers
#: whose outputs only feed other tensor-core layers exchange fp16 activations (10-bit mantissa = what TF32 keeps of an operand;
#: fp32 accumulation; residual trunks, interpolation skips and everything a CUDA-core kernel reads stay fp32)
USE_FP16_OPERANDS = os.environ.get("LFSR_FP16_OPS", "1") != "0"

#: LFSR_CUDA_GRAPH=0 launches every kernel of a forward individually (profiling per-op, debugging)
USE_CUDA_GRAPH = os.environ.get("LFSR_CUDA_GRAPH", "1") != "0"


def slots(mods: Dict[int, nn.Module]) -> nn.ModuleDict:
    """nn.Sequential-compatible key layout ("0", "2", ...) without placeholder modules."""
    return nn.ModuleDict({str(i): m for i, m in mods.items()})


def bn_affine(bn: nn.BatchNorm2d):
    """eval-mode BatchNorm as y = x*scale + shift."""
    scale = bn.weight.detach() / torch.sqrt(bn.running_var.detach() + bn.eps)
    shift = bn.bias.detach() - bn.running_mean.detach() * scale
    return scale, shift


def tail_table(w_head: torch.Tensor, channels: int, device) -> torch.Tensor:
    """[channels][12] projection table of a 3x3 reconstruction conv to one channel (weight [1, c, 3, 3], c <= channels):
    column ky*3+kx holds W[0, :, ky, kx]; used as lfsr_conv_desc.tail_w by the last upsampler conv."""
    w = w_head.detach().float().cpu()
    t = torch.zeros(channels, 12, dtype=torch.float32)
    t[: w.shape[1], :9] = w[0].reshape(w.shape[1], 9)
    d = t.contiguous().to(device)
    d._lfsr_host = (d._version, t.contiguous())       # (kernels.tail_host: the host copy the launches read)
    return d


def upsample_tail(net, ops, pk, cur, ch, cw, Y, width, LR, shuf_mode):
    """PixelShuffleUpsampler stages + 3x3 head + skip (MyEfficientLFNet.py:104-109, MyEfficientLFNetV4_5.py:100-109).
    The last stage does not write its `width`-channel activation: its epilogue projects every output pixel onto the 9
    taps of the head conv and lfsr_tap_gather sums the shifted responses onto the interpolated skip already in Y.
    With pk["f16"] the activation between two stages exists in fp16 only (it feeds nothing but the next stage's MMAs)."""
    n_up = len(pk["up"])
    f16 = bool(pk.get("f16")) and width % 8 == 0
    for j, (pcv, r) in enumerate(pk["up"]):
        shuffle = (r, r, shuf_mode)
        if j == n_up - 1 and pk.get("tail_w") is not None and ops.tail_supported(pcv, width, shuffle):
            taps = net._buf("head_taps", cur.shape[0], ch * r, cw * r, 9, cur.device)
            ops.conv(cur, pcv, taps, act=LR, slope=0.1, shuffle=shuffle, tail=(pk["tail_w"], 9, width))
            ops.tap_gather(taps, 3, 3, pk["out"].bias, Y, Y)
            return
        if f16 and j < n_up - 1 and pk.get("tail_w") is not None:
            nb = net._buf16(f"up{j}", cur.shape[0], ch * r, cw * r, width, cur.device)
            ops.conv(cur, pcv, None, out16=nb, act=LR, slope=0.1, shuffle=shuffle)
        else:
            nb = net._buf(f"up{j}", cur.shape[0], ch * r, cw * r, width, cur.device)
            ops.conv(cur, pcv, nb, act=LR, slope=0.1, shuffle=shuffle)
        cur, ch, cw = nb, ch * r, cw * r
    ops.conv(cur, pk["out"], Y, res=Y)


def fp16_plan(ops) -> bool:
    """do this backend's tensor-core layers exchange fp16 activations? (USE_FP16_OPERANDS, CudaOps with tensor cores, or a
    test backend that declares fp16_operands)"""
    return bool(USE_FP16_OPERANDS and getattr(ops, "fp16_operands", getattr(ops, "use_tc", False)) and hasattr(ops, "to_f16"))


class LFNetBase(nn.Module):
    """forward(x[B,1,A*h,A*w] float32 cuda, info=None) -> [B,1,A*h*s,A*w*s] (train.py:291-313)."""

    #: channel layouts, tensor-core eligibility etc. are decided per subclass in _pack / _run
    def __init__(self, args):
        super().__init__()
        self.angRes = int(args.angRes_in)
        self.scale = int(args.scale_factor)
        self._ops = None
        self._packed = None
        self._packed_key = None
        self._arena: Dict[tuple, torch.Tensor] = {}
        self._graphs: Dict[tuple, tuple] = {}
        self.graph_launches = 0       # kernels launched through graph replays (the C-side counter only sees direct launches)
        # reference checkpoints arrive through load_state_dict (test.py:40-55): repack on the next forward
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.invalidate())

    def invalidate(self) -> None:
        """Drop the packed weights and captured graphs; the next forward repacks. Called automatically after
        load_state_dict / .to() / set_backend and whenever a parameter's (data_ptr, _version) changes. Edits made through
        `p.data` (e.g. `m.weight.data.normal_()`) bypass torch's version counter: call this after such edits."""
        self._packed = None
        self._packed_key = None
        self._graphs = {}

    # -- backend ---------------------------------------------------------------------------------
    def set_backend(self, ops) -> None:
        """Tests inject tests/opref.RefOps here; the product default is kernels.CudaOps."""
        self._ops = ops
        self.invalidate()

    def _backend(self, x: torch.Tensor):
        if self._ops is not None:
            return self._ops
        if not x.is_cuda:
            raise N.LfsrError(
                f"{type(self).__module__}: input is on {x.device}; this implementation only runs on a CUDA "
                "(sm_100a) device and has no CPU fallback")
        return K.default_ops()

    # -- weight packing cache ----------------------------------------------------------------------
    def _fingerprint(self, device):
        key = [str(device)]
        for t in list(self.parameters()) + list(self.buffers()):
            key.append((t.data_ptr(), t._version))
        return tuple(key)

    def _get_packed(self, device, ops):
        key = self._fingerprint(device)
        if self._packed is None or key != self._packed_key:
            with torch.no_grad():
                self._packed = self._pack(device, ops)
            self._packed_key = key
            self._graphs = {}          # captured graphs hold pointers into the previous packing
        return self._packed

    def _pack(self, device, ops):  # pragma: no cover - abstract
        raise NotImplementedError

    def _run(self, ops, pk, x, out):  # pragma: no cover - abstract
        raise NotImplementedError

    # -- workspace arena --------------------------------------------------------------------------
    def _buf(self, name: str, n: int, h: int, w: int, c: int, device) -> torch.Tensor:
        key = (name, n, h, w, c, str(device))
        t = self._arena.get(key)
        if t is None:
            t = K.alloc_nhwc(n, h, w, c, device, zero=True)
            self._arena[key] = t
        return t

    def _buf16(self, name: str, n: int, h: int, w: int, c: int, device) -> torch.Tensor:
        """fp16 NHWC operand buffer (activations that only tensor-core layers read)"""
        key = (name, "f16", n, h, w, c, str(device))
        t = self._arena.get(key)
        if t is None:
            t = K.alloc_nhwc16(n, h, w, c, device)
            self._arena[key] = t
        return t

    def release_workspace(self) -> None:
        self._graphs = {}
        self._arena.clear()

    def _apply(self, fn, *a, **kw):  # .to()/.cpu()/.cuda(): packed weights and arena are stale
        self._packed = None
        self._graphs = {}
        self._arena = {}
        return super()._apply(fn, *a, **kw)

    # -- forward -------------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, info=None) -> torch.Tensor:
        if x.dim() != 4 or x.shape[1] != 1:
            raise ValueError(f"expected a [B,1,A*h,A*w] Y-channel SAI mosaic, got {tuple(x.shape)}")
        if x.dtype != torch.float32:
            raise ValueError(f"expected float32 input, got {x.dtype}")
        A = self.angRes
        B, _, H, W = x.shape
        if H % A or W % A:
            raise ValueError(f"mosaic {H}x{W} is not divisible by angRes={A}")
        ops = self._backend(x)
        if x.is_cuda and x.device.index != torch.cuda.current_device():
            with torch.cuda.device(x.device):          # kernels launch on the thread's current device
                return self.forward(x, info)
        pk = self._get_packed(x.device, ops)
        x = x.contiguous()
        if (USE_CUDA_GRAPH and self._ops is None and x.is_cuda and not torch.cuda.is_current_stream_capturing()):
            return self._forward_graphed(ops, pk, x)
        out = torch.empty((B, 1, H * self.scale, W * self.scale), dtype=torch.float32, device=x.device)
        with torch.no_grad():
            self._run(ops, pk, x, out)
        return out

    def forward_static(self, x: torch.Tensor) -> torch.Tensor:
        """forward() for callers that consume the result before the next forward of the same shape (scene.SceneRunner feeds
        it straight to LFintegrate): returns the graph's own static output buffer instead of a clone."""
        ops = self._backend(x)
        if not (USE_CUDA_GRAPH and self._ops is None and x.is_cuda) or torch.cuda.is_current_stream_capturing():
            return self.forward(x)
        if x.device.index != torch.cuda.current_device():
            with torch.cuda.device(x.device):
                return self.forward_static(x)
        pk = self._get_packed(x.device, ops)
        return self._forward_graphed(ops, pk, x.contiguous(), clone=False)

    def _forward_graphed(self, ops, pk, x: torch.Tensor, clone: bool = True) -> torch.Tensor:
        """One CUDA graph per input shape: a forward is ~100 launches of a few microseconds of host work each, which at the
        reference's minibatch sizes (train.py:303-314 feeds ONE patch per call) costs more than the kernels themselves.
        The workspace arena makes every pointer of a forward stable, so the launch sequence is captured once and replayed
        with the input copied into / the result copied out of two static tensors."""
        key = tuple(x.shape)
        ent = self._graphs.get(key)
        if ent is None:
            B, _, H, W = x.shape
            sx = torch.empty_like(x)
            so = torch.empty((B, 1, H * self.scale, W * self.scale), dtype=torch.float32, device=x.device)
            sx.copy_(x)
            with torch.no_grad():
                self._run(ops, pk, sx, so)        # allocates the workspace and sets kernel attributes outside the capture
                torch.cuda.current_stream(x.device).synchronize()
                l0 = ops.lib.lfsr_launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._run(ops, pk, sx, so)
                n = ops.lib.lfsr_launch_count() - l0
            ent = (g, sx, so, n)
            self._graphs[key] = ent
        g, sx, so, n = ent
        sx.copy_(x)
        g.replay()
        self.graph_launches += n
        return so.clone() if clone else so


class L1Loss(nn.Module):
    """get_loss(args) of EPIT/DistgSSR/LF_InterNet (e.g. DistgSSR.py:158-166): plain L1."""

    def __init__(self, args=None):
        super().__init__()
        self.criterion_Loss = nn.L1Loss()

    def forward(self, SR, HR, criterion_data=None):
        if isinstance(SR, dict):
            SR = SR["SR"]
        return self.criterion_Loss(SR, HR)
