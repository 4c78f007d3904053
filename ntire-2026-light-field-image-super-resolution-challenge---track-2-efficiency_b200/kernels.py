"""Host-side launchers: torch tensors -> raw pointers -> C ABI (include/lfsr.h).

Feature tensors are fp32 NHWC *views*: ``t[n, y, x, c]`` with ``stride(3) == 1`` and dense rows,
so a channel slice ``buf[..., a:b]`` of a wider buffer is a valid operand (torch.cat/torch.split
of the reference become pointer arithmetic). ``CudaOps`` is the only product backend; it raises
when the tensors are not on a CUDA device. (tests/opref.py implements the same op contracts in
plain torch to check each kernel and, on CPU, the layer graphs.)
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _native as N


def ld_for(c: int) -> int:
    """pixel stride (floats) for a c-channel buffer: 16-byte aligned rows for float4 / TMA."""
    return c if c == 1 else (c + 3) // 4 * 4


def alloc_nhwc(n: int, h: int, w: int, c: int, device, zero: bool = False) -> torch.Tensor:
    ld = ld_for(c)
    buf = (torch.zeros if zero else torch.empty)((n, h, w, ld), dtype=torch.float32, device=device)
    return buf[..., :c] if ld != c else buf


def alloc_nhwc16(n: int, h: int, w: int, c: int, device) -> torch.Tensor:
    """fp16 NHWC buffer (operand copies between tensor-core layers): pixel stride a multiple of 8 halves (16 bytes)."""
    ld = (c + 15) // 16 * 16 if c <= 64 else (c + 7) // 8 * 8      # rows of whole 32-byte sectors (TMA boxes are 128-byte rows)
    if 32 < c <= 64:
        ld = 64
    buf = torch.zeros((n, h, w, ld), dtype=torch.float16, device=device)
    return buf[..., :c] if ld != c else buf


def as_tensor(t: torch.Tensor, what: str = "tensor", f16: bool = False) -> N.Tensor:
    """Describe a 4-D fp32 (or, with f16, fp16) NHWC view to the C ABI; rows must be dense with pixel stride ld = stride(2)."""
    if t.dtype != (torch.float16 if f16 else torch.float32) or t.dim() != 4:
        raise N.LfsrError(f"{what}: expected a 4-D {'float16' if f16 else 'float32'} NHWC view, got {tuple(t.shape)} {t.dtype}")
    n, h, w, c = t.shape
    s = t.stride()
    ld = s[2]
    ok = (c == 1 or s[3] == 1) and ld >= c and (h == 1 or s[1] == w * ld) and (n == 1 or s[0] == h * w * ld)
    if not ok:
        raise N.LfsrError(f"{what}: not a dense-row NHWC view (shape {tuple(t.shape)}, strides {s})")
    return N.Tensor(t.data_ptr(), n, h, w, c, ld)


_NULL_T = N.Tensor(None, 0, 0, 0, 0, 0)


@dataclass
class PackedConv:
    """One convolution's constants, packed once per weight version.

    w_f32: [kh*kw*cin, cout] fp32 (tap-major, cout fastest) for lfsr_conv2d_f32.
    w_tc : TMA/UMMA-friendly packing for lfsr_conv2d_tc, or None when the layer stays on CUDA cores.
    """
    w_f32: torch.Tensor
    bias: Optional[torch.Tensor]
    kh: int
    kw: int
    cin: int
    cout: int
    stride: Tuple[int, int] = (1, 1)
    dil: Tuple[int, int] = (1, 1)
    pad: Tuple[int, int] = (0, 0)
    w_tc: Optional[torch.Tensor] = None
    w_tc16: Optional[torch.Tensor] = None   # fp16 packing (lfsr_pack_conv_tc16) for layers fed with fp16 activations
    tc_perm_r2: int = 0   # >0: w_tc rows were permuted to factor-major for a fused nn.PixelShuffle of r2 sub-pixels
    #: per-image gated copies of w_tc (lfsr_scale_pack_tc), keyed by batch size. Owned by the packing, so the scratch lives
    #: exactly as long as the weights it was sized for (a cache on the backend keyed by data_ptr could match a stale entry
    #: after the allocator reuses the address)
    gated: Optional[dict] = None

    def gated_scratch(self, nimg: int, device) -> torch.Tensor:
        if self.gated is None:
            self.gated = {}
        t = self.gated.get(nimg)
        if t is None:
            t = torch.empty((nimg, self.w_tc.numel()), dtype=torch.float32, device=device)
            self.gated[nimg] = t
        if tuple(t.shape) != (nimg, self.w_tc.numel()) or t.device != self.w_tc.device:
            raise N.LfsrError("gated weight scratch does not match its packing (stale cache)")
        return t


def pack_conv(weight: torch.Tensor, bias: Optional[torch.Tensor] = None, stride=(1, 1), dil=(1, 1), pad=(0, 0),
              device=None, tc: bool = False, tc_shuffle=(1, 1, 0), tc16: bool = False) -> PackedConv:
    """weight is torch-layout [cout, cin, kh, kw] (any device); returns device-resident packing.
    tc_shuffle: the PixelShuffle (ry, rx, mode) this layer will always be launched with; for
    nn.PixelShuffle order the tensor-core packing stores output channels sub-pixel-major so the
    epilogue writes contiguous channel runs per output pixel."""
    w = weight.detach().to(torch.float32)
    cout, cin, kh, kw = w.shape
    dev = device if device is not None else w.device
    w_f32 = w.permute(2, 3, 1, 0).reshape(kh * kw * cin, cout).contiguous().to(dev)
    b = None if bias is None else bias.detach().to(torch.float32).contiguous().to(dev)
    w_tc = None
    w_tc16 = None
    perm_r2 = 0
    if tc or tc16:
        lib = N.load()
        nfl = lib.lfsr_conv2d_tc_packed_floats(kh, kw, cin, cout)
        if nfl > 0:
            src = w
            r2 = tc_shuffle[0] * tc_shuffle[1]
            if r2 > 1 and tc_shuffle[2] == N.SHUF_CHANNEL_MAJOR:
                cq = cout // r2
                perm = torch.arange(cout).view(cq, r2).t().reshape(-1)      # packed row sub*cq+c <- logical c*r2+sub
                src = w[perm.to(w.device)]
                perm_r2 = r2
            src = src.contiguous().cpu()
            if tc:
                dst = torch.empty(nfl, dtype=torch.float32)
                N.check(lib.lfsr_pack_conv_tc(src.data_ptr(), dst.data_ptr(), kh, kw, cin, cout), "lfsr_pack_conv_tc")
                w_tc = dst.to(dev)
            if tc16:
                dst = torch.empty(lib.lfsr_conv2d_tc16_packed_bytes(kh, kw, cin, cout), dtype=torch.uint8)
                N.check(lib.lfsr_pack_conv_tc16(src.data_ptr(), dst.data_ptr(), kh, kw, cin, cout), "lfsr_pack_conv_tc16")
                w_tc16 = dst.to(dev)
    return PackedConv(w_f32, b, kh, kw, cin, cout, tuple(stride), tuple(dil), tuple(pad), w_tc, w_tc16, perm_r2)


class CudaOps:
    """The product backend: every method enqueues sm_100a kernels on torch's current stream."""

    name = "cuda"

    def __init__(self, use_tc: bool = True):
        self.lib = N.load()
        self.use_tc = use_tc
        self.use_thin = True      # FFMA2 kernel for the 18 -> 20 channel layers (tests switch it off to reach the TC path)

    # -- helpers ---------------------------------------------------------------------------
    @staticmethod
    def _stream(t: torch.Tensor) -> int:
        """stream the launch goes to. Kernels launch on the thread's CURRENT device, so a tensor that lives on another GPU
        is refused here (the callers - LFNetBase.forward, lfutils, scene - enter torch.cuda.device(x.device) first)."""
        if not t.is_cuda:
            raise N.LfsrError("lfsr_b200 kernels need CUDA tensors; there is no CPU fallback")
        if t.device.index != torch.cuda.current_device():
            raise N.LfsrError(f"tensor on {t.device} but the current CUDA device is {torch.cuda.current_device()}: "
                              "wrap the call in torch.cuda.device(tensor.device)")
        return torch.cuda.current_stream(t.device).cuda_stream

    @staticmethod
    def _ptr(t: Optional[torch.Tensor]):
        return None if t is None else t.data_ptr()

    # -- patch pipeline ----------------------------------------------------------------------
    def divide_rows(self, scene, patches, ang, h0, w0, patch, stride, u0, u1):
        N.check(self.lib.lfsr_divide_rows(scene.data_ptr(), patches.data_ptr(), ang, h0, w0, patch, stride, u0, u1,
                                          self._stream(scene)), "lfsr_divide_rows")

    def integrate_rows(self, patches, out, ang, pz, stride, h, w, num_u, num_v, u0, u1):
        N.check(self.lib.lfsr_integrate_rows(patches.data_ptr(), out.data_ptr(), ang, pz, stride, h, w, num_u, num_v,
                                             u0, u1, self._stream(out)), "lfsr_integrate_rows")

    def divide_rows_d8(self, scene, patches, ang, h0, w0, patch, stride, u0, u1):
        """the 8 self-ensemble variants of every patch of rows [u0, u1): patches [n][8][A*P][A*P] (include/lfsr.h)"""
        N.check(self.lib.lfsr_divide_rows_d8(scene.data_ptr(), patches.data_ptr(), ang, h0, w0, patch, stride, u0, u1,
                                             self._stream(scene)), "lfsr_divide_rows_d8")

    def integrate_rows_d8(self, patches8, out, ang, pz, stride, h, w, num_u, num_v, u0, u1):
        """LFintegrate of the per-patch means of the 8 un-transformed SR variants in patches8 [n][8][A*pz][A*pz]"""
        N.check(self.lib.lfsr_integrate_rows_d8(patches8.data_ptr(), out.data_ptr(), ang, pz, stride, h, w, num_u, num_v,
                                                u0, u1, self._stream(out)), "lfsr_integrate_rows_d8")

    def window_accumulate(self, win, grid, ang, n, h, w, o_u, o_v, modes):
        """merge the SR window mosaic win [(ang h), (ang w)] into the N x N mosaic grid [(n h), (n w)] at view offset
        (o_u, o_v); modes: ang * ang ints, per window view 0 = store, 1 = add, c >= 2 = add then divide by c
        (include/lfsr.h, "Angular window tiling")"""
        self.window_accumulate_uv(win, grid, ang, n, n, h, w, o_u, o_v, modes)

    def window_accumulate_uv(self, win, grid, ang, n_u, n_v, h, w, o_u, o_v, modes):
        """window_accumulate into an n_u x n_v mosaic grid [(n_u h), (n_v w)]"""
        if not (win.is_contiguous() and grid.is_contiguous() and win.dtype == grid.dtype == torch.float32):
            raise N.LfsrError("window_accumulate: dense fp32 mosaics required")
        if len(modes) != ang * ang:
            raise N.LfsrError(f"window_accumulate: {len(modes)} modes for {ang * ang} window views")
        m = (C.c_int32 * (ang * ang))(*[int(x) for x in modes])
        N.check(self.lib.lfsr_window_accumulate_uv(win.data_ptr(), grid.data_ptr(), ang, n_u, n_v, h, w, o_u, o_v, m,
                                                   self._stream(grid)), "lfsr_window_accumulate_uv")

    def interp(self, x, out, n, h, w, scale, mode, block_h, block_w):
        N.check(self.lib.lfsr_interp(x.data_ptr(), out.data_ptr(), n, h, w, scale, mode, block_h, block_w,
                                     self._stream(x)), "lfsr_interp")

    # -- convolutions ---------------------------------------------------------------------------
    def conv(self, x, pc: PackedConv, out, act=N.ACT_NONE, slope=0.0, alpha=1.0, mul=None, mul_act=N.ACT_NONE, res=None,
             in_scale=None,
             in_perm=0, out_perm=0, perm_a=0, shuffle=(1, 1, 0), block=(0, 0), tail=None, out16=None):
        """tail = (tail_w [c][12] device tensor, taps, c): store the projection of the shuffled activation onto `taps`
        vectors instead of the activation (lfsr_conv_desc.tail_w); tensor-core path only.
        fp16 operand path (tensor cores only, raises when the layer does not qualify): `x` may be a float16 NHWC view (then
        pc.w_tc16 is used); `out16` is a float16 view that receives a copy of the output; `out=None` with `out16` writes the
        fp16 tensor only."""
        if (pc.cin == 1 and out16 is not None and out is not None and x.dtype == torch.float32 and mul is None and res is None
                and in_scale is None and tail is None and not in_perm and not out_perm):
            # 1-channel stem that also writes the fp16 operand copy of its output (no separate conversion pass)
            d = N.ConvDesc()
            d.kh, d.kw = pc.kh, pc.kw
            d.stride_h, d.stride_w = pc.stride
            d.dil_h, d.dil_w = pc.dil
            d.pad_h, d.pad_w = pc.pad
            d.shuf_ry, d.shuf_rx, d.shuf_mode = shuffle
            d.block_h, d.block_w = block
            d.act, d.act_slope, d.alpha = act, slope, alpha
            d.bias = self._ptr(pc.bias)
            d.out16 = as_tensor(out16, "conv.out16", f16=True)
            d.out_mode = N.OUT_BOTH
            tin, tout = as_tensor(x, "conv.in"), as_tensor(out, "conv.out")
            if self.lib.lfsr_conv2d_stem_supported(C.byref(tin), C.byref(tout), C.byref(d)):
                N.check(self.lib.lfsr_conv2d_stem(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), self._stream(x)),
                        "lfsr_conv2d_stem")
                return
            self.conv(x, pc, out, act=act, slope=slope, alpha=alpha, shuffle=shuffle, block=block)      # stem, then the conversion
            self.to_f16(out, out16)
            return
        if x.dtype == torch.float16 or out16 is not None:
            return self._conv16(x, pc, out, out16, act, slope, alpha, mul, mul_act, res, shuffle, block, tail, in_scale)
        d = N.ConvDesc()
        d.kh, d.kw = pc.kh, pc.kw
        d.stride_h, d.stride_w = pc.stride
        d.dil_h, d.dil_w = pc.dil
        d.pad_h, d.pad_w = pc.pad
        d.in_perm, d.out_perm, d.perm_a = in_perm, out_perm, perm_a
        d.shuf_ry, d.shuf_rx, d.shuf_mode = shuffle
        d.block_h, d.block_w = block
        d.act, d.act_slope, d.alpha, d.mul_act = act, slope, alpha, mul_act
        d.bias = self._ptr(pc.bias)
        d.in_scale = self._ptr(in_scale)
        if in_scale is not None:      # [n,1,1,cin] NHWC view (possibly padded rows) or dense [n,cin]
            d.in_scale_ld = in_scale.stride(0) if in_scale.shape[0] > 1 else pc.cin
        d.mul = as_tensor(mul, "conv.mul") if mul is not None else _NULL_T
        d.res = as_tensor(res, "conv.res") if res is not None else _NULL_T
        if tail is not None:
            d.tail_w, d.tail_taps, d.tail_c = tail[0].data_ptr(), tail[1], tail[2]
        tin, tout = as_tensor(x, "conv.in"), as_tensor(out, "conv.out")
        if x.shape[3] != pc.cin:
            raise N.LfsrError(f"conv: input has {x.shape[3]} channels, weights expect {pc.cin}")
        st = self._stream(x)
        if tail is not None:
            if not (self.use_tc and pc.w_tc is not None and self.lib.lfsr_conv2d_tc_supported(C.byref(tin), C.byref(tout), C.byref(d))):
                raise N.LfsrError("conv: tail projection is only available on the tensor-core path (query tail_supported first)")
            N.check(self.lib.lfsr_conv2d_tc(C.byref(tin), pc.w_tc.data_ptr(), C.byref(tout), C.byref(d), st), "lfsr_conv2d_tc")
            return
        if pc.cin == 1 and self.lib.lfsr_conv2d_stem_supported(C.byref(tin), C.byref(tout), C.byref(d)):
            N.check(self.lib.lfsr_conv2d_stem(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), st), "lfsr_conv2d_stem")
            return
        if (pc.cout == 20 and pc.cin <= 20 and self.use_thin and
                self.lib.lfsr_conv2d_thin_supported(C.byref(tin), C.byref(tout), C.byref(d))):
            N.check(self.lib.lfsr_conv2d_thin(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), st), "lfsr_conv2d_thin")
            return
        if pc.cout in (8, 16) and pc.w_tc is None and self.lib.lfsr_conv1x1_few_supported(C.byref(tin), C.byref(tout), C.byref(d)):
            N.check(self.lib.lfsr_conv1x1_few(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), st), "lfsr_conv1x1_few")
            return
        if pc.cout <= 4 and self.lib.lfsr_conv2d_small_cout_supported(C.byref(tin), C.byref(tout), C.byref(d)):
            N.check(self.lib.lfsr_conv2d_small_cout(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), st),
                    "lfsr_conv2d_small_cout")
            return
        if self.use_tc and pc.w_tc is not None and in_scale is not None:
            # per-sample gate folded into per-image weight sets (a few KB each), then the tensor-core conv
            nimg = x.shape[0]
            scratch = pc.gated_scratch(nimg, x.device)
            N.check(self.lib.lfsr_scale_pack_tc(pc.w_tc.data_ptr(), in_scale.data_ptr(), d.in_scale_ld, scratch.data_ptr(),
                                                nimg, pc.kh, pc.kw, pc.cin, pc.cout, st), "lfsr_scale_pack_tc")
            d.w_batch_stride = pc.w_tc.numel()
            if self.lib.lfsr_conv2d_tc_supported(C.byref(tin), C.byref(tout), C.byref(d)):
                N.check(self.lib.lfsr_conv2d_tc(C.byref(tin), scratch.data_ptr(), C.byref(tout), C.byref(d), st),
                        "lfsr_conv2d_tc")
                return
            d.w_batch_stride = 0
        r2 = shuffle[0] * shuffle[1]
        perm_ok = pc.tc_perm_r2 == (r2 if (r2 > 1 and shuffle[2] == N.SHUF_CHANNEL_MAJOR) else 0)
        if (self.use_tc and pc.w_tc is not None and perm_ok and
                self.lib.lfsr_conv2d_tc_supported(C.byref(tin), C.byref(tout), C.byref(d))):
            N.check(self.lib.lfsr_conv2d_tc(C.byref(tin), pc.w_tc.data_ptr(), C.byref(tout), C.byref(d), st),
                    "lfsr_conv2d_tc")
        else:
            N.check(self.lib.lfsr_conv2d_f32(C.byref(tin), pc.w_f32.data_ptr(), C.byref(tout), C.byref(d), st),
                    "lfsr_conv2d_f32")

    def _conv16(self, x, pc, out, out16, act, slope, alpha, mul, mul_act, res, shuffle, block, tail, in_scale=None):
        d = N.ConvDesc()
        d.kh, d.kw = pc.kh, pc.kw
        d.stride_h, d.stride_w = pc.stride
        d.dil_h, d.dil_w = pc.dil
        d.pad_h, d.pad_w = pc.pad
        d.shuf_ry, d.shuf_rx, d.shuf_mode = shuffle
        d.block_h, d.block_w = block
        d.act, d.act_slope, d.alpha, d.mul_act = act, slope, alpha, mul_act
        d.bias = self._ptr(pc.bias)
        d.mul = as_tensor(mul, "conv.mul") if mul is not None else _NULL_T
        d.res = as_tensor(res, "conv.res") if res is not None else _NULL_T
        if tail is not None:
            d.tail_w, d.tail_taps, d.tail_c = tail[0].data_ptr(), tail[1], tail[2]
        in16 = x.dtype == torch.float16
        d.in_f16 = 1 if in16 else 0
        w = pc.w_tc16 if in16 else pc.w_tc
        if w is None or not self.use_tc:
            raise N.LfsrError("conv: the fp16 operand path needs tensor-core packed weights (pack_conv(tc16=True) / tc=True)")
        if in_scale is not None:      # per-sample gate folded into per-image (TF32) weight sets; fp32 input only
            if in16:
                raise N.LfsrError("conv: per-sample gated weights exist for fp32 inputs only")
            nimg = x.shape[0]
            d.in_scale = in_scale.data_ptr()
            d.in_scale_ld = in_scale.stride(0) if in_scale.shape[0] > 1 else pc.cin
            scratch = pc.gated_scratch(nimg, x.device)
            N.check(self.lib.lfsr_scale_pack_tc(pc.w_tc.data_ptr(), in_scale.data_ptr(), d.in_scale_ld, scratch.data_ptr(),
                                                nimg, pc.kh, pc.kw, pc.cin, pc.cout, self._stream(x)), "lfsr_scale_pack_tc")
            d.w_batch_stride = pc.w_tc.numel()
            w = scratch
        r2 = shuffle[0] * shuffle[1]
        if pc.tc_perm_r2 != (r2 if (r2 > 1 and shuffle[2] == N.SHUF_CHANNEL_MAJOR) else 0):
            raise N.LfsrError("conv: weights were packed for a different PixelShuffle")
        tin = as_tensor(x, "conv.in", f16=in16)
        if out16 is not None:
            d.out16 = as_tensor(out16, "conv.out16", f16=True)
            d.out_mode = N.OUT_BOTH if out is not None else N.OUT_F16
        if out is not None:
            tout = as_tensor(out, "conv.out")
        else:           # geometry only: the fp32 pointer is not written in OUT_F16 mode
            tout = N.Tensor(out16.data_ptr(), out16.shape[0], out16.shape[1], out16.shape[2], out16.shape[3], out16.stride(2))
        if x.shape[3] != pc.cin:
            raise N.LfsrError(f"conv: input has {x.shape[3]} channels, weights expect {pc.cin}")
        if not self.lib.lfsr_conv2d_tc_supported(C.byref(tin), C.byref(tout), C.byref(d)):
            raise N.LfsrError("conv: this layer does not qualify for the fp16 operand path")
        N.check(self.lib.lfsr_conv2d_tc(C.byref(tin), w.data_ptr(), C.byref(tout), C.byref(d), self._stream(x)), "lfsr_conv2d_tc")

    def split_tf32(self, x, hi, lo):
        """dense fp32 tensors: hi = tf32(x), lo = x - hi"""
        if not (x.is_contiguous() and hi.is_contiguous() and lo.is_contiguous()):
            raise N.LfsrError("split_tf32: dense tensors required")
        N.check(self.lib.lfsr_split_tf32(x.data_ptr(), hi.data_ptr(), lo.data_ptr(), x.numel(), self._stream(x)), "lfsr_split_tf32")

    def macpi_unshuffle(self, x, out, ang, r, accumulate):
        """x [n,H,W,r*r] (MacPI arrangement) -> out [n,1,H*r,W*r] SAI image (+= when accumulate)"""
        N.check(self.lib.lfsr_macpi_unshuffle(C.byref(as_tensor(x, "unshuffle.in")), out.data_ptr(), ang, r, 1 if accumulate else 0,
                                              self._stream(x)), "lfsr_macpi_unshuffle")

    def to_f16(self, x, out16):
        N.check(self.lib.lfsr_to_f16(C.byref(as_tensor(x, "to_f16.in")), C.byref(as_tensor(out16, "to_f16.out", f16=True)),
                                     self._stream(x)), "lfsr_to_f16")

    def tail_supported(self, pc: PackedConv, cq: int, shuffle) -> bool:
        """can `pc` (a conv + PixelShuffle to cq channels) end in a tail projection on this backend?"""
        return bool(self.use_tc and pc.w_tc is not None and shuffle[0] * shuffle[1] > 1 and cq % 4 == 0
                    and (pc.cout <= 240 or (cq % 32 == 0 and 256 % cq == 0 and (pc.cout <= 256 or pc.cout % 256 == 0)))
                    and pc.stride == (1, 1))

    def tap_gather(self, taps, kh, kw, bias, res, out):
        rt = as_tensor(res, "tap_gather.res") if res is not None else _NULL_T
        N.check(self.lib.lfsr_tap_gather(C.byref(as_tensor(taps, "tap_gather.taps")), kh, kw, self._ptr(bias), C.byref(rt),
                                         C.byref(as_tensor(out, "tap_gather.out")), self._stream(taps)), "lfsr_tap_gather")

    def dwconv(self, x, w, out, kh, kw, dil=(1, 1), scale=None, shift=None, act=N.ACT_NONE, slope=0.0):
        N.check(self.lib.lfsr_dwconv_f32(C.byref(as_tensor(x, "dwconv.in")), w.data_ptr(), self._ptr(scale),
                                         self._ptr(shift), C.byref(as_tensor(out, "dwconv.out")), kh, kw, dil[0],
                                         dil[1], act, slope, self._stream(x)), "lfsr_dwconv_f32")

    def dwconv_multi(self, x, out, branches):
        """branches: dicts(w, kh, kw, dil=(1,1), in_c0=0, out_c0=0, c, scale=None, shift=None, act=0, slope=0.0)"""
        arr = (N.DwBranch * len(branches))()
        for d, b in zip(arr, branches):
            d.w, d.scale, d.shift = b["w"].data_ptr(), self._ptr(b.get("scale")), self._ptr(b.get("shift"))
            d.kh, d.kw = b["kh"], b["kw"]
            d.dil_h, d.dil_w = b.get("dil", (1, 1))
            d.in_c0, d.out_c0, d.c = b.get("in_c0", 0), b.get("out_c0", 0), b["c"]
            d.act, d.act_slope = b.get("act", N.ACT_NONE), b.get("slope", 0.0)
        N.check(self.lib.lfsr_dwconv_multi(C.byref(as_tensor(x, "dwconv_multi.in")), C.byref(as_tensor(out, "dwconv_multi.out")),
                                           arr, len(branches), self._stream(x)), "lfsr_dwconv_multi")

    def mel_epi_branch(self, x, w_packed, out, klen, dil, slope, tc=False):
        """tc=True: the 1x1 contractions on the tensor cores (fp16 operands), used on the fp16 operand plan"""
        fn = self.lib.lfsr_mel_epi_branch_tc if (tc and self.use_tc) else self.lib.lfsr_mel_epi_branch
        N.check(fn(C.byref(as_tensor(x, "epi.in")), w_packed.data_ptr(), C.byref(as_tensor(out, "epi.out")), klen, dil, slope,
                   self._stream(x)), "lfsr_mel_epi_branch")

    def mel_epi_pack(self, w_packed: torch.Tensor, klen: int, device) -> Optional[torch.Tensor]:
        """operand image of lfsr_mel_epi_branch_mma for the packed EPI-block weights (None: kernel length not supported)"""
        nbytes = self.lib.lfsr_mel_epi_pack_bytes(klen)
        if not (self.use_tc and nbytes):
            return None
        w = w_packed.detach().to("cpu", torch.float32).contiguous()
        img = torch.zeros(nbytes, dtype=torch.uint8)
        N.check(self.lib.lfsr_mel_epi_pack(w.data_ptr(), img.data_ptr(), klen), "lfsr_mel_epi_pack")
        return img.to(device)

    def mel_epi_branch_mma(self, x, x16, image, out, klen, dil, slope):
        """x16: the fp16 copy of x (same pixels, >= 16 channels) written by x's producer"""
        N.check(self.lib.lfsr_mel_epi_branch_mma(C.byref(as_tensor(x, "epi.in")), C.byref(as_tensor(x16, "epi.in16", f16=True)),
                                                 image.data_ptr(), C.byref(as_tensor(out, "epi.out")), klen, dil, slope,
                                                 self._stream(x)), "lfsr_mel_epi_branch_mma")

    # -- reductions / gates -------------------------------------------------------------------------
    def block_mean(self, x, out, bh, bw):
        N.check(self.lib.lfsr_block_mean(C.byref(as_tensor(x, "block_mean.in")), C.byref(as_tensor(out, "block_mean.out")),
                                         bh, bw, self._stream(x)), "lfsr_block_mean")

    def ang_expand(self, x, w, res, out, A, act=N.ACT_NONE, slope=0.0, alpha=1.0):
        """out[n, A*Y+i, A*X+j, :] = res + alpha * act(x[n, Y, X, :] @ w[i][j]); w is [A, A, cin, cout] on the device"""
        rt = as_tensor(res, "ang_expand.res") if res is not None else _NULL_T
        N.check(self.lib.lfsr_ang_expand(C.byref(as_tensor(x, "ang_expand.in")), w.data_ptr(), C.byref(rt),
                                         C.byref(as_tensor(out, "ang_expand.out")), A, act, slope, alpha, self._stream(x)),
                "lfsr_ang_expand")

    def pooled_mlp(self, x, out, pc1: PackedConv, act1, pc2: Optional[PackedConv] = None, act2=N.ACT_NONE, pool=False):
        """one launch for a chain of 1x1 convs on the few positions of `x` [n,h,w,c] (pool: on their mean): the stage gates
        and the SA modulator's angular MLP of the Track-2 model"""
        if pc1.kh != 1 or pc1.kw != 1 or pc1.cin != x.shape[3] or (pc2 is not None and (pc2.kh != 1 or pc2.kw != 1 or pc2.cin != pc1.cout)):
            raise N.LfsrError("pooled_mlp: 1x1 layers whose widths chain are required")
        N.check(self.lib.lfsr_pooled_mlp(C.byref(as_tensor(x, "mlp.in")), 1 if pool else 0, pc1.w_f32.data_ptr(), self._ptr(pc1.bias),
                                         pc1.cout, act1, None if pc2 is None else pc2.w_f32.data_ptr(),
                                         None if pc2 is None else self._ptr(pc2.bias), 0 if pc2 is None else pc2.cout, act2,
                                         C.byref(as_tensor(out, "mlp.out")), self._stream(x)), "lfsr_pooled_mlp")

    def sa_modulate(self, x, dw_w, bn_scale, bn_shift, amod, w0, w1, res, out, dil, out16=None, skip16=(0, 0)):
        """out16: fp16 copy of the first out16.shape[3] output channels, minus the channel window skip16 = (lo, hi)"""
        rt = as_tensor(res, "sa.res") if res is not None else _NULL_T
        if out16 is not None:
            N.check(self.lib.lfsr_sa_modulate16w(C.byref(as_tensor(x, "sa.x")), dw_w.data_ptr(), bn_scale.data_ptr(),
                                                 bn_shift.data_ptr(), C.byref(as_tensor(amod, "sa.amod")), w0, w1, C.byref(rt),
                                                 C.byref(as_tensor(out, "sa.out")), C.byref(as_tensor(out16, "sa.out16", f16=True)),
                                                 skip16[0], skip16[1], dil, self._stream(x)), "lfsr_sa_modulate16w")
            return
        N.check(self.lib.lfsr_sa_modulate(C.byref(as_tensor(x, "sa.x")), dw_w.data_ptr(), bn_scale.data_ptr(),
                                          bn_shift.data_ptr(), C.byref(as_tensor(amod, "sa.amod")), w0, w1, C.byref(rt),
                                          C.byref(as_tensor(out, "sa.out")), dil, self._stream(x)), "lfsr_sa_modulate")

    def scale_add(self, x, scale, res, out, out16=None):
        """out = x * scale[n][c] + res; with out16 (and out=None) the result is written as fp16 only"""
        rt = as_tensor(res, "scale_add.res") if res is not None else _NULL_T
        if out16 is not None:
            N.check(self.lib.lfsr_scale_add16(C.byref(as_tensor(x, "scale_add.x")), C.byref(as_tensor(scale, "scale_add.scale")),
                                              C.byref(rt), C.byref(as_tensor(out16, "scale_add.out16", f16=True)), self._stream(x)),
                    "lfsr_scale_add16")
            return
        N.check(self.lib.lfsr_scale_add(C.byref(as_tensor(x, "scale_add.x")), C.byref(as_tensor(scale, "scale_add.scale")),
                                        C.byref(rt), C.byref(as_tensor(out, "scale_add.out")), self._stream(x)),
                "lfsr_scale_add")

    # -- EPIT token ops ------------------------------------------------------------------------------
    def layernorm(self, x, gamma, beta, eps, out):
        N.check(self.lib.lfsr_layernorm(C.byref(as_tensor(x, "ln.in")), gamma.data_ptr(), beta.data_ptr(), eps,
                                        C.byref(as_tensor(out, "ln.out")), self._stream(x)), "lfsr_layernorm")

    def epi_attention(self, qk, v, out, heads, head_dim, A, S, half_window, nb, np_, nq, stride_a, stride_s, stride_b,
                      stride_p, stride_q):
        d = N.EpiAttnDesc(heads, head_dim, A, S, half_window, nb, np_, nq, stride_a, stride_s, stride_b, stride_p,
                          stride_q)
        N.check(self.lib.lfsr_epi_attention(qk.data_ptr(), v.data_ptr(), out.data_ptr(), C.byref(d), self._stream(qk)),
                "lfsr_epi_attention")

    # -- fused BasicTrans (EPIT.py:110-128) ------------------------------------------------------------------------
    def pack_basictrans(self, w_in, w_qkv, w_o, w_ff1, w_ff2, w_out, ln1, ln2, heads, device):
        """weights in torch layout (any device) -> (packed device buffer, descriptor template with the LayerNorm constants)"""
        host = [t.detach().to("cpu", torch.float32).contiguous() for t in (w_in, w_qkv, w_o, w_ff1, w_ff2, w_out)]
        E, Cc = host[0].shape
        if (E, Cc) != (128, 64) or tuple(host[1].shape) != (3 * E, E) or tuple(host[3].shape) != (2 * E, E) or heads != 8:
            return None
        buf = torch.empty(self.lib.lfsr_basictrans_packed_bytes(), dtype=torch.uint8)
        N.check(self.lib.lfsr_pack_basictrans(*[t.data_ptr() for t in host], buf.data_ptr()), "lfsr_pack_basictrans")
        d = N.BasicTransDesc()
        d.heads, d.E, d.C = heads, E, Cc
        for name, t in (("ln1_g", ln1[0]), ("ln1_b", ln1[1]), ("ln2_g", ln2[0]), ("ln2_b", ln2[1])):
            arr = getattr(d, name)
            for i, v in enumerate(t.detach().to("cpu", torch.float32).tolist()):
                arr[i] = v
        d.eps1, d.eps2 = float(ln1[2]), float(ln2[2])
        return buf.to(device), d

    def basictrans(self, x, packed, desc, y, A, S, half_window, nb, np_, nq, stride_a, stride_s, stride_b, stride_p, stride_q,
                   check_only=False):
        """x, y: float16 [n,h,w,64] NHWC views (operand copies: the kernel reads and writes fp16); sequences addressed as in
        epi_attention. Returns False when the geometry is unsupported (check_only: just answer)."""
        d = desc
        d.A, d.S, d.half_window, d.nb, d.np, d.nq = A, S, half_window, nb, np_, nq
        d.stride_a, d.stride_s, d.stride_b, d.stride_p, d.stride_q = stride_a, stride_s, stride_b, stride_p, stride_q
        tx, ty = as_tensor(x, "basictrans.x", f16=True), as_tensor(y, "basictrans.y", f16=True)
        if not self.lib.lfsr_basictrans_supported(C.byref(tx), C.byref(ty), C.byref(d)):
            return False
        if not check_only:
            N.check(self.lib.lfsr_epit_basictrans(C.byref(tx), packed.data_ptr(), C.byref(ty), C.byref(d), self._stream(x)),
                    "lfsr_epit_basictrans")
        return True

    # -- metrics -----------------------------------------------------------------------------------------
    def metric_sums(self, label, out, ang, h, w, acc):
        N.check(self.lib.lfsr_metric_sums(label.data_ptr(), out.data_ptr(), ang, h, w, acc.data_ptr(),
                                          self._stream(label)), "lfsr_metric_sums")

    def metric_sums_uv(self, label, out, ang_u, ang_v, h, w, acc):
        """metric_sums over an ang_u x ang_v mosaic [(ang_u h), (ang_v w)]: 2 * ang_u * ang_v sums"""
        N.check(self.lib.lfsr_metric_sums_uv(label.data_ptr(), out.data_ptr(), ang_u, ang_v, h, w, acc.data_ptr(),
                                             self._stream(label)), "lfsr_metric_sums_uv")

    def metric_sums_batched(self, label, out, n, ang, h, w, acc):
        """label/out [n,1,A*h,A*w] contiguous; acc [n*A*A*2] float64, zeroed by the caller"""
        N.check(self.lib.lfsr_metric_sums_batched(label.data_ptr(), out.data_ptr(), n, ang, h, w, acc.data_ptr(),
                                                  self._stream(label)), "lfsr_metric_sums_batched")


_default_ops = None


def default_ops() -> CudaOps:
    global _default_ops
    if _default_ops is None:
        _default_ops = CudaOps()
    return _default_ops
