"""Track-2 model `MyEfficientLFNet` (v2.0) on liblfsr_b200 kernels.

Mirror of /root/reference/model/SR/MyEfficientLFNet.py: same `get_model(args)`, `get_loss(args)`,
`weights_init(m)` symbols and the same state_dict (279 entries, 547 540 parameters at x4), but the
eval forward is a fixed launch plan over NHWC fp32 buffers:

  bicubic(mosaic) -> Y                                       lfsr_interp      (:88-90)
  RepConv stem 1->54 (3 branches + BN folded to one conv)    lfsr_conv2d_*    (:40-43, :374-385)
  5 x ProgressiveDisentanglingStage                          (:183-208)
      spatial  RepConv(18) LReLU conv3x3 d5                  -> cat[0:18]
      angular  5x5/s5, gate chain, 1x1->450 + PixelShuffle(5) fused store, x+scale*out -> cat[18:36]
      EPI      dw 1x11 / 11x1 / 3x3 d5 + 1x1, fuse 1x1       -> cat[36:54]
      gates    per-view means -> global means -> block-diagonal FC+sigmoid -> folded into the
               fusion 1x1 as a per-sample input-channel scale
      fusion   1x1 LReLU, 3x3 d5 ; SAModulator tail + stage residual in one kernel
  global fusion 1x1 LReLU, RepConv(54) + shallow residual
  upsampler  [3x3 54->216 + PixelShuffle(2) + LReLU fused] x2 (:555-565)
  3x3 54->1 + bias + bicubic residual (in place on Y)        (:70-73, :105)

torch.cat / torch.split never materialise: branches read and write channel slices of one buffer.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import _native as N
from .. import kernels as K
from .common import LFNetBase, bn_affine, slots, tail_table, upsample_tail, fp16_plan


def _conv(cin, cout, k, **kw):
    return nn.Conv2d(cin, cout, k, **kw)


class _RepConvParams(nn.Module):
    """parameter holder with RepConvBlock's names (MyEfficientLFNet.py:330-372)."""

    def __init__(self, cin, cout, dil):
        super().__init__()
        self.conv_3x3 = _conv(cin, cout, 3, padding=dil, dilation=dil, bias=False)
        self.bn_3x3 = nn.BatchNorm2d(cout)
        self.conv_1x1 = _conv(cin, cout, 1, bias=False)
        self.bn_1x1 = nn.BatchNorm2d(cout)
        self.bn_identity = nn.BatchNorm2d(cout) if cin == cout else None

    def merged(self):
        """One 3x3 kernel + bias equal to bn(conv3x3)+bn(conv1x1)[+bn(x)] in eval mode. (The
        reference's own switch_to_deploy is broken - SURVEY 7f - so this is derived, not copied.)"""
        s3, b3 = bn_affine(self.bn_3x3)
        s1, b1 = bn_affine(self.bn_1x1)
        w = self.conv_3x3.weight.detach() * s3.view(-1, 1, 1, 1)
        w = w.clone()
        w[:, :, 1, 1] += self.conv_1x1.weight.detach()[:, :, 0, 0] * s1.view(-1, 1)
        b = b3 + b1
        if self.bn_identity is not None:
            si, bi = bn_affine(self.bn_identity)
            idx = torch.arange(w.shape[0], device=w.device)
            w[idx, idx, 1, 1] += si
            b = b + bi
        return w, b


class _AngularParams(nn.Module):
    def __init__(self, c, A):
        super().__init__()
        hidden = max(c // 4, 16)
        self.scale = nn.Parameter(torch.ones(1) * 0.1)
        self.to_angular = _conv(c, c, A, stride=A, bias=False)
        self.attention = slots({0: _conv(c, hidden, 1, bias=False),
                                2: _conv(hidden, hidden, 3, padding=1, groups=hidden, bias=False),
                                4: _conv(hidden, c, 1, bias=False)})
        self.cross_view = slots({0: _conv(c, c, 3, padding=1, bias=False)})
        self.expand = slots({0: _conv(c, c * A * A, 1, bias=False)})


class _EpiParams(nn.Module):
    def __init__(self, c, A):
        super().__init__()
        k = 2 * A + 1
        self.epi_h = slots({0: _conv(c, c, (1, k), padding=(0, A), groups=c, bias=False), 1: _conv(c, c, 1, bias=False)})
        self.epi_v = slots({0: _conv(c, c, (k, 1), padding=(A, 0), groups=c, bias=False), 1: _conv(c, c, 1, bias=False)})
        self.epi_diag = slots({0: _conv(c, c, 3, padding=A, dilation=A, groups=c, bias=False),
                               1: _conv(c, c, 1, bias=False)})
        self.fuse = slots({0: _conv(3 * c, c, 1, bias=False)})


class _SAModParams(nn.Module):
    def __init__(self, c, A):
        super().__init__()
        self.combine = nn.Parameter(torch.ones(2) * 0.5)
        self.spatial_mod = slots({0: _conv(c, c, 3, padding=A, dilation=A, groups=c, bias=False), 1: nn.BatchNorm2d(c)})
        self.angular_conv = slots({0: _conv(c, c // 4, 1, bias=False), 2: _conv(c // 4, c, 1, bias=False)})


class _StageParams(nn.Module):
    def __init__(self, c, A):
        super().__init__()
        self.split = [c // 3, c // 3, c - 2 * (c // 3)]
        s0, s1, s2 = self.split
        self.spatial_branch = slots({0: _RepConvParams(s0, s0, A), 2: _conv(s0, s0, 3, padding=A, dilation=A, bias=False)})
        self.angular_branch = _AngularParams(s1, A)
        self.epi_branch = _EpiParams(s2, A)
        self.gate_spatial = slots({1: _conv(s0, s0, 1, bias=True)})
        self.gate_angular = slots({1: _conv(s1, s1, 1, bias=True)})
        self.gate_epi = slots({1: _conv(s2, s2, 1, bias=True)})
        self.fusion = slots({0: _conv(c, c, 1, bias=False), 2: _conv(c, c, 3, padding=A, dilation=A, bias=False)})
        self.sa_modulator = _SAModParams(c, A)


class _UpsamplerParams(nn.Module):
    def __init__(self, c, scale):
        super().__init__()
        if scale == 4:
            self.up = slots({0: _conv(c, 4 * c, 3, padding=1, bias=False), 3: _conv(c, 4 * c, 3, padding=1, bias=False)})
            self.steps = [(0, 2), (3, 2)]
        elif scale == 2:
            self.up = slots({0: _conv(c, 4 * c, 3, padding=1, bias=False)})
            self.steps = [(0, 2)]
        else:
            self.up = slots({0: _conv(c, c * scale * scale, 3, padding=1, bias=False)})
            self.steps = [(0, scale)]


def _dw_pack(w, device):
    """depthwise weight [C,1,kh,kw] -> [kh*kw, C]"""
    c, _, kh, kw = w.shape
    return w.detach().reshape(c, kh * kw).t().contiguous().to(device=device, dtype=torch.float32)


class get_model(LFNetBase):
    def __init__(self, args):
        super().__init__(args)
        A = self.angRes
        self.channels = 54
        self.n_stages = 5
        c = self.channels
        self.shallow_feat = _RepConvParams(1, c, A)
        self.stages = nn.ModuleList([_StageParams(c, A) for _ in range(self.n_stages)])
        self.global_fusion = slots({0: _conv(c, c, 1, bias=False), 2: _RepConvParams(c, c, A)})
        self.upsampler = _UpsamplerParams(c, self.scale)
        self.output_conv = _conv(c, 1, 3, stride=1, padding=1, bias=True)

    # -- channel layout ------------------------------------------------------------------------------
    # The 54 trunk channels are the concat of three 18-channel branches. They live in HBM as three groups
    # of GS = 20 floats (18 real + 2 always-zero pad): every branch slice then starts 16-byte aligned, which
    # is what lets the 18-channel convs run on the TMA/tcgen05 path and the elementwise kernels use 128-bit
    # accesses. Weights of 54-channel producers/consumers are expanded with zero rows/columns accordingly.
    def _groups(self):
        c = self.channels
        sp = [c // 3, c // 3, c - 2 * (c // 3)]
        gs = (max(sp) + 3) // 4 * 4
        return sp, gs

    def _exp(self, t, dim, fill=0.0):
        """insert the pad channels along `dim` of a tensor whose size there is self.channels"""
        sp, gs = self._groups()
        shape = list(t.shape)
        shape[dim] = gs * len(sp)
        out = t.new_full(shape, fill)
        o = 0
        for g, n in enumerate(sp):
            out.narrow(dim, g * gs, n).copy_(t.narrow(dim, o, n))
            o += n
        return out

    # -- pack ---------------------------------------------------------------------------------------
    def _pack(self, device, ops):
        A = self.angRes
        pc = lambda w, b=None, **kw: K.pack_conv(w.detach().float().cpu(), None if b is None else b.detach().float().cpu(),
                                                 device=device, **kw)
        dil = dict(dil=(A, A), pad=(A, A))
        dev_t = lambda t: t.detach().to(device=device, dtype=torch.float32).contiguous()

        def pad_out(w, b=None, to=None):
            """zero output rows up to a multiple of 4 channels (or `to`): the layer then writes its pad floats too (with
            zeros, the value they must hold) and qualifies for the 16-byte-granular TMA-store epilogue / the thin kernel"""
            w = w.detach().float().cpu()
            n = (to if to is not None else (w.shape[0] + 3) // 4 * 4) - w.shape[0]
            if n:
                w = torch.cat([w, w.new_zeros((n,) + tuple(w.shape[1:]))], 0)
                b = None if b is None else torch.cat([b.detach().float().cpu(), torch.zeros(n)])
            return w, b
        f16 = fp16_plan(ops)
        pk = {"f16": f16}
        w, b = self.shallow_feat.merged()
        pk["stem"] = pc(self._exp(w, 0), self._exp(b, 0), **dil)
        stages = []
        gs_ = self._groups()[1]
        for st in self.stages:
            s = {}
            w, b = st.spatial_branch["0"].merged()
            s["spa0"] = pc(*pad_out(w, b), tc=True, **dil)
            s["spa2"] = pc(*pad_out(st.spatial_branch["2"].weight), tc=True, **dil)
            if f16:
                # fp16 operand plan: both 18-channel convs on the tensor cores over 32-channel fp16 pixels (64 contiguous bytes:
                # a TMA box row of 18 or 24 channels is 2.4x slower, run_thin_vs_lean.py); input channels 18..31 carry zero
                # weights (they are the next group's channels / the zero pad), 0.25 -> 0.15 ms per layer against the FFMA2 kernel
                def pad_in(wb, to=32):
                    w_, b_ = wb
                    return torch.cat([w_, w_.new_zeros((w_.shape[0], to - w_.shape[1]) + tuple(w_.shape[2:]))], 1), b_
                s["spa0h"] = pc(*pad_in(pad_out(w, b, to=24)), tc=True, tc16=True, **dil)
                s["spa2h"] = pc(*pad_in(pad_out(st.spatial_branch["2"].weight)), tc=True, tc16=True, **dil)
            ab = st.angular_branch
            # the small angular-resolution tensors are all 20-float pixels (real channels + zeros): every layer of the
            # attention runs on the thin FFMA2 kernel / the tiled depthwise kernel
            s["ang_to"] = pc(*pad_out(ab.to_angular.weight), stride=(A, A), tc=True)
            s["ang_a0"] = pc(*pad_out(ab.attention["0"].weight, to=gs_))
            dwp = _dw_pack(ab.attention["2"].weight, "cpu")                          # [9][hid]
            s["ang_a2"] = torch.cat([dwp, dwp.new_zeros(dwp.shape[0], gs_ - dwp.shape[1])], 1).contiguous().to(device)
            s["ang_hid"] = dwp.shape[1]
            s["ang_a4"] = pc(*pad_out(ab.attention["4"].weight, to=gs_))
            s["ang_cv"] = pc(*pad_out(ab.cross_view["0"].weight, to=gs_), pad=(1, 1))
            # expand conv 1x1 + PixelShuffle(A) for the streaming kernel (lfsr_ang_expand): [A][A][cin][cout padded to gs],
            # nn.PixelShuffle order; the padded output channels make the layer write whole 20-float slots
            wx = ab.expand["0"].weight.detach().float().cpu()[:, :, 0, 0]            # [c*A*A + i*A + j, cin]
            ce = wx.shape[0] // (A * A)
            wx = wx.view(ce, A, A, wx.shape[1]).permute(1, 2, 3, 0)                   # [i, j, cin, c]
            s["ang_exw"] = torch.cat([wx, wx.new_zeros(A, A, wx.shape[2], gs_ - ce)], 3).contiguous().to(device)
            s["ang_scale"] = float(ab.scale.detach().item())
            eb = st.epi_branch
            pw_t = lambda m: m.weight.detach().float()[:, :, 0, 0].t().contiguous().reshape(-1).cpu()   # [in][out]
            dw_t = lambda m: _dw_pack(m.weight, "cpu").reshape(-1)
            s["epi_w"] = torch.cat([dw_t(eb.epi_h["0"]), dw_t(eb.epi_v["0"]), dw_t(eb.epi_diag["0"]),
                                    pw_t(eb.epi_h["1"]), pw_t(eb.epi_v["1"]), pw_t(eb.epi_diag["1"]),
                                    pw_t(eb.fuse["0"])]).to(device)
            s["epi_klen"] = eb.epi_h["0"].weight.shape[-1]
            # fp16 operand plan: pre-swizzled tensor-core operands of the all-MMA EPI kernel, its depthwise taps as shifted-row
            # tcgen05 MMAs (0.27 ms per stage at batch 64 against 0.34 for the hybrid kernel). None when the packer does not
            # take the kernel length (2A+1 > 15) or the backend has none: the hybrid kernel runs the block then
            s["epi_img"] = (ops.mel_epi_pack(s["epi_w"], s["epi_klen"], device)
                            if (f16 and hasattr(ops, "mel_epi_pack")) else None)
            # three gate FCs as one block-diagonal 1x1 over the grouped layout (MyEfficientLFNet.py:159-173)
            sp, gs = self._groups()
            CP = gs * len(sp)
            gw = torch.zeros(CP, CP, 1, 1)
            gb = torch.zeros(CP)
            for g, (gate, n) in enumerate(zip((st.gate_spatial, st.gate_angular, st.gate_epi), sp)):
                gw[g * gs:g * gs + n, g * gs:g * gs + n] = gate["1"].weight.detach().float().cpu()
                gb[g * gs:g * gs + n] = gate["1"].bias.detach().float().cpu()
            s["gate"] = pc(gw, gb)
            s["fus0"] = pc(*pad_out(self._exp(st.fusion["0"].weight.detach().float().cpu(), 1)), tc=True)
            s["fus2"] = pc(self._exp(st.fusion["2"].weight.detach().float().cpu(), 0), tc=True, tc16=f16, **dil)
            sm = st.sa_modulator
            s["sa_dw"] = dev_t(self._exp(_dw_pack(sm.spatial_mod["0"].weight, "cpu"), 1))
            sc, sh = bn_affine(sm.spatial_mod["1"])
            s["sa_bns"] = dev_t(self._exp(sc.float().cpu(), 0, 1.0))
            s["sa_bnb"] = dev_t(self._exp(sh.float().cpu(), 0))
            s["sa_c0"] = pc(self._exp(sm.angular_conv["0"].weight.detach().float().cpu(), 1))
            s["sa_c2"] = pc(self._exp(sm.angular_conv["2"].weight.detach().float().cpu(), 0))
            wts = torch.softmax(sm.combine.detach().float(), dim=0)
            s["sa_w"] = (float(wts[0]), float(wts[1]))
            stages.append(s)
        pk["stages"] = stages
        pk["gf0"] = pc(*pad_out(self._exp(self.global_fusion["0"].weight.detach().float().cpu(), 1)), tc=True)
        w, b = self.global_fusion["2"].merged()
        # fp16 operand plan: 64 output channels (60 + 4 zero rows), so the layer can write the fp16-only tensor the first
        # upsampler conv reads (fp16 outputs need whole 16-byte channel groups)
        pk["gf2"] = pc(*pad_out(self._exp(w.float().cpu(), 0), self._exp(b.float().cpu(), 0), to=64 if f16 else None), tc=True,
                       tc16=f16, **dil)
        # upsampler activations carry CU = 56 channels (54 + 2 zero): 128-bit epilogue stores, and 4*56 = 224 is
        # exactly the MMA N the 216 real output channels were padded to anyway
        C = self.channels
        CU = (C + 3) // 4 * 4
        def pad_ch(w, dim, r2=1):
            """zero-pad the channel dim from C(*r2) to CU(*r2); nn.PixelShuffle order keeps r2 innermost"""
            shape = list(w.shape)
            wv = w.reshape(shape[:dim] + [C, r2] + shape[dim + 1:])
            padshape = list(wv.shape)
            padshape[dim] = CU - C
            return torch.cat([wv, wv.new_zeros(padshape)], dim).reshape(shape[:dim] + [CU * r2] + shape[dim + 1:])
        ups = []
        for j, (i, r) in enumerate(self.upsampler.steps):
            w = self.upsampler.up[str(i)].weight.detach().float().cpu()
            w = self._exp(w, 1) if j == 0 else pad_ch(w, 1)          # reads the grouped trunk / the padded up buffer
            if j == 0 and f16:                                      # ... as the 64-channel fp16 tensor of the fp16 operand plan
                w = torch.cat([w, w.new_zeros((w.shape[0], 64 - w.shape[1]) + tuple(w.shape[2:]))], 1)
            w = pad_ch(w, 0, r * r)
            ups.append((pc(w, pad=(1, 1), tc=True, tc16=f16, tc_shuffle=(r, r, N.SHUF_CHANNEL_MAJOR)), r))
        pk["up"] = ups
        pk["out"] = pc(pad_ch(self.output_conv.weight.detach().float().cpu(), 1), self.output_conv.bias, pad=(1, 1))
        pk["CU"] = CU
        pk["tail_w"] = tail_table(self.output_conv.weight, CU, device)
        return pk

    # -- run ------------------------------------------------------------------------------------------
    def _run(self, ops, pk, x, out):
        A, s, C = self.angRes, self.scale, self.channels
        sp, gs = self._groups()
        CP = gs * len(sp)
        c0 = sp[0]
        sl = [slice(g * gs, g * gs + n) for g, n in enumerate(sp)]
        B, _, H, W = x.shape
        dev = x.device
        buf = lambda name, h, w, c: self._buf(name, B, h, w, c, dev)
        LR = N.ACT_LRELU
        xin = x.view(B, H, W, 1)
        Y = out.view(B, H * s, W * s, 1)
        ops.interp(x, out, B, H, W, s, N.INTERP_BICUBIC, H, W)

        f16 = pk.get("f16")
        # (fp16 operand plan: pixel stride 64 with zero pad floats, so the same buffer is the 64-channel residual of gf2)
        shallow64 = buf("shallow64", H, W, 64) if f16 else None
        shallow = shallow64[..., 0:CP] if f16 else buf("shallow", H, W, CP)
        # fp16 copy of the whole trunk (64-half pixels), written by the stem / the SA tail of the previous stage: channels 0..31 feed
        # the spatial branch's tensor-core convs, 40..57 the all-MMA EPI kernel
        epi_mma = bool(f16) and pk["stages"][0].get("epi_img") is not None
        trunk16 = self._buf16("trunk16", B, H, W, 64, dev) if epi_mma else None
        if epi_mma:
            ops.conv(xin, pk["stem"], shallow, out16=trunk16[..., 0:CP])      # (the stem kernel writes the copy itself)
        else:
            ops.conv(xin, pk["stem"], shallow)
        feat = shallow
        pp = [buf("feat_a", H, W, CP), buf("feat_b", H, W, CP)]
        hA, wA = H // A, W // A
        cat = buf("cat", H, W, CP)
        t18 = buf("t18", H, W, gs)                 # c0 real channels + zero pad, written whole by spa0
        hid = pk["stages"][0]["ang_hid"]
        ang1, ang4, ang5 = buf("ang1", hA, wA, gs), buf("ang4", hA, wA, gs), buf("ang5", hA, wA, gs)
        ang2, ang3 = buf("ang2", hA, wA, gs), buf("ang3", hA, wA, gs)
        vmean, gmean, gate = buf("vmean", A, A, CP), buf("gmean", 1, 1, CP), buf("gate", 1, 1, CP)
        CU = pk["CU"]
        # fu1 (fusion 1x1 output) feeds nothing but the 3x3 that follows: fp16 only on the fp16 operand plan
        fu1 = self._buf16("fu1", B, H, W, CU, dev) if f16 else buf("fu1", H, W, CU)
        fu2 = buf("fu2", H, W, CP)
        if f16:
            xs16 = trunk16[..., 0:32] if epi_mma else self._buf16("xs16", B, H, W, 32, dev)
            t18h = self._buf16("t18h", B, H, W, 32, dev)
        pm, am1, am = buf("pm", A, A, CP), buf("am1", A, A, C // 4), buf("am", A, A, CP)
        for i, st in enumerate(pk["stages"]):
            xs, xa, xe = feat[..., sl[0]], feat[..., sl[1]], feat[..., sl[2]]
            # spatial branch
            if f16:
                if i == 0:          # later stages: the SA modulator of the previous stage wrote the copy next to the trunk
                    if not epi_mma:
                        ops.to_f16(feat[..., 0:32], xs16)
                ops.conv(xs16, st["spa0h"], None, out16=t18h[..., 0:24], act=LR, slope=0.1)
                ops.conv(t18h, st["spa2h"], cat[..., 0:gs])
            else:
                ops.conv(xs, st["spa0"], t18, act=LR, slope=0.1)
                ops.conv(t18[..., 0:c0], st["spa2"], cat[..., 0:gs])
            # angular branch
            ops.conv(xa, st["ang_to"], ang1)
            ops.conv(ang1[..., 0:c0], st["ang_a0"], ang2, act=N.ACT_RELU)
            ops.dwconv(ang2, st["ang_a2"], ang3, 3, 3, act=N.ACT_RELU)
            ops.conv(ang3[..., 0:hid], st["ang_a4"], ang4, act=N.ACT_SIGMOID, mul=ang1)
            ops.conv(ang4[..., 0:c0], st["ang_cv"], ang5, act=LR, slope=0.1)
            ops.ang_expand(ang5[..., 0:c0], st["ang_exw"], feat[..., gs:2 * gs], cat[..., gs:2 * gs], A, LR, 0.1, st["ang_scale"])
            # EPI branch: three depthwise+pointwise paths and their fuse conv in one kernel
            if f16 and epi_mma:
                ops.mel_epi_branch_mma(xe, trunk16[..., 2 * gs:2 * gs + sp[2]], st["epi_img"], cat[..., sl[2]], st["epi_klen"], A, 0.1)
            else:
                ops.mel_epi_branch(xe, st["epi_w"], cat[..., sl[2]], st["epi_klen"], A, 0.1, tc=bool(f16))
            # gates -> per-sample channel scale of the fusion 1x1
            ops.block_mean(cat, vmean, hA, wA)
            ops.pooled_mlp(vmean, gate, st["gate"], N.ACT_SIGMOID, pool=True)      # mean over the views -> FC + sigmoid
            if f16:
                ops.conv(cat, st["fus0"], None, out16=fu1, act=LR, slope=0.1, in_scale=gate)
            else:
                ops.conv(cat, st["fus0"], fu1, act=LR, slope=0.1, in_scale=gate)
            ops.conv(fu1[..., 0:C], st["fus2"], fu2)
            # SA modulator + stage residual
            ops.block_mean(fu2, pm, hA, wA)
            ops.pooled_mlp(pm, am, st["sa_c0"], N.ACT_RELU, st["sa_c2"], N.ACT_SIGMOID)
            nxt = pp[i & 1]
            if f16 and i + 1 < len(pk["stages"]):
                ops.sa_modulate(fu2, st["sa_dw"], st["sa_bns"], st["sa_bnb"], am, st["sa_w"][0], st["sa_w"][1], feat, nxt, A,
                                out16=trunk16[..., 0:CP] if epi_mma else xs16)
                # (leaving the unread channels 20..39 out of the copy - skip16=(gs, 2 * gs) - was SLOWER, 0.397 vs 0.347 ms per
                # call: the copy then ends in 8- and 16-byte pieces of 32-byte sectors)
            else:
                ops.sa_modulate(fu2, st["sa_dw"], st["sa_bns"], st["sa_bnb"], am, st["sa_w"][0], st["sa_w"][1], feat, nxt, A)
            feat = nxt
        if f16:
            ops.conv(feat, pk["gf0"], None, out16=fu1, act=LR, slope=0.1)
        else:
            ops.conv(feat, pk["gf0"], fu1, act=LR, slope=0.1)
        if f16:
            # the trunk's last tensor feeds nothing but the first upsampler conv: written as fp16 only, so that layer runs on
            # kind::f16 operands like the second one
            fu2h = self._buf16("fu2h", B, H, W, 64, dev)
            ops.conv(fu1[..., 0:C], pk["gf2"], None, out16=fu2h, res=shallow64)
            upsample_tail(self, ops, pk, fu2h, H, W, Y, pk["CU"], LR, N.SHUF_CHANNEL_MAJOR)
        else:
            ops.conv(fu1[..., 0:C], pk["gf2"], fu2, res=shallow)
            upsample_tail(self, ops, pk, fu2, H, W, Y, pk["CU"], LR, N.SHUF_CHANNEL_MAJOR)

    # -- measurement hook --------------------------------------------------------------------------
    def dominant_kernel(self, batch: int, h: int = 32):
        """(callable, info) for the layer that dominates HBM bytes and FLOPs: the last upsampler
        conv 3x3 C->4C + PixelShuffle(2) + LReLU (MyEfficientLFNet.py:560-565): 55 % of the MACs,
        reads C x (2H)^2, writes C x (4H)^2 per patch. Used by bench.py's roofline entry."""
        dev = next(self.parameters()).device
        ops = K.default_ops()
        pk = self._get_packed(dev, ops)
        A, C = self.angRes, self.channels
        pcv, r = pk["up"][-1]
        hin = A * h * (self.scale // r)
        if len(pk["up"]) > 1:       # the previous upsampler stage's activation: fp16 on the fp16 operand plan
            mk = self._buf16 if (pk.get("f16") and pcv.w_tc16 is not None) else self._buf
            src = mk(f"up{len(pk['up']) - 2}", batch, hin, hin, pcv.cin, dev)
        else:
            src = self._buf("fu2", batch, hin, hin, pcv.cin, dev)
        shuffle = (r, r, N.SHUF_CHANNEL_MAJOR)
        # (per-layer bytes as SURVEY 8d counts them: fp32 in + out + weights of the real 54 / 216-channel layer)
        conv_bytes = batch * (hin * hin * C + hin * r * hin * r * C) * 4 + pcv.kh * pcv.kw * C * C * r * r * 4
        f16_in = src.dtype == torch.float16
        info = {
            "ncu_json": "r02_dominant_kernel_ncu.json" if f16_in else "r01_dominant_kernel_ncu.json",
            "name": "conv3x3 %d->%d + PixelShuffle(%d) + LReLU @%dx%d (upsampler.up.%s)" % (C, C * r * r, r, hin, hin,
                                                                                        self.upsampler.steps[-1][0]),
            # algorithmic figures use the reference layer's real 54 -> 216 channels, not the padded buffers
            "bytes": conv_bytes,
            "flops": 2 * batch * hin * hin * pcv.kh * pcv.kw * C * C * r * r,
        }
        if pk.get("tail_w") is not None and ops.tail_supported(pcv, pk["CU"], shuffle):
            # the forward runs this layer with the head conv's channel contraction in its epilogue (common.upsample_tail):
            # per-layer bytes of what the kernel covers = this layer + the head conv's input read and weights
            dst = self._buf("head_taps", batch, hin * r, hin * r, 9, dev)
            info["name"] += " + 3x3 head-conv tap projection (output_conv) fused in the epilogue"
            info["bytes_conv_layer_only"] = conv_bytes
            info["bytes"] = conv_bytes + batch * hin * r * hin * r * C * 4 + 9 * C * 4
            info["flops"] += 2 * batch * hin * r * hin * r * 9 * C
            tail = (pk["tail_w"], 9, pk["CU"])
            return (lambda: ops.conv(src, pcv, dst, act=N.ACT_LRELU, slope=0.1, shuffle=shuffle, tail=tail)), info
        dst = self._buf(f"up{len(pk['up']) - 1}", batch, hin * r, hin * r, pk["CU"], dev)
        return (lambda: ops.conv(src, pcv, dst, act=N.ACT_LRELU, slope=0.1, shuffle=shuffle)), info


class get_loss(nn.Module):
    """L1 + 0.05 * L1 of rFFT magnitudes (MyEfficientLFNet.py:585-609); training only."""

    def __init__(self, args=None):
        super().__init__()
        self.l1_loss = nn.L1Loss()
        self.use_freq = True
        self.freq_weight = 0.05

    def forward(self, SR, HR, criterion_data=None):
        loss = self.l1_loss(SR, HR)
        if self.use_freq:
            loss = loss + self.freq_weight * nn.functional.l1_loss(torch.fft.rfft2(SR).abs(), torch.fft.rfft2(HR).abs())
        return loss


def weights_init(m):
    """Kaiming-normal (a=0.1, fan_in) on conv/linear, unit BatchNorm (MyEfficientLFNet.py:612-624)."""
    if isinstance(m, (nn.Conv2d, nn.Linear)):
        nn.init.kaiming_normal_(m.weight, a=0.1, mode="fan_in", nonlinearity="leaky_relu")
        if m.bias is not None:
            nn.init.zeros_(m.bias)
    elif isinstance(m, nn.BatchNorm2d):
        nn.init.ones_(m.weight)
        nn.init.zeros_(m.bias)
