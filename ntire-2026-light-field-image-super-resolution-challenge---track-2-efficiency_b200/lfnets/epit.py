"""EPIT on liblfsr_b200 kernels - mirror of /root/reference/model/SR/EPIT.py.

All features stay in ONE layout, the SAI mosaic as NHWC fp32 [B, A*h, A*w, 64]:
  * the per-view Conv3d(1,3,3) stacks (:24-31, :138-143) are 3x3 convs with view blocking (taps that
    leave the output pixel's view read zero);
  * the token tensor of BasicTrans (:113) is the same memory viewed as [T, 64]; the four einops
    permute-copies per AltFilter (:150-159) become stride sets of the attention kernel: the
    horizontal pass runs sequences over (u, h) for fixed (b, v, w), the vertical pass over (v, w)
    for fixed (b, u, h);
  * the 160x160 additive mask that the reference rebuilds on the CPU ten times per forward
    (:93-108, :112) is never materialised: mask_field = [2A, 11] allows every angular row and
    |s - s'| <= 5 along the spatial axis, which the kernel evaluates analytically.
BasicTrans (:110-128): linear_in 64->128; LN; Q,K from LN(x), V from x (:117-122), 8 heads x 16, no
biases; out_proj + x; LN; 128->256 ReLU 256->128 + x; linear_out 128->64. Linears run as 1x1 convs.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import _native as N
from .. import kernels as K
from .common import LFNetBase, L1Loss, slots, tail_table


def _c3(cin, cout):
    return nn.Conv3d(cin, cout, kernel_size=(1, 3, 3), padding=(0, 1, 1), bias=False)


class _BasicTrans(nn.Module):
    def __init__(self, channels, spa_dim, num_heads=8):
        super().__init__()
        self.num_heads = num_heads
        self.linear_in = nn.Linear(channels, spa_dim, bias=False)
        self.norm = nn.LayerNorm(spa_dim)
        self.attention = nn.MultiheadAttention(spa_dim, num_heads, 0.0, bias=False)
        nn.init.kaiming_uniform_(self.attention.in_proj_weight, a=math.sqrt(5))
        self.feed_forward = slots({0: nn.LayerNorm(spa_dim), 1: nn.Linear(spa_dim, spa_dim * 2, bias=False),
                                   4: nn.Linear(spa_dim * 2, spa_dim, bias=False)})
        self.linear_out = nn.Linear(spa_dim, channels, bias=False)


class _AltFilter(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.epi_trans = _BasicTrans(channels, channels * 2)
        self.conv = slots({0: _c3(channels, channels), 2: _c3(channels, channels), 4: _c3(channels, channels)})


class get_model(LFNetBase):
    def __init__(self, args):
        super().__init__(args)
        ch = 64
        self.channels = ch
        if self.angRes > 5:
            raise N.LfsrError("EPIT: the analytic mask assumes mask_field[0] = 2A covers all A rows (A <= 5)")
        self.conv_init0 = slots({0: _c3(1, ch)})
        self.conv_init = slots({0: _c3(ch, ch), 2: _c3(ch, ch), 4: _c3(ch, ch)})
        self.altblock = nn.ModuleList([_AltFilter(ch) for _ in range(5)])
        self.upsampling = slots({0: nn.Conv2d(ch, ch * self.scale ** 2, 1, bias=False),
                                 3: nn.Conv2d(ch, 1, 3, padding=1, bias=False)})

    def _pack(self, device, ops):
        from . import common
        f16 = bool(common.USE_FP16_OPERANDS and hasattr(ops, "to_f16") and hasattr(ops, "pack_basictrans") and
                   getattr(ops, "fp16_operands", getattr(ops, "use_tc", False)))
        pc = lambda w, b=None, **kw: K.pack_conv(w, b, device=device, **kw)
        c3 = lambda m: pc(m.weight[:, :, 0], pad=(1, 1), tc=True, tc16=f16)          # [co, ci, 1, 3, 3] -> 2-D 3x3
        lin = lambda w: pc(w.reshape(w.shape[0], w.shape[1], 1, 1), tc=True)
        vec = lambda t: t.detach().to(device=device, dtype=torch.float32).contiguous()
        pk = {"f16": f16, "init0": pc(self.conv_init0["0"].weight[:, :, 0], pad=(1, 1)),
              "init": [c3(self.conv_init[k]) for k in ("0", "2", "4")], "alt": []}
        for af in self.altblock:
            t = af.epi_trans
            E = t.norm.weight.numel()
            ipw = t.attention.in_proj_weight
            # the whole BasicTrans as one tcgen05 kernel (lfsr_epit_basictrans) when the backend has it
            bt = None
            if f16:
                bt = ops.pack_basictrans(t.linear_in.weight, ipw, t.attention.out_proj.weight, t.feed_forward["1"].weight,
                                         t.feed_forward["4"].weight, t.linear_out.weight,
                                         (t.norm.weight, t.norm.bias, t.norm.eps),
                                         (t.feed_forward["0"].weight, t.feed_forward["0"].bias, t.feed_forward["0"].eps),
                                         t.num_heads, device)
            pk["alt"].append(dict(
                bt=bt, lin_in=lin(t.linear_in.weight), ln1=(vec(t.norm.weight), vec(t.norm.bias), t.norm.eps),
                wqk=lin(ipw[:2 * E]), wv=lin(ipw[2 * E:]), wo=lin(t.attention.out_proj.weight),
                ln2=(vec(t.feed_forward["0"].weight), vec(t.feed_forward["0"].bias), t.feed_forward["0"].eps),
                ff1=lin(t.feed_forward["1"].weight), ff2=lin(t.feed_forward["4"].weight), lin_out=lin(t.linear_out.weight),
                conv=[c3(af.conv[k]) for k in ("0", "2", "4")], heads=t.num_heads, E=E))
        pk["up0"] = pc(self.upsampling["0"].weight, tc=True, tc16=f16, tc_shuffle=(self.scale, self.scale, N.SHUF_CHANNEL_MAJOR))
        pk["up3"] = pc(self.upsampling["3"].weight, pad=(1, 1), tc=True)
        pk["tail_w"] = tail_table(self.upsampling["3"].weight, self.channels, device)
        return pk

    def _run16(self, ops, pk, x, out):
        """fp16 operand plan: the feature trunk (`cur`, residual of every AltFilter pass) stays fp32 and carries an fp16 copy;
        the fused BasicTrans reads that copy and writes fp16 tokens; the two inner convolutions of each pass exchange fp16
        only. Geometries the fused kernel does not take fall back to the separate launches on the fp32 trunk."""
        A, s, C = self.angRes, self.scale, self.channels
        B, _, H, W = x.shape
        h, w = H // A, W // A
        dev = x.device
        buf = lambda name, hh, ww, c: self._buf(name, B, hh, ww, c, dev)
        b16 = lambda name, hh, ww, c: self._buf16(name, B, hh, ww, c, dev)
        LR = N.ACT_LRELU
        blk = (h, w)
        xin = x.view(B, H, W, 1)
        Y = out.view(B, H * s, W * s, 1)
        ops.interp(x, out, B, H, W, s, N.INTERP_BICUBIC, h, w)
        f0, f0h = buf("f0", H, W, C), b16("f0", H, W, C)
        t1h, t2h, ybh = b16("t1", H, W, C), b16("t2", H, W, C), b16("yb", H, W, C)
        fa, fah, fb = buf("fa", H, W, C), b16("fa", H, W, C), buf("fb", H, W, C)
        ops.conv(xin, pk["init0"], f0, out16=f0h, block=blk)             # the stem kernel writes the fp16 operand copy itself
        ops.conv(f0h, pk["init"][0], None, out16=t1h, act=LR, slope=0.2, block=blk)
        ops.conv(t1h, pk["init"][1], None, out16=t2h, act=LR, slope=0.2, block=blk)
        ops.conv(t2h, pk["init"][2], fa, out16=fah, act=LR, slope=0.2, res=f0, block=blk)
        hw_img = H * W
        passes = [
            dict(A=A, S=h, stride_a=h * W, stride_s=W, stride_b=hw_img, stride_p=w, stride_q=1, np_=A, nq=w),
            dict(A=A, S=w, stride_a=w, stride_s=1, stride_b=hw_img, stride_p=h * W, stride_q=W, np_=A, nq=h),
        ]
        ring = [(buf(f"r{i}", H, W, C), b16(f"r{i}", H, W, C)) for i in range(3)]
        cur, ri = (fa, fah), 0
        for al in pk["alt"]:
            short = cur[0]
            for p in passes:
                if not ops.basictrans(cur[1], al["bt"][0], al["bt"][1], ybh, p["A"], p["S"], 5, B, p["np_"], p["nq"], p["stride_a"],
                                      p["stride_s"], p["stride_b"], p["stride_p"], p["stride_q"]):
                    self._basictrans_unfused(ops, al, cur[0], p, B, H, W)
                    ops.to_f16(self._buf("yb", B, H, W, C, dev), ybh)
                ops.conv(ybh, al["conv"][0], None, out16=t1h, act=LR, slope=0.2, block=blk)
                ops.conv(t1h, al["conv"][1], None, out16=t2h, act=LR, slope=0.2, block=blk)
                nxt = ring[ri]
                ri = (ri + 1) % 3
                if nxt[0] is short:
                    nxt = ring[ri]
                    ri = (ri + 1) % 3
                ops.conv(t2h, al["conv"][2], nxt[0], out16=nxt[1], res=short, block=blk)
                cur = nxt
        # altblock(buffer) + buffer (:64): the last AltFilter already consumed its own shortcut as the fused residual; this
        # second skip is an exact fp32 add on the elementwise kernel
        # (fb feeds nothing but the upsampling conv: written as fp16 only, that conv then runs on kind::f16 operands)
        if pk["up0"].w_tc16 is not None:
            fbh = self._buf16("fbh", B, H, W, C, dev)
            ops.scale_add(cur[0], self._ones(pk, B, dev), fa, None, out16=fbh)
            self._head(ops, pk, fbh, Y, B, H, W)
        else:
            ops.scale_add(cur[0], self._ones(pk, B, dev), fa, fb)
            self._head(ops, pk, fb, Y, B, H, W)

    def _basictrans_unfused(self, ops, al, cur, p, B, H, W):
        """BasicTrans as separate launches on the fp32 trunk -> the fp32 token buffer "yb" (EPIT.py:110-128)"""
        A, C = self.angRes, self.channels
        dev = cur.device
        E = al["E"]
        buf = lambda name, c: self._buf(name, B, H, W, c, dev)
        T = B * H * W
        tok = lambda t: t.view(1, 1, T, t.shape[3])
        X, Nn, Ao, X2 = buf("X", E), buf("Nn", E), buf("Ao", E), buf("X2", E)
        QK, F1, Vv, yb = buf("QK", 2 * E), buf("F1", 2 * E), buf("V", E), buf("yb", C)
        ops.conv(tok(cur), al["lin_in"], tok(X))
        ops.layernorm(tok(X), al["ln1"][0], al["ln1"][1], al["ln1"][2], tok(Nn))
        ops.conv(tok(Nn), al["wqk"], tok(QK))
        ops.conv(tok(X), al["wv"], tok(Vv))
        ops.epi_attention(QK, Vv, Ao, al["heads"], E // al["heads"], p["A"], p["S"], 5, B, p["np_"], p["nq"],
                          p["stride_a"], p["stride_s"], p["stride_b"], p["stride_p"], p["stride_q"])
        ops.conv(tok(Ao), al["wo"], tok(X2), res=tok(X))
        ops.layernorm(tok(X2), al["ln2"][0], al["ln2"][1], al["ln2"][2], tok(Nn))
        ops.conv(tok(Nn), al["ff1"], tok(F1), act=N.ACT_RELU)
        ops.conv(tok(F1), al["ff2"], tok(X), res=tok(X2))
        ops.conv(tok(X), al["lin_out"], tok(yb))

    def _head(self, ops, pk, fb, Y, B, H, W):
        A, s, C = self.angRes, self.scale, self.channels
        LR = N.ACT_LRELU
        dev = fb.device
        shuffle = (s, s, N.SHUF_CHANNEL_MAJOR)
        if ops.tail_supported(pk["up0"], C, shuffle):
            taps = self._buf("head_taps", B, H * s, W * s, 9, dev)
            ops.conv(fb, pk["up0"], taps, act=LR, slope=0.2, shuffle=shuffle, tail=(pk["tail_w"], 9, C))
            ops.tap_gather(taps, 3, 3, None, Y, Y)
        else:
            up = self._buf("up", B, H * s, W * s, C, dev)
            ops.conv(fb, pk["up0"], up, act=LR, slope=0.2, shuffle=shuffle)
            ops.conv(up, pk["up3"], Y, res=Y)

    def _run(self, ops, pk, x, out):
        if pk.get("f16"):
            return self._run16(ops, pk, x, out)
        A, s, C = self.angRes, self.scale, self.channels
        B, _, H, W = x.shape
        h, w = H // A, W // A
        dev = x.device
        buf = lambda name, hh, ww, c: self._buf(name, B, hh, ww, c, dev)
        LR = N.ACT_LRELU
        blk = (h, w)
        xin = x.view(B, H, W, 1)
        Y = out.view(B, H * s, W * s, 1)
        ops.interp(x, out, B, H, W, s, N.INTERP_BICUBIC, h, w)                 # per view (:164-169)
        f0, t1, t2 = buf("f0", H, W, C), buf("t1", H, W, C), buf("t2", H, W, C)
        fa, fb = buf("fa", H, W, C), buf("fb", H, W, C)
        ops.conv(xin, pk["init0"], f0, block=blk)
        ops.conv(f0, pk["init"][0], t1, act=LR, slope=0.2, block=blk)
        ops.conv(t1, pk["init"][1], t2, act=LR, slope=0.2, block=blk)
        ops.conv(t2, pk["init"][2], fa, act=LR, slope=0.2, res=f0, block=blk)   # conv_init(buffer) + buffer
        E = pk["alt"][0]["E"]
        T = B * H * W
        tok = lambda t: t.view(1, 1, T, t.shape[3])        # 64/128/256-channel buffers are dense: tokens = pixels
        X, Nn, Ao, X2 = buf("X", H, W, E), buf("Nn", H, W, E), buf("Ao", H, W, E), buf("X2", H, W, E)
        QK, F1 = buf("QK", H, W, 2 * E), buf("F1", H, W, 2 * E)
        Vv = buf("V", H, W, E)
        yb = buf("yb", H, W, C)
        hw_img = H * W
        passes = [  # (A, S, strides a, s, b, p, q, np, nq)
            dict(A=A, S=h, stride_a=h * W, stride_s=W, stride_b=hw_img, stride_p=w, stride_q=1, np_=A, nq=w),    # (u,h)|(v,w)
            dict(A=A, S=w, stride_a=w, stride_s=1, stride_b=hw_img, stride_p=h * W, stride_q=W, np_=A, nq=h),    # (v,w)|(u,h)
        ]
        cur = fa
        ring = [buf("r0", H, W, C), buf("r1", H, W, C), buf("r2", H, W, C)]
        state = {"ri": 0, "cur": fa}
        for al in pk["alt"]:
            short = cur
            for p in passes:
                ops.conv(tok(cur), al["lin_in"], tok(X))
                ops.layernorm(tok(X), al["ln1"][0], al["ln1"][1], al["ln1"][2], tok(Nn))
                ops.conv(tok(Nn), al["wqk"], tok(QK))
                ops.conv(tok(X), al["wv"], tok(Vv))
                ops.epi_attention(QK, Vv, Ao, al["heads"], E // al["heads"], p["A"], p["S"], 5, B, p["np_"], p["nq"],
                                  p["stride_a"], p["stride_s"], p["stride_b"], p["stride_p"], p["stride_q"])
                ops.conv(tok(Ao), al["wo"], tok(X2), res=tok(X))
                ops.layernorm(tok(X2), al["ln2"][0], al["ln2"][1], al["ln2"][2], tok(Nn))
                ops.conv(tok(Nn), al["ff1"], tok(F1), act=N.ACT_RELU)
                ops.conv(tok(F1), al["ff2"], tok(X), res=tok(X2))
                ops.conv(tok(X), al["lin_out"], tok(yb))
                self._conv_tail(ops, al, yb, t1, t2, ring, short, blk, LR, state)
                cur = state["cur"]
        # altblock(buffer) + buffer (:64): the last AltFilter already consumed its own shortcut as the
        # fused residual, so this second skip is an exact fp32 add on the elementwise kernel
        ops.scale_add(cur, self._ones(pk, B, dev), fa, fb)
        shuffle = (s, s, N.SHUF_CHANNEL_MAJOR)
        if ops.tail_supported(pk["up0"], C, shuffle):
            # 1x1 C -> C*s^2 + PixelShuffle + LReLU with the 3x3 head conv's channel contraction in its epilogue, then the
            # 9-tap gather onto the bicubic skip (EPIT.py:45-48, :64-66): the C-channel HR activation is never written
            taps = buf("head_taps", H * s, W * s, 9)
            ops.conv(fb, pk["up0"], taps, act=LR, slope=0.2, shuffle=shuffle, tail=(pk["tail_w"], 9, C))
            ops.tap_gather(taps, 3, 3, None, Y, Y)
        else:
            up = buf("up", H * s, W * s, C)
            ops.conv(fb, pk["up0"], up, act=LR, slope=0.2, shuffle=shuffle)
            ops.conv(up, pk["up3"], Y, res=Y)

    @staticmethod
    def _conv_tail(ops, al, yb, t1, t2, ring, short, blk, LR, state):
        """the three per-view convs + shortcut that follow BasicTrans in AltFilter (EPIT.py:152-153, :160-161)"""
        ops.conv(yb, al["conv"][0], t1, act=LR, slope=0.2, block=blk)
        ops.conv(t1, al["conv"][1], t2, act=LR, slope=0.2, block=blk)
        ri = state["ri"]
        nxt = ring[ri]
        ri = (ri + 1) % 3
        if nxt is short:
            nxt = ring[ri]
            ri = (ri + 1) % 3
        ops.conv(t2, al["conv"][2], nxt, res=short, block=blk)
        state["ri"], state["cur"] = ri, nxt

    def _ones(self, pk, B, dev):
        key = ("ones", B)
        if key not in pk:
            pk[key] = torch.ones((B, 1, 1, self.channels), dtype=torch.float32, device=dev)
        return pk[key]


get_loss = L1Loss


def weights_init(m):
    """EPIT.py:183-184: a no-op."""
    pass
