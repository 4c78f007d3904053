"""GPU parity of every C-ABI kernel against the torch statement of its contract (tests/opref.py)
and, for the bit-exact ones, against the numpy oracle and the committed reference goldens."""
import numpy as np
import pytest
import torch

import lfsr_b200
from lfsr_b200 import kernels as K
from lfsr_b200 import _native as N
from opref import RefOps
from oracle import lf_oracle, weights

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    return K.CudaOps(use_tc=False)


@pytest.fixture(scope="module")
def ref():
    return RefOps()


def rnd(*shape, seed=0, lo=-1.0, hi=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(*shape, generator=g) * (hi - lo) + lo).to(DEV)


def nhwc(n, h, w, c, seed=0, ld=None):
    ld = ld or K.ld_for(c)
    return rnd(n, h, w, ld, seed=seed)[..., :c]


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h0,w0", [(32, 32), (47, 61), (64, 40), (125, 125), (108, 156)])
def test_divide_integrate_bit_exact(ops, h0, w0):
    A, P, S, s = 5, 32, 16, 2
    scene = np.random.RandomState(h0 * 1000 + w0).random_sample((A * h0, A * w0)).astype(np.float32)
    want = lf_oracle.lfdivide(scene, A, P, S)
    got = lfsr_b200.lfutils.LFdivide(torch.from_numpy(scene).to(DEV), A, P, S)
    assert got.shape == want.shape
    assert np.array_equal(got.cpu().numpy(), want)
    # integrate on nearest-upsampled patches: integrate(up(divide(x))) == up(x)  (SURVEY 8c)
    up = got.view(*got.shape[:2], A, P, 1, A, P, 1).expand(-1, -1, -1, -1, s, -1, -1, s).reshape(
        got.shape[0], got.shape[1], A * P * s, A * P * s).contiguous()
    lf = lfsr_b200.lfutils.LFintegrate(up, A, P * s, S * s, h0 * s, w0 * s)
    want_i = lf_oracle.lfintegrate(up.cpu().numpy(), A, P * s, S * s, h0 * s, w0 * s)
    assert np.array_equal(lf.cpu().numpy(), want_i)
    views = scene.reshape(A, h0, A, w0).transpose(0, 2, 1, 3)
    assert np.array_equal(want_i, np.repeat(np.repeat(views, s, axis=2), s, axis=3))


@pytest.mark.parametrize("A,h0,w0,P,S,s", [(3, 20, 75, 32, 16, 4), (7, 23, 23, 32, 16, 2), (2, 40, 56, 64, 32, 2), (2, 12, 30, 16, 8, 3),
                                           (7, 33, 47, 32, 16, 1)])
def test_divide_integrate_edge_geometries(ops, A, h0, w0, P, S, s):
    """other angular resolutions / patch sizes and views smaller than a patch - bit-exact against the oracle; geometries
    the reference cannot tile (its unfold / rearrange raises: utils.py:160-164) raise here as well"""
    scene = np.random.RandomState(h0 * 131 + w0).random_sample((A * h0, A * w0)).astype(np.float32)
    want = lf_oracle.lfdivide(scene, A, P, S)
    got = lfsr_b200.lfutils.LFdivide(torch.from_numpy(scene).to(DEV), A, P, S)
    assert got.shape == want.shape and np.array_equal(got.cpu().numpy(), want)
    up = got.view(*got.shape[:2], A, P, 1, A, P, 1).expand(-1, -1, -1, -1, s, -1, -1, s).reshape(
        got.shape[0], got.shape[1], A * P * s, A * P * s).contiguous()
    lf = lfsr_b200.lfutils.LFintegrate(up, A, P * s, S * s, h0 * s, w0 * s)
    want_i = lf_oracle.lfintegrate(up.cpu().numpy(), A, P * s, S * s, h0 * s, w0 * s)
    assert lf.shape == want_i.shape and np.array_equal(lf.cpu().numpy(), want_i)
    for bad in ((40, 40, 16, 16), (17, 16, 32, 16)):
        with pytest.raises(ValueError):
            lfsr_b200.lfutils.LFdivide(torch.zeros(5 * bad[0], 5 * bad[1], device=DEV), 5, bad[2], bad[3])


def test_divide_integrate_goldens(ops):
    g = weights.load_pipeline_golden()
    for (h0, w0) in ((32, 32), (47, 61), (64, 40)):
        scene = g[f"div_{h0}x{w0}_scene"]
        got = lfsr_b200.lfutils.LFdivide(torch.from_numpy(scene).to(DEV), 5, 32, 16).cpu().numpy()
        assert tuple(g[f"div_{h0}x{w0}_shape"]) == got.shape
        assert np.array_equal(got[0, min(1, got.shape[1] - 1)], g[f"div_{h0}x{w0}_sub_u0v1"])
        assert np.array_equal(got[-1, -1], g[f"div_{h0}x{w0}_sub_last"])
        assert float(got.astype(np.float64).sum()) == float(g[f"div_{h0}x{w0}_sum"])
        up = np.repeat(np.repeat(got, 2, axis=2), 2, axis=3).reshape(got.shape[0], got.shape[1], 5, 32, 2, 5, 32, 2)
        up = np.ascontiguousarray(up).reshape(got.shape[0], got.shape[1], 320, 320)
        lf = lfsr_b200.lfutils.LFintegrate(torch.from_numpy(up).to(DEV), 5, 64, 32, h0 * 2, w0 * 2)
        assert np.array_equal(lf.cpu().numpy(), g[f"int_{h0}x{w0}_out"])


def test_divide_row_shards_and_6d(ops):
    A, P, S = 5, 32, 16
    scene = rnd(A * 70, A * 52, seed=5, lo=0.0)
    full = lfsr_b200.lfutils.LFdivide(scene, A, P, S)
    nu = full.shape[0]
    parts = [lfsr_b200.lfutils.LFdivide(scene, A, P, S, rows=(u, min(u + 2, nu))) for u in range(0, nu, 2)]
    assert torch.equal(torch.cat(parts, 0), full)
    six = full.view(nu, full.shape[1], A, P, A, P).permute(0, 1, 2, 4, 3, 5).contiguous()
    a = lfsr_b200.lfutils.LFintegrate(full, A, P, S, 70, 52)
    b = lfsr_b200.lfutils.LFintegrate(six, A, P, S, 70, 52)
    assert torch.equal(a, b)
    small = rnd(A * 10, A * 10)                                    # the reference's unfold finds no window here
    with pytest.raises(ValueError):
        lfsr_b200.lfutils.LFdivide(small, A, P, S)
    with pytest.raises(N.LfsrError):                               # ... and the C ABI refuses it by itself
        ops.divide_rows(small, torch.empty(1, 1, A * P, A * P, device=DEV), A, 10, 10, P, S, 0, 1)


@pytest.mark.parametrize("mode,block", [(0, None), (0, 8), (1, None)])
@pytest.mark.parametrize("scale", [2, 4])
def test_interp(ops, ref, mode, block, scale):
    n, h, w = 3, 40, 40
    x = rnd(n, 1, h, w, seed=1, lo=0.0)
    bh = block or h
    a = torch.empty(n, 1, h * scale, w * scale, device=DEV)
    b = torch.empty_like(a)
    ops.interp(x, a, n, h, w, scale, mode, bh, bh)
    ref.interp(x, b, n, h, w, scale, mode, bh, bh)
    assert (a - b).abs().max().item() <= 2e-6


CONV_CASES = [
    # cin cout kh kw stride dil pad extra
    dict(cin=1, cout=54, k=(3, 3), dil=(5, 5), pad=(5, 5), bias=True),
    dict(cin=1, cout=60, k=(3, 3), dil=(5, 5), pad=(5, 5), bias=True),              # stem, tiled kernel
    dict(cin=1, cout=64, k=(3, 3), pad=(1, 1), block=(8, 40), act=2),               # ... with view blocking (rows)
    dict(cin=1, cout=64, k=(3, 3), pad=(1, 1), block=(8, 8)),                       # ... blocks narrower than a tile: per-tap predicates
    dict(cin=18, cout=18, k=(3, 3), dil=(5, 5), pad=(5, 5), bias=True, act=2),
    dict(cin=18, cout=18, k=(5, 5), stride=(5, 5)),
    dict(cin=18, cout=16, k=(1, 1), act=1),
    dict(cin=16, cout=18, k=(1, 1), act=3, mul=True),
    dict(cin=18, cout=450, k=(1, 1), act=2, alpha=0.1, res=True, shuffle=(5, 5, 0)),
    dict(cin=54, cout=54, k=(1, 1), act=2, in_scale=True),
    dict(cin=54, cout=54, k=(3, 3), dil=(5, 5), pad=(5, 5), res=True, bias=True),
    dict(cin=54, cout=216, k=(3, 3), pad=(1, 1), act=2, shuffle=(2, 2, 0)),
    dict(cin=54, cout=1, k=(3, 3), pad=(1, 1), bias=True, res=True),
    dict(cin=64, cout=32, k=(1, 25), stride=(1, 5), pad=(0, 10), act=2),
    dict(cin=64, cout=32, k=(25, 1), stride=(5, 1), pad=(10, 0), act=2),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(1, 5, 1)),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(5, 1, 1)),
    dict(cin=1, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), in_perm=True),
    dict(cin=1, cout=64, k=(5, 5), stride=(5, 5), in_perm=True),
    dict(cin=64, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), res=True, out_perm=True),
    dict(cin=64, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), out_perm=True, shuffle=(2, 2, 0)),
    dict(cin=64, cout=64, k=(3, 3), pad=(1, 1), act=2, block=(8, 8)),
    dict(cin=144, cout=64, k=(1, 1), act=2),
    dict(cin=128, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=1, res=True),
    dict(cin=64, cout=128, k=(1, 1), act=4, bias=True),                 # FastConvSSM gate conv + GELU
    dict(cin=256, cout=64, k=(1, 1), mul=True, mul_act=5),              # ... fuse conv * silu(gate)
    dict(cin=64, cout=16, k=(1, 1), act=5),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_conv_f32(ops, ref, case):
    n, h, w = 2, 40, 40
    cin, cout = case["cin"], case["cout"]
    kh, kw = case["k"]
    stride, dil, pad = case.get("stride", (1, 1)), case.get("dil", (1, 1)), case.get("pad", (0, 0))
    g = torch.Generator().manual_seed(cin * 131 + cout)
    wt = (torch.rand(cout, cin, kh, kw, generator=g) - 0.5) * (2.0 / (cin * kh * kw) ** 0.5)
    bias = (torch.rand(cout, generator=g) - 0.5) if case.get("bias") else None
    pc = K.pack_conv(wt, bias, stride=stride, dil=dil, pad=pad, device=DEV)
    x = nhwc(n, h, w, cin, seed=3)
    oh = (h + 2 * pad[0] - dil[0] * (kh - 1) - 1) // stride[0] + 1
    ow = (w + 2 * pad[1] - dil[1] * (kw - 1) - 1) // stride[1] + 1
    ry, rx, sm = case.get("shuffle", (1, 1, 0))
    co = cout // (ry * rx)
    kw_args = dict(act=case.get("act", 0), slope=0.1, alpha=case.get("alpha", 1.0), shuffle=(ry, rx, sm),
                   block=case.get("block", (0, 0)))
    if case.get("mul"):
        kw_args["mul"] = nhwc(n, oh, ow, cout, seed=4)
        kw_args["mul_act"] = case.get("mul_act", 0)
    if case.get("res"):
        kw_args["res"] = nhwc(n, oh * ry, ow * rx, co, seed=5)
    if case.get("in_scale"):
        kw_args["in_scale"] = rnd(n, 1, 1, cin, seed=6, lo=0.0)
    if case.get("in_perm"):
        kw_args.update(in_perm=1, perm_a=5)
    if case.get("out_perm"):
        kw_args.update(out_perm=1, perm_a=5)
    a = nhwc(n, oh * ry, ow * rx, co, seed=7)
    b = a.clone()
    ops.conv(x, pc, a, **kw_args)
    ref.conv(x, pc, b, **kw_args)
    err = (a - b).abs().max().item()
    assert err <= 2e-5, f"max err {err}"


@pytest.mark.parametrize("cin,cout,act", [(64, 16, 0), (64, 8, 2), (60, 16, 0)])
def test_conv1x1_few(ops, ref, cin, cout, act):
    """fp32 1x1 conv to 8 / 16 channels (DistgSSR's reconstruction tail): exact fp32, odd pixel counts, strided views"""
    n, h, w = 3, 37, 45
    g = torch.Generator().manual_seed(cin + cout)
    pc = K.pack_conv((torch.rand(cout, cin, 1, 1, generator=g) - 0.5) * 0.3, torch.rand(cout, generator=g) - 0.5, device=DEV)
    xfull = nhwc(n, h, w, 64, seed=3)
    x = xfull[..., :cin]
    a, b = nhwc(n, h, w, cout, seed=7), nhwc(n, h, w, cout, seed=7)
    before = ops.lib.lfsr_launch_count()
    ops.conv(x, pc, a, act=act, slope=0.1)
    assert ops.lib.lfsr_launch_count() == before + 1
    ref.conv(x, pc, b, act=act, slope=0.1)
    assert (a - b).abs().max().item() <= 2e-5


@pytest.mark.parametrize("block", [(0, 0), (8, 40), (8, 8)])
def test_stem_with_fp16_copy(ops, ref, block):
    """1-channel stem that also writes the fp16 operand copy of its output (tiled kernel; blocks narrower than a tile fall back to
    stem + conversion): fp32 output unchanged, the copy is exactly its rounding, pad halves stay untouched"""
    n, h, w, cout = 2, 40, 40, 56
    g = torch.Generator().manual_seed(5)
    pad = (1, 1) if block != (0, 0) else (5, 5)
    pc = K.pack_conv((torch.rand(cout, 1, 3, 3, generator=g) - 0.5) * 0.6, torch.rand(cout, generator=g) - 0.5, dil=pad, pad=pad, device=DEV)
    x = nhwc(n, h, w, 1, seed=3)
    a, b = nhwc(n, h, w, 64, seed=7), nhwc(n, h, w, 64, seed=7)
    full16 = torch.full((n, h, w, 64), 3.0, dtype=torch.float16, device=DEV)
    ops.conv(x, pc, a[..., :cout], out16=full16[..., :cout], block=block)
    ref.conv(x, pc, b[..., :cout], block=block)
    assert (a - b).abs().max().item() <= 2e-5
    assert torch.equal(full16[..., :cout], a[..., :cout].half()) and bool((full16[..., cout:] == 3.0).all())


def test_conv_residual_in_place(ops, ref):
    n, h, w, c = 1, 24, 24, 54
    wt = (torch.rand(1, c, 3, 3) - 0.5) * 0.1
    pc = K.pack_conv(wt, torch.tensor([0.25]), pad=(1, 1), device=DEV)
    x = nhwc(n, h, w, c, seed=9)
    y = rnd(n, h, w, 1, seed=10)
    y2 = y.clone()
    ops.conv(x, pc, y, res=y)
    ref.conv(x, pc, y2, res=y2.clone())
    assert (y - y2).abs().max().item() <= 2e-5


@pytest.mark.parametrize("kh,kw,dil,c", [(1, 11, (1, 1), 18), (11, 1, (1, 1), 18), (3, 3, (5, 5), 18), (3, 3, (1, 1), 18),
                                         (7, 7, (1, 1), 64), (3, 3, (8, 8), 64), (3, 3, (4, 4), 64)])
def test_dwconv(ops, ref, kh, kw, dil, c):
    n, h, w = 2, 40, 40
    x = nhwc(n, h, w, c, seed=1)
    wt = rnd(kh * kw, c, seed=2)
    sc, sh = rnd(c, seed=3, lo=0.5, hi=1.5), rnd(c, seed=4)
    for scale, shift, act in ((None, None, 0), (sc, sh, 3), (None, None, 1)):
        a, b = nhwc(n, h, w, c, seed=5), nhwc(n, h, w, c, seed=5)
        ops.dwconv(x, wt, a, kh, kw, dil, scale, shift, act, 0.1)
        ref.dwconv(x, wt, b, kh, kw, dil, scale, shift, act, 0.1)
        assert (a - b).abs().max().item() <= 1e-5


@pytest.mark.parametrize("h,w", [(40, 40), (37, 53), (160, 160)])
def test_dwconv_multi(ops, ref, h, w):
    """MultiScaleSpatial's sliced 1/3/5/7 branches and FastConvSSM's four dilations of the y half of [gate | y]
    (MyEfficientLFNetV4_5.py:218-221, :268-280), including tiles that overhang the image"""
    n, C, c = 2, 64, 16
    x = nhwc(n, h, w, C, seed=1)
    br = [dict(w=torch.ones(1, c, device=DEV), kh=1, kw=1, in_c0=0, out_c0=0, c=c)]
    for j, k in enumerate((3, 5, 7), 1):
        br.append(dict(w=rnd(k * k, c, seed=10 + j), kh=k, kw=k, in_c0=j * c, out_c0=j * c, c=c))
    a, b = nhwc(n, h, w, C, seed=2), nhwc(n, h, w, C, seed=2)
    l0 = ops.lib.lfsr_launch_count()
    ops.dwconv_multi(x, a, br)
    assert ops.lib.lfsr_launch_count() == l0 + 1
    ref.dwconv_multi(x, b, br)
    assert (a - b).abs().max().item() <= 1e-5
    g = nhwc(n, h, w, 2 * C, seed=3)
    br = [dict(w=rnd(9, C, seed=20 + k), kh=3, kw=3, dil=(d, d), in_c0=C, out_c0=k * C, c=C, act=(2 if k == 1 else 0), slope=0.1,
               scale=(rnd(C, seed=30, lo=0.5, hi=1.5) if k == 2 else None), shift=(rnd(C, seed=31) if k == 2 else None))
          for k, d in enumerate((1, 2, 4, 8))]
    a, b = nhwc(n, h, w, 4 * C, seed=4), nhwc(n, h, w, 4 * C, seed=4)
    ops.dwconv_multi(g, a, br)
    ref.dwconv_multi(g, b, br)
    assert (a - b).abs().max().item() <= 1e-5


@pytest.mark.parametrize("h,w,c,bh,bw", [(40, 40, 54, 8, 8), (5, 5, 54, 5, 5), (160, 160, 54, 32, 32), (20, 30, 130, 4, 5)])
def test_block_mean(ops, ref, h, w, c, bh, bw):
    x = nhwc(3, h, w, c, seed=1)
    a, b = nhwc(3, h // bh, w // bw, c, seed=2), nhwc(3, h // bh, w // bw, c, seed=2)
    ops.block_mean(x, a, bh, bw)
    ref.block_mean(x, b, bh, bw)
    assert (a - b).abs().max().item() <= 1e-5


@pytest.mark.parametrize("n,h,w,cin,with_res", [(2, 8, 8, 18, True), (3, 32, 32, 18, True), (2, 7, 9, 20, False), (2, 8, 8, 16, True)])
def test_ang_expand(ops, ref, n, h, w, cin, with_res):
    """AngularAttention.expand + PixelShuffle(5) + LReLU * alpha + residual as one streaming kernel, and == the conv path"""
    A, cq = 5, 20
    full = nhwc(n, h, w, 20, seed=1)
    x = full[..., :cin]
    wts = rnd(A, A, cin, cq, seed=2) * 0.3
    trunk = nhwc(n, h * A, w * A, 60, seed=3)
    a_full, b_full = nhwc(n, h * A, w * A, 60, seed=4), nhwc(n, h * A, w * A, 60, seed=4)
    res = trunk[..., 20:40] if with_res else None
    ops.ang_expand(x, wts, res, a_full[..., 20:40], A, N.ACT_LRELU, 0.1, 0.37)
    ref.ang_expand(x, wts, res, b_full[..., 20:40], A, N.ACT_LRELU, 0.1, 0.37)
    assert (a_full - b_full).abs().max().item() <= 2e-5
    assert torch.equal(a_full[..., 40:], b_full[..., 40:]) and torch.equal(a_full[..., :20], b_full[..., :20])
    if cin == 18 and with_res:       # the conv formulation of the same layer (nn.PixelShuffle channel order)
        wc = wts.permute(3, 0, 1, 2).reshape(cq * A * A, cin, 1, 1).cpu()
        pc = K.pack_conv(wc, device=DEV)
        c_full = nhwc(n, h * A, w * A, 60, seed=4)
        ref.conv(x, pc, c_full[..., 20:40], act=N.ACT_LRELU, slope=0.1, alpha=0.37, res=res, shuffle=(A, A, N.SHUF_CHANNEL_MAJOR))
        assert (a_full - c_full).abs().max().item() <= 2e-5


@pytest.mark.parametrize("pool,two", [(True, False), (False, True), (True, True), (False, False)])
def test_pooled_mlp(ops, ref, pool, two):
    """the stage gates (pooled, one layer + bias) and the SA modulator's angular MLP (two layers) as one launch each"""
    n, A, c, hid = 5, 5, 60, 13
    full = nhwc(n, A, A, 64, seed=1)
    x = full[..., :c]
    g = torch.Generator().manual_seed(3)
    pc1 = K.pack_conv((torch.rand(hid if two else c, c, 1, 1, generator=g) - 0.5) * 0.5,
                      None if two else torch.rand(c, generator=g) - 0.5, device=DEV)
    pc2 = K.pack_conv((torch.rand(c, hid, 1, 1, generator=g) - 0.5) * 0.5, None, device=DEV) if two else None
    shape = (n, 1, 1, c) if pool else (n, A, A, c)
    a, b = nhwc(*shape, seed=2), nhwc(*shape, seed=2)
    ops.pooled_mlp(x, a, pc1, N.ACT_RELU if two else N.ACT_SIGMOID, pc2, N.ACT_SIGMOID, pool=pool)
    ref.pooled_mlp(x, b, pc1, N.ACT_RELU if two else N.ACT_SIGMOID, pc2, N.ACT_SIGMOID, pool=pool)
    assert (a - b).abs().max().item() <= 2e-6


@pytest.mark.parametrize("c,h,w", [(54, 40, 40), (60, 40, 40), (60, 45, 35), (64, 160, 160)])
def test_sa_modulate(ops, ref, c, h, w):
    n, A = 2, 5
    x, res = nhwc(n, h, w, c, seed=1), nhwc(n, h, w, c, seed=2)
    dw, bs, bb = rnd(9, c, seed=3), rnd(c, seed=4, lo=0.5, hi=1.5), rnd(c, seed=5)
    am = nhwc(n, A, A, c, seed=6)
    a, b = nhwc(n, h, w, c, seed=7), nhwc(n, h, w, c, seed=7)
    ops.sa_modulate(x, dw, bs, bb, am, 0.4, 0.6, res, a, A)
    ref.sa_modulate(x, dw, bs, bb, am, 0.4, 0.6, res, b, A)
    assert (a - b).abs().max().item() <= 1e-5


@pytest.mark.parametrize("c,c16,h,w", [(60, 32, 40, 40), (60, 20, 45, 35), (64, 64, 160, 160)])
def test_sa_modulate_with_fp16_copy(ops, ref, c, c16, h, w):
    """the SA tail also stores the first c16 output channels as fp16 (operand of the next stage's spatial-branch convs):
    the copy is exactly the rounded fp32 output, pad channels of the fp16 buffer stay untouched"""
    n, A = 2, 5
    x, res = nhwc(n, h, w, c, seed=1), nhwc(n, h, w, c, seed=2)
    dw, bs, bb = rnd(9, c, seed=3), rnd(c, seed=4, lo=0.5, hi=1.5), rnd(c, seed=5)
    am = nhwc(n, A, A, c, seed=6)
    a, b = nhwc(n, h, w, c, seed=7), nhwc(n, h, w, c, seed=7)
    full16 = torch.full((n, h, w, 64), 3.0, dtype=torch.float16, device=DEV)
    ops.sa_modulate(x, dw, bs, bb, am, 0.4, 0.6, res, a, A, out16=full16[..., :c16])
    ref.sa_modulate(x, dw, bs, bb, am, 0.4, 0.6, res, b, A)
    assert (a - b).abs().max().item() <= 1e-5
    assert torch.equal(full16[..., :c16], a[..., :c16].half())
    assert bool((full16[..., c16:] == 3.0).all())
    # a skipped channel window stays untouched as well
    full16.fill_(3.0)
    ops.sa_modulate(x, dw, bs, bb, am, 0.4, 0.6, res, a, A, out16=full16[..., :c16], skip16=(8, 16))
    assert torch.equal(full16[..., :8], a[..., :8].half()) and torch.equal(full16[..., 16:c16], a[..., 16:c16].half())
    assert bool((full16[..., 8:16] == 3.0).all()) and bool((full16[..., c16:] == 3.0).all())


@pytest.mark.parametrize("r", [2, 4])
@pytest.mark.parametrize("accumulate", [False, True])
def test_macpi_unshuffle_bit_exact(ops, ref, r, accumulate):
    """MacPI2SAI + PixelShuffle(r) of the reconstruction (LF_InterNet.py:150-158, DistgSSR.py:42-46): pure index work"""
    n, A, h = 3, 5, 8
    x = nhwc(n, A * h, A * h, r * r, seed=5)
    a = torch.randn(n, 1, A * h * r, A * h * r, device="cuda")
    b = a.clone()
    ops.macpi_unshuffle(x, a, A, r, accumulate)
    ref.macpi_unshuffle(x, b, A, r, accumulate)
    assert torch.equal(a, b)


def test_split_tf32_exact(ops, ref):
    """hi is TF32-representable, hi + lo == x exactly, and both match the integer restatement"""
    x = torch.randn(5, 8, 8, 64, device="cuda") * torch.logspace(-6, 3, 64, device="cuda")
    hi, lo, hr, lr = (torch.empty_like(x) for _ in range(4))
    ops.split_tf32(x, hi, lo)
    ref.split_tf32(x, hr, lr)
    assert torch.equal(hi, hr) and torch.equal(lo, lr)
    assert torch.equal(hi + lo, x)
    assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0


@pytest.mark.parametrize("c,sliced,with_res", [(64, False, True), (64, True, True), (54, False, False), (18, True, True)])
def test_scale_add(ops, ref, c, sliced, with_res):
    """out = x * scale[n, c] + res (ChannelAttention + block residual, MyEfficientLFNetV4_5.py:147-148, :297-299)"""
    n, h, w = 3, 40, 40
    x = nhwc(n, h, w, c, seed=1)
    sc = nhwc(n, 1, 1, c, seed=2)
    res = nhwc(n, h, w, 4 * c, seed=3)[..., c:2 * c] if sliced else nhwc(n, h, w, c, seed=3)
    res = res if with_res else None
    fa, fb = nhwc(n, h, w, 4 * c, seed=4), nhwc(n, h, w, 4 * c, seed=4)
    a, b = (fa[..., 2 * c:3 * c], fb[..., 2 * c:3 * c]) if sliced else (fa[..., :c], fb[..., :c])
    ops.scale_add(x, sc, res, a)
    ref.scale_add(x, sc, res, b)
    assert torch.equal(fa, fb) or (fa - fb).abs().max().item() <= 1e-6


def test_layernorm(ops, ref):
    x = nhwc(1, 1, 5000, 128, seed=1)
    g, bta = rnd(128, seed=2, lo=0.5, hi=1.5), rnd(128, seed=3)
    a, b = nhwc(1, 1, 5000, 128, seed=4), nhwc(1, 1, 5000, 128, seed=4)
    ops.layernorm(x, g, bta, 1e-5, a)
    ref.layernorm(x, g, bta, 1e-5, b)
    assert (a - b).abs().max().item() <= 2e-5


@pytest.mark.parametrize("direction", ["h", "v"])
def test_epi_attention(ops, ref, direction):
    B, A, S, E, heads = 2, 5, 8, 128, 8
    HW = A * S
    T = B * HW * HW
    qk = rnd(T, 2 * E, seed=1)
    v = rnd(T, E, seed=2)
    a = torch.zeros(T, E, device=DEV)
    b = torch.zeros(T, E, device=DEV)
    # SAI-mosaic token index = (b*HW + u*S + h)*HW + v*S + w
    if direction == "h":   # sequences over (u, h) for fixed (v, w)  (EPIT.py:150-151)
        args = dict(stride_a=S * HW, stride_s=HW, stride_b=HW * HW, stride_p=S, stride_q=1)
    else:                  # sequences over (v, w) for fixed (u, h)  (EPIT.py:156-157)
        args = dict(stride_a=S, stride_s=1, stride_b=HW * HW, stride_p=S * HW, stride_q=HW)
    ops.epi_attention(qk, v, a, heads, E // heads, A, S, 5, B, A, S, **args)
    ref.epi_attention(qk, v, b, heads, E // heads, A, S, 5, B, A, S, **args)
    assert (a - b).abs().max().item() <= 2e-5


from opref import basictrans_ref as _basictrans_ref


@pytest.mark.parametrize("B,hv", [(2, 8), (1, 16), (2, 32)])
def test_epit_basictrans_fused(ops, B, hv):
    """lfsr_epit_basictrans (one tcgen05 kernel: linear_in .. linear_out, fp16 operands / fp32 accumulate) vs plain torch
    fp32, both EPI directions, sequences of 40 / 80 / 160 tokens (one tile, one tile, two tiles with halo)."""
    A = 5
    H = W = A * hv
    g = torch.Generator().manual_seed(B * 100 + hv)
    r = lambda *sh, sc=1.0: ((torch.rand(*sh, generator=g) - 0.5) * 2 * sc).to(DEV)
    Wt = {"in": r(128, 64, sc=0.125), "qkv": r(384, 128, sc=0.09), "o": r(128, 128, sc=0.09), "ff1": r(256, 128, sc=0.09),
          "ff2": r(128, 256, sc=0.06), "out": r(64, 128, sc=0.09)}
    ln1 = (1.0 + r(128, sc=0.2), r(128, sc=0.1), 1e-5)
    ln2 = (1.0 + r(128, sc=0.2), r(128, sc=0.1), 1e-5)
    packed = ops.pack_basictrans(Wt["in"], Wt["qkv"], Wt["o"], Wt["ff1"], Wt["ff2"], Wt["out"], ln1, ln2, 8, DEV)
    assert packed is not None
    x16 = (torch.rand(B, H, W, 64, generator=g) * 2 - 1).to(DEV).half()      # the kernel's I/O is fp16 (operand copies)
    x = x16.float()
    hw_img = H * W
    passes = [dict(A=A, S=hv, stride_a=hv * W, stride_s=W, stride_b=hw_img, stride_p=hv, stride_q=1, np_=A, nq=hv),
              dict(A=A, S=hv, stride_a=hv, stride_s=1, stride_b=hw_img, stride_p=hv * W, stride_q=W, np_=A, nq=hv)]
    for pi, p in enumerate(passes):
        y16 = torch.full_like(x16, 7.0)
        l0 = ops.lib.lfsr_launch_count()
        assert ops.basictrans(x16, packed[0], packed[1], y16, p["A"], p["S"], 5, B, p["np_"], p["nq"], p["stride_a"], p["stride_s"],
                              p["stride_b"], p["stride_p"], p["stride_q"])
        torch.cuda.synchronize()
        assert ops.lib.lfsr_launch_count() == l0 + 1
        want = _basictrans_ref(x, Wt, ln1, ln2, A, hv, 5, B, p["np_"], p["nq"], p["stride_a"], p["stride_s"], p["stride_b"],
                               p["stride_p"], p["stride_q"])
        err = (y16.float() - want).abs().max().item()
        scale = max(1.0, want.abs().max().item())
        print(f"basictrans B={B} hv={hv} pass {pi}: max err {err:.3e} (ref max {scale:.3f})")
        assert err <= 1.5e-3 * scale, (pi, err, scale)          # 1e-3 + half an fp16 ulp of the output


def test_metrics_vs_oracle_and_golden(ops):
    g = weights.load_pipeline_golden()
    lab, noisy = g["met_label"], g["met_out"]

    class MA:
        angRes_in = 5
        task = "SR"
    p, s = lfsr_b200.lfutils.cal_metrics(MA, torch.from_numpy(lab).to(DEV), torch.from_numpy(noisy).to(DEV))
    assert abs(p - float(g["met_psnr"])) <= 1e-3       # dB; tolerance budget is 0.01 dB
    assert abs(s - float(g["met_ssim"])) <= 1e-5
    # host tensors are staged transparently (reference keeps Hr_SAI_y on the CPU, train.py:322)
    p2, s2 = lfsr_b200.lfutils.cal_metrics(MA, torch.from_numpy(lab), torch.from_numpy(noisy))
    assert abs(p2 - p) < 1e-9 and abs(s2 - s) < 1e-9
    # odd view sizes, per-view values
    rs = np.random.RandomState(1)
    la = rs.random_sample((5 * 37, 5 * 53)).astype(np.float32)
    ou = np.clip(la + rs.normal(0, 0.02, la.shape), 0, 1).astype(np.float32)
    pv, sv = lfsr_b200.lfutils.metric_views(torch.from_numpy(la).to(DEV), torch.from_numpy(ou).to(DEV), 5)
    _, _, po, so = lf_oracle.cal_metrics(la, ou, 5)
    assert np.abs(pv - po).max() <= 1e-3 and np.abs(sv - so).max() <= 1e-5


def _sinusoid_lf(A, hv, seed):
    """HR light field [(a1 hv), (a2 hv)] in [0,1]: a sum of seeded 2-D sinusoids with a per-view disparity shift
    (SURVEY 8d config 5: structured content so that PSNR lands in the 20-35 dB band instead of noise-vs-noise)."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:hv, 0:hv].astype(np.float64)
    out = np.zeros((A, hv, A, hv))
    comps = [(rs.uniform(0.01, 0.7), rs.uniform(0.01, 0.7), rs.uniform(0, 6.28), rs.uniform(0.3, 1.0)) for _ in range(12)]
    for u in range(A):
        for v in range(A):
            img = np.zeros((hv, hv))
            for fy, fx, ph, amp in comps:
                img += amp * np.sin(fy * (yy + 0.7 * u) + fx * (xx + 0.7 * v) + ph)
            out[u, :, v, :] = img
    out = (out - out.min()) / (out.max() - out.min())
    return out.reshape(A * hv, A * hv).astype(np.float32)


@pytest.mark.parametrize("hv", [128, 256, 512])
def test_metrics_realistic_band_large_views(ops, hv):
    """row Q at the sizes and PSNR band of BASELINE config 5: HR views of 128^2..512^2 (x4 of 32^2..128^2 LR views), LR made
    with the reference's own imresize (x0.25 per view), 'SR' = imresize x4 of it -> 20-35 dB. GPU kernel vs the oracle."""
    A = 5
    hr = _sinusoid_lf(A, hv, seed=hv)
    sr = np.empty_like(hr)
    for u in range(A):
        for v in range(A):
            view = hr[u * hv:(u + 1) * hv, v * hv:(v + 1) * hv].astype(np.float64)
            lo = lf_oracle.imresize(view, scalar_scale=0.25)
            sr[u * hv:(u + 1) * hv, v * hv:(v + 1) * hv] = np.clip(lf_oracle.imresize(lo, scalar_scale=4.0), 0, 1)
    pv, sv = lfsr_b200.lfutils.metric_views(torch.from_numpy(hr).to(DEV), torch.from_numpy(sr).to(DEV), A, ops)
    pm, sm, po, so = lf_oracle.cal_metrics(hr, sr, A)
    print(f"metrics hv={hv}: oracle PSNR {pm:.3f} dB SSIM {sm:.5f}; max |dPSNR| {np.abs(pv - po).max():.2e} "
          f"max |dSSIM| {np.abs(sv - so).max():.2e}")
    assert 20.0 <= pm <= 35.0, pm
    assert np.abs(pv - po).max() <= 1e-3 and np.abs(sv - so).max() <= 1e-5


def test_metric_sums_batched_equals_per_mosaic(ops):
    A, hv, n = 5, 48, 3
    rs = np.random.RandomState(3)
    la = torch.from_numpy(rs.random_sample((n, 1, A * hv, A * hv)).astype(np.float32)).to(DEV)
    ou = (la + 0.03 * torch.randn_like(la)).clamp_(0, 1)
    acc = torch.zeros(n * 2 * A * A, dtype=torch.float64, device=DEV)
    ops.metric_sums_batched(la, ou, n, A, hv, hv, acc)
    for i in range(n):
        one = torch.zeros(2 * A * A, dtype=torch.float64, device=DEV)
        ops.metric_sums(la[i, 0], ou[i, 0], A, hv, hv, one)
        got = acc.view(n, -1)[i]
        assert torch.allclose(got, one, rtol=1e-12, atol=0)


def test_metric_shape_mismatch_raises(ops):
    la = torch.rand(5 * 24, 5 * 24, device=DEV)
    with pytest.raises(ValueError):
        lfsr_b200.lfutils.metric_views(la, la[:-5], 5, ops)


# ---- tcgen05 / TMEM / TMA TF32 implicit GEMM -----------------------------------------------------
TC_CASES = [
    dict(cin=54, cout=216, k=(3, 3), pad=(1, 1), act=2, shuffle=(2, 2, 0), hw=(40, 40)),
    dict(cin=54, cout=216, k=(3, 3), pad=(1, 1), act=2, shuffle=(2, 2, 0), hw=(160, 160)),
    dict(cin=54, cout=54, k=(3, 3), dil=(5, 5), pad=(5, 5), res=True, bias=True, hw=(160, 160)),
    dict(cin=64, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=2, hw=(40, 40)),
    dict(cin=64, cout=64, k=(3, 3), pad=(1, 1), act=2, block=(8, 8), res=True, hw=(40, 40)),
    dict(cin=64, cout=64, k=(3, 3), pad=(1, 1), act=2, block=(32, 32), hw=(160, 160)),
    dict(cin=128, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=1, res=True, hw=(160, 160)),
    dict(cin=320, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=1, res=True, hw=(40, 40)),
    dict(cin=144, cout=64, k=(1, 1), act=2, hw=(160, 160)),
    dict(cin=64, cout=1024, k=(1, 1), act=2, shuffle=(4, 4, 0), hw=(40, 40)),
    dict(cin=64, cout=1600, k=(1, 1), shuffle=(5, 5, 0), hw=(32, 32)),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(1, 5, 1), hw=(40, 32)),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(5, 1, 1), hw=(32, 40)),
    dict(cin=128, cout=256, k=(1, 1), hw=(1, 5000)),
    dict(cin=256, cout=128, k=(1, 1), res=True, hw=(1, 5000)),
    dict(cin=64, cout=128, k=(1, 1), hw=(1, 25600)),
    dict(cin=54, cout=1, k=(3, 3), pad=(1, 1), bias=True, res=True, hw=(160, 160)),
    dict(cin=64, cout=32, k=(1, 25), stride=(1, 5), pad=(0, 10), act=2, hw=(160, 160)),
    dict(cin=64, cout=32, k=(25, 1), stride=(5, 1), pad=(10, 0), act=2, hw=(160, 160)),
    dict(cin=64, cout=32, k=(1, 25), stride=(1, 5), pad=(0, 10), act=2, hw=(40, 40)),
    dict(cin=64, cout=32, k=(25, 1), stride=(5, 1), pad=(10, 0), act=2, hw=(40, 40)),
    dict(cin=64, cout=16, k=(5, 5), stride=(5, 5), act=2, hw=(160, 160)),
    dict(cin=64, cout=64, k=(5, 5), stride=(5, 5), act=1, hw=(40, 40)),
    dict(cin=16, cout=400, k=(1, 1), act=2, shuffle=(5, 5, 0), hw=(32, 32)),
    dict(cin=64, cout=1, k=(3, 3), pad=(1, 1), res=True, hw=(40, 40)),
    dict(cin=64, cout=1024, k=(1, 1), act=2, shuffle=(4, 4, 0), hw=(160, 160)),
    dict(cin=128, cout=384, k=(1, 1), hw=(1, 25600)),
    dict(cin=64, cout=128, k=(1, 1), act=4, bias=True, hw=(160, 160)),               # V4_5 gate conv + GELU
    dict(cin=256, cout=64, k=(1, 1), mul=True, mul_act=5, hw=(160, 160)),            # V4_5 fuse * silu(gate)
    dict(cin=64, cout=64, k=(1, 1), mul=True, alpha=0.1, res=True, hw=(40, 40)),
    dict(cin=128, cout=64, k=(1, 1), act=5, hw=(40, 40)),
]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_conv_tc(ref, case):
    _run_tc_case(ref, case)


@pytest.mark.parametrize("switch", ["LFSR_TC_HALO", "LFSR_TC_PAIR"])
def test_conv_tc_halo_block_kernel(ref, switch):
    """the opt-in variants (halo-block kernel, CTA-pair weight multicast) in a subprocess so the env switch is seen
    at first use"""
    import subprocess, sys, os
    env = dict(os.environ, **{switch: "1"})
    code = ("import sys; sys.path[:0]=['.','tests']; import torch, opref, test_kernels_gpu as t; "
            "torch.backends.cudnn.allow_tf32=False; torch.backends.cuda.matmul.allow_tf32=False; r=opref.RefOps();\n"
            "for c in t.TC_CASES:\n    if c['k']==(3,3) and c['cin']<=64: t._run_tc_case(r, c)\nprint('halo ok')")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert out.returncode == 0 and "halo ok" in out.stdout, out.stderr[-2000:]


def _run_tc_case(ref, case):
    tc_ops = K.CudaOps(use_tc=True)
    n = 2
    h, w = case["hw"]
    cin, cout = case["cin"], case["cout"]
    kh, kw = case["k"]
    dil, pad, stride = case.get("dil", (1, 1)), case.get("pad", (0, 0)), case.get("stride", (1, 1))
    g = torch.Generator().manual_seed(cin * 131 + cout)
    wt = (torch.rand(cout, cin, kh, kw, generator=g) - 0.5) * (2.0 / (cin * kh * kw) ** 0.5)
    bias = (torch.rand(cout, generator=g) - 0.5) if case.get("bias") else None
    ry, rx, sm = case.get("shuffle", (1, 1, 0))
    pc = K.pack_conv(wt, bias, stride=stride, dil=dil, pad=pad, device=DEV, tc=True, tc_shuffle=(ry, rx, sm))
    assert pc.w_tc is not None
    x = nhwc(n, h, w, cin, seed=3)
    co = cout // (ry * rx)
    kw_args = dict(act=case.get("act", 0), slope=0.1, alpha=case.get("alpha", 1.0), shuffle=(ry, rx, sm),
                   block=case.get("block", (0, 0)))
    oh, ow = h // stride[0], w // stride[1]
    if case.get("res"):
        kw_args["res"] = nhwc(n, oh * ry, ow * rx, co, seed=5)
    if case.get("mul"):      # a channel window of a wider buffer, like the gate half of FastConvSSM's [gate | y]
        kw_args["mul"] = nhwc(n, oh, ow, 2 * cout, seed=4)[..., :cout]
        kw_args["mul_act"] = case.get("mul_act", 0)
    a = nhwc(n, oh * ry, ow * rx, co, seed=7)
    b = a.clone()
    lib = tc_ops.lib
    l0 = lib.lfsr_launch_count()
    tc_ops.conv(x, pc, a, **kw_args)
    torch.cuda.synchronize()
    ref.conv(x, pc, b, **kw_args)
    err = (a - b).abs().max().item()
    scale = max(1.0, b.abs().max().item())
    print(f"tc conv {case}: max err {err:.3e} (ref max {scale:.3f})")
    assert lib.lfsr_launch_count() == l0 + 1
    assert err <= 1e-3 * scale, f"max err {err}"        # the end-to-end budget (north_star: 1e-3 on [0,1] outputs)


F16_CASES = [
    dict(cin=64, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=2, hw=(40, 40), both=True),
    dict(cin=64, cout=64, k=(3, 3), pad=(1, 1), act=2, block=(8, 8), res=True, hw=(40, 40), both=True),
    dict(cin=64, cout=64, k=(1, 1), act=2, hw=(40, 40)),
    dict(cin=144, cout=64, k=(1, 1), act=2, hw=(40, 40)),
    dict(cin=64, cout=16, k=(5, 5), stride=(5, 5), act=2, hw=(40, 40)),
    dict(cin=64, cout=32, k=(1, 25), stride=(1, 5), pad=(0, 10), act=2, hw=(40, 40)),
    dict(cin=64, cout=32, k=(25, 1), stride=(5, 1), pad=(10, 0), act=2, hw=(40, 40)),
    dict(cin=16, cout=400, k=(1, 1), act=2, shuffle=(5, 5, 0), hw=(8, 8)),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(1, 5, 1), hw=(40, 32)),
    dict(cin=32, cout=160, k=(1, 1), act=2, shuffle=(5, 1, 1), hw=(32, 40)),
    dict(cin=128, cout=64, k=(3, 3), dil=(5, 5), pad=(5, 5), act=1, res=True, hw=(40, 40), both=True),
    dict(cin=56, cout=224, k=(3, 3), pad=(1, 1), act=2, shuffle=(2, 2, 0), hw=(40, 40)),
]


LEAN_CASES = [
    # (cin, cout, k, dil, stride, hw, n, mode, res, bias, act)       mode: 0 fp32 out, 1 fp32 + fp16, 2 fp16 only
    (64, 64, 3, 5, 1, (160, 160), 2, 1, True, True, 2),
    (64, 64, 3, 1, 1, (150, 150), 3, 2, False, False, 2),           # clipped tiles on both edges
    (64, 64, 3, 5, 1, (160, 160), 2, 0, False, True, 1),
    (64, 64, 1, 1, 1, (160, 160), 2, 0, True, False, 0),
    (144, 64, 1, 1, 1, (160, 160), 2, 2, False, True, 2),            # three channel groups, the last one 16 wide
    (128, 64, 3, 5, 1, (160, 160), 2, 1, True, False, 1),
    (64, 16, 1, 1, 1, (160, 160), 2, 2, False, False, 2),            # one 16-column half block, warps 4..7 idle
    (64, 48, 3, 1, 1, (160, 160), 2, 1, True, True, 2),              # second block half full
    (64, 32, 1, 1, 1, (200, 160), 3, 0, False, True, 2),
    (64, 16, 5, 1, 5, (400, 400), 8, 2, False, False, 2),            # DistgSSR AngConv: 5x5 stride 5
    (56, 60, 3, 5, 1, (160, 160), 2, 0, False, True, 0),             # Track-2 fus2: 60 output channels, clipped last block
    (60, 56, 1, 1, 1, (160, 160), 2, 2, False, False, 2, True),      # fp32 input (TF32 MMAs) -> fp16 only (Track-2 fus0 shape)
    (64, 64, 3, 1, 1, (160, 160), 2, 0, True, True, 1, True),        # fp32 input, fp32 output + residual
    (96, 64, 1, 1, 1, (150, 150), 3, 1, False, True, 2, True),       # fp32 input, three 32-channel groups
]


@pytest.mark.parametrize("case", LEAN_CASES, ids=lambda c: f"{c[0]}-{c[1]}-k{c[2]}d{c[3]}s{c[4]}-m{c[7]}")
def test_conv_tc_lean_two_ctas_per_sm(ref, case):
    """the narrow-layer kernel (two CTAs per SM, 16-column half blocks, bias from shared memory): same contract as the
    general tcgen05 kernel, and the test asserts that this kernel is the one that ran"""
    cin, cout, k, dil, stride, (h, w), n, mode, has_res, has_bias, act = case[:11]
    f32in = len(case) > 11 and case[11]
    tc_ops = K.CudaOps()
    g = torch.Generator().manual_seed(cin * 31 + cout * 7 + k)
    wt = (torch.rand(cout, cin, k, k, generator=g) - 0.5) * (2.0 / (cin * k * k) ** 0.5)
    bias = (torch.rand(cout, generator=g) - 0.5) if has_bias else None
    pad = (dil * (k // 2),) * 2 if stride == 1 else (0, 0)
    pc = K.pack_conv(wt, bias, stride=(stride, stride), dil=(dil, dil), pad=pad, device=DEV, tc=True, tc16=True)
    if f32in:
        x16 = nhwc(n, h, w, cin, seed=3)
    else:
        x16 = K.alloc_nhwc16(n, h, w, cin, DEV)
        x16.copy_(nhwc(n, h, w, cin, seed=3))
    oh, ow = h // stride, w // stride
    kw_args = dict(act=act, slope=0.1)
    if has_res:
        kw_args["res"] = nhwc(n, oh, ow, cout, seed=5)
    want = nhwc(n, oh, ow, cout, seed=7)
    ref.conv(x16.float(), pc, want, **kw_args)
    scale = max(1.0, want.abs().max().item())
    o16 = K.alloc_nhwc16(n, oh, ow, cout, DEV)
    o16.fill_(7.0)
    o32 = torch.full_like(want, 7.0)
    c0 = tc_ops.lib.lfsr_conv_tc_lean_count()
    if mode == 0:
        tc_ops.conv(x16, pc, o32, **kw_args)
    elif mode == 1:
        tc_ops.conv(x16, pc, o32, out16=o16, **kw_args)
    else:
        tc_ops.conv(x16, pc, None, out16=o16, **kw_args)
    torch.cuda.synchronize()
    assert tc_ops.lib.lfsr_conv_tc_lean_count() == c0 + 1, "the lean kernel did not take this layer"
    if mode != 2:
        e32 = (o32 - want).abs().max().item()
        assert e32 <= 1e-3 * scale, e32
    if mode == 1:
        assert torch.equal(o16, o32.half())
    if mode == 2:
        e16 = (o16.float() - want).abs().max().item()
        assert e16 <= 1e-3 * scale + scale * 2 ** -10, e16
    # in-place residual (the trunk update of the networks): out aliases res
    if has_res and mode != 2:
        r2 = kw_args["res"].clone()
        kw2 = dict(kw_args); kw2["res"] = r2
        tc_ops.conv(x16, pc, r2, **kw2) if mode == 0 else tc_ops.conv(x16, pc, r2, out16=o16, **kw2)
        torch.cuda.synchronize()
        assert torch.equal(r2, o32)


@pytest.mark.parametrize("case", F16_CASES, ids=lambda c: f"{c['cin']}-{c['cout']}-{c['k'][0]}x{c['k'][1]}")
def test_conv_tc_fp16_operands(ref, case):
    """fp16 activations in (kind::f16 MMAs), fp16-only / fp32 + fp16 outputs, against the plain-torch conv of the SAME fp16
    input values in fp32: only the fp16 rounding of the weights, the accumulation order and the output rounding differ."""
    tc_ops = K.CudaOps()
    n = 2
    h, w = case["hw"]
    cin, cout = case["cin"], case["cout"]
    kh, kw = case["k"]
    dil, pad, stride = case.get("dil", (1, 1)), case.get("pad", (0, 0)), case.get("stride", (1, 1))
    g = torch.Generator().manual_seed(cin * 17 + cout)
    wt = (torch.rand(cout, cin, kh, kw, generator=g) - 0.5) * (2.0 / (cin * kh * kw) ** 0.5)
    ry, rx, sm = case.get("shuffle", (1, 1, 0))
    pc = K.pack_conv(wt, None, stride=stride, dil=dil, pad=pad, device=DEV, tc=True, tc16=True, tc_shuffle=(ry, rx, sm))
    assert pc.w_tc16 is not None
    x16 = K.alloc_nhwc16(n, h, w, cin, DEV)
    x16.copy_(nhwc(n, h, w, cin, seed=3))
    co = cout // (ry * rx)
    oh, ow = h // stride[0], w // stride[1]
    kw_args = dict(act=case.get("act", 0), slope=0.1, shuffle=(ry, rx, sm), block=case.get("block", (0, 0)))
    if case.get("res"):
        kw_args["res"] = nhwc(n, oh * ry, ow * rx, co, seed=5)
    want = nhwc(n, oh * ry, ow * rx, co, seed=7)
    ref.conv(x16.float(), pc, want, **kw_args)
    scale = max(1.0, want.abs().max().item())
    o16 = K.alloc_nhwc16(n, oh * ry, ow * rx, co, DEV)
    if case.get("both"):
        o32 = torch.zeros_like(want)
        tc_ops.conv(x16, pc, o32, out16=o16, **kw_args)
        e32 = (o32 - want).abs().max().item()
        assert e32 <= 1e-3 * scale, e32
        assert torch.equal(o16, o32.half())               # the copy is the rounded fp32 result
    else:
        tc_ops.conv(x16, pc, None, out16=o16, **kw_args)
    torch.cuda.synchronize()
    e16 = (o16.float() - want).abs().max().item()
    print(f"fp16 conv {case}: max err of the fp16 output {e16:.3e} (ref max {scale:.3f})")
    assert e16 <= 1.5e-3 * scale, e16                    # + half an fp16 ulp of the output itself


def test_mel_epi_branch(ops, ref):
    n, h, w, c, klen, A = 2, 40, 40, 18, 11, 5
    full = nhwc(n, h, w, 60, seed=1)
    x = full[..., 40:58]
    wts = rnd((2 * klen + 9) * c + 6 * c * c, seed=2) * 0.3
    a_full, b_full = nhwc(n, h, w, 60, seed=3), nhwc(n, h, w, 60, seed=3)
    ops.mel_epi_branch(x, wts, a_full[..., 40:58], klen, A, 0.1)
    ref.mel_epi_branch(x, wts, b_full[..., 40:58], klen, A, 0.1)
    assert (a_full - b_full).abs().max().item() <= 2e-5
    assert torch.equal(a_full[..., 58:], b_full[..., 58:]) and torch.equal(a_full[..., :40], b_full[..., :40])


@pytest.mark.parametrize("n,h,w", [(2, 40, 40), (3, 37, 70), (64, 160, 160)])
def test_mel_epi_branch_tc(ops, ref, n, h, w):
    """the block with its 1x1 contractions on tcgen05 (fp16 operands, fp32 accumulate) vs the fp32 formulation"""
    c, klen, A = 18, 11, 5
    full = nhwc(n, h, w, 60, seed=1)
    x = full[..., 40:58]
    wts = rnd((2 * klen + 9) * c + 6 * c * c, seed=2) * 0.3
    a_full, b_full = nhwc(n, h, w, 60, seed=3), nhwc(n, h, w, 60, seed=3)
    K.CudaOps(use_tc=True).mel_epi_branch(x, wts, a_full[..., 40:58], klen, A, 0.1, tc=True)
    ops.mel_epi_branch(x, wts, b_full[..., 40:58], klen, A, 0.1) if n > 8 else ref.mel_epi_branch(x, wts, b_full[..., 40:58], klen, A, 0.1)
    scale = max(1.0, b_full[..., 40:58].abs().max().item())
    err = (a_full - b_full).abs().max().item()
    print(f"mel_epi_branch_tc {n}x{h}x{w}: max err {err:.3e} (ref max {scale:.3f})")
    assert 0.0 < err <= 2e-3 * scale, err               # 0 would mean the fp32 kernel ran
    assert torch.equal(a_full[..., 58:], b_full[..., 58:]) and torch.equal(a_full[..., :40], b_full[..., :40])


@pytest.mark.parametrize("n,h,w", [(2, 40, 40), (3, 37, 70), (64, 160, 160)])
def test_mel_epi_branch_mma(ops, ref, n, h, w):
    """the block with the depthwise taps as shifted-row tcgen05 MMAs (pre-swizzled operand image) vs the fp32 formulation"""
    c, klen, A = 18, 11, 5
    full = nhwc(n, h, w, 60, seed=1)
    x = full[..., 40:58]
    wts = rnd((2 * klen + 9) * c + 6 * c * c, seed=2) * 0.3
    a_full, b_full = nhwc(n, h, w, 60, seed=3), nhwc(n, h, w, 60, seed=3)
    tc_ops = K.CudaOps(use_tc=True)
    img = tc_ops.mel_epi_pack(wts, klen, DEV)
    assert img is not None and img.numel() == tc_ops.lib.lfsr_mel_epi_pack_bytes(klen)
    full16 = K.alloc_nhwc16(n, h, w, 64, DEV)
    full16[..., :60].copy_(full)
    tc_ops.mel_epi_branch_mma(x, full16[..., 40:58], img, a_full[..., 40:58], klen, A, 0.1)
    ops.mel_epi_branch(x, wts, b_full[..., 40:58], klen, A, 0.1) if n > 8 else ref.mel_epi_branch(x, wts, b_full[..., 40:58], klen, A, 0.1)
    scale = max(1.0, b_full[..., 40:58].abs().max().item())
    err = (a_full - b_full).abs().max().item()
    print(f"mel_epi_branch_mma {n}x{h}x{w}: max err {err:.3e} (ref max {scale:.3f})")
    assert 0.0 < err <= 2e-3 * scale, err
    assert torch.equal(a_full[..., 58:], b_full[..., 58:]) and torch.equal(a_full[..., :40], b_full[..., :40])


@pytest.mark.parametrize("cin,cout,k,dil", [(54, 1, 3, 1), (64, 1, 3, 1), (64, 3, 3, 5), (18, 2, 1, 1), (60, 4, 3, 1)])
def test_conv_small_cout(ops, ref, cin, cout, k, dil):
    n, h, w = 2, 50, 70
    g = torch.Generator().manual_seed(cin + cout)
    wt = (torch.rand(cout, cin, k, k, generator=g) - 0.5) * 0.2
    bias = torch.rand(cout, generator=g) - 0.5
    pad = dil * (k - 1) // 2
    pc = K.pack_conv(wt, bias, dil=(dil, dil), pad=(pad, pad), device=DEV)
    x = nhwc(n, h, w, cin, seed=3)
    a = rnd(n, h, w, cout, seed=4)
    b = a.clone()
    l0 = ops.lib.lfsr_launch_count()
    ops.conv(x, pc, a, res=a, act=2, slope=0.2, alpha=0.5)
    ref.conv(x, pc, b, res=b.clone(), act=2, slope=0.2, alpha=0.5)
    assert ops.lib.lfsr_launch_count() == l0 + 1
    assert (a - b).abs().max().item() <= 2e-5


def test_conv_tc_18ch_slices(ref):
    """18-channel branch slices of the grouped 60-channel trunk run on the tensor-core path."""
    tc_ops = K.CudaOps(use_tc=True)
    n, h, w = 2, 160, 160
    trunk = nhwc(n, h, w, 60, seed=1)
    cat_a, cat_b = nhwc(n, h, w, 60, seed=2), nhwc(n, h, w, 60, seed=2)
    wt = (torch.rand(18, 18, 3, 3) - 0.5) * 0.3
    pc = K.pack_conv(wt, torch.rand(18) - 0.5, dil=(5, 5), pad=(5, 5), device=DEV, tc=True)
    for sl in (slice(0, 18), slice(20, 38), slice(40, 58)):
        tc_ops.conv(trunk[..., sl], pc, cat_a[..., sl], act=2, slope=0.1)
        ref.conv(trunk[..., sl], pc, cat_b[..., sl], act=2, slope=0.1)
    assert (cat_a - cat_b).abs().max().item() <= 2e-3
    ang = nhwc(n, 32, 32, 18, seed=5)
    wt2 = (torch.rand(450, 18, 1, 1) - 0.5) * 0.3
    pc2 = K.pack_conv(wt2, device=DEV, tc=True, tc_shuffle=(5, 5, 0))
    kw = dict(act=2, slope=0.1, alpha=0.1, res=trunk[..., 20:38], shuffle=(5, 5, 0))
    tc_ops.conv(ang, pc2, cat_a[..., 20:38], **kw)
    ref.conv(ang, pc2, cat_b[..., 20:38], **kw)
    assert (cat_a - cat_b).abs().max().item() <= 2e-3


def test_conv_tc_per_sample_gate(ref):
    """in_scale (per-sample input-channel gate) on the tensor-core path via per-image weight sets"""
    tc_ops = K.CudaOps(use_tc=True)
    n, h, w, cin, cout = 3, 160, 160, 60, 54
    wt = (torch.rand(cout, cin, 1, 1) - 0.5) * 0.3
    pc = K.pack_conv(wt, device=DEV, tc=True)
    x = nhwc(n, h, w, cin, seed=1)
    gate = nhwc(n, 1, 1, cin, seed=2).abs()
    a, b = nhwc(n, h, w, cout, seed=3), nhwc(n, h, w, cout, seed=3)
    l0 = tc_ops.lib.lfsr_launch_count()
    tc_ops.conv(x, pc, a, act=2, slope=0.1, in_scale=gate)
    assert tc_ops.lib.lfsr_launch_count() == l0 + 2          # scale-pack + tcgen05 conv, no fp32 fallback
    ref.conv(x, pc, b, act=2, slope=0.1, in_scale=gate)
    assert (a - b).abs().max().item() <= 2e-3


@pytest.mark.parametrize("cin,cq,hw,bias", [(56, 56, (80, 80), True), (64, 64, (40, 48), False), (56, 56, (37, 45), False)])
def test_conv_tc_tail_projection_and_tap_gather(ref, cin, cq, hw, bias):
    """last upsampler conv + PixelShuffle + LReLU with the 3x3 head conv's channel contraction in its epilogue, then the
    9-tap gather (MyEfficientLFNet.py:104-109): equals conv -> shuffle -> act -> conv3x3(cq->1) + bias + skip"""
    tc_ops = K.CudaOps(use_tc=True)
    n, (h, w), r = 2, hw, 2
    g = torch.Generator().manual_seed(cin + cq)
    wt = (torch.rand(cq * r * r, cin, 3, 3, generator=g) - 0.5) * (2.0 / (cin * 9) ** 0.5)
    b = (torch.rand(cq * r * r, generator=g) - 0.5) if bias else None
    pc = K.pack_conv(wt, b, pad=(1, 1), device=DEV, tc=True, tc_shuffle=(r, r, 0))
    head = (torch.rand(1, cq, 3, 3, generator=g) - 0.5) * 0.2
    tw = torch.zeros(cq, 12)
    tw[:, :9] = head[0].reshape(cq, 9)
    tw = tw.to(DEV)
    hb = torch.tensor([0.125], device=DEV)
    x = nhwc(n, h, w, cin, seed=3)
    assert tc_ops.tail_supported(pc, cq, (r, r, 0))
    ta, tb = nhwc(n, h * r, w * r, 9, seed=4), nhwc(n, h * r, w * r, 9, seed=4)
    kw = dict(act=2, slope=0.1, shuffle=(r, r, 0), tail=(tw, 9, cq))
    l0 = tc_ops.lib.lfsr_launch_count()
    tc_ops.conv(x, pc, ta, **kw)
    assert tc_ops.lib.lfsr_launch_count() == l0 + 1
    ref.conv(x, pc, tb, **kw)
    assert (ta - tb).abs().max().item() <= 2e-3
    ya, yb = rnd(n, h * r, w * r, 1, seed=5), rnd(n, h * r, w * r, 1, seed=5)
    tc_ops.tap_gather(ta, 3, 3, hb, ya, ya)
    ref.tap_gather(ta, 3, 3, hb, yb.clone(), yb)
    assert (ya - yb).abs().max().item() <= 1e-5
    # and the whole thing against the unfused layer pair
    full = nhwc(n, h * r, w * r, cq, seed=6)
    ref.conv(x, pc, full, act=2, slope=0.1, shuffle=(r, r, 0))
    y2 = rnd(n, h * r, w * r, 1, seed=5)
    ref.conv(full, K.pack_conv(head, hb, pad=(1, 1), device=DEV), y2, res=y2.clone())
    assert (ya - y2).abs().max().item() <= 2e-3


@pytest.mark.parametrize("cin,cq,hw,n,bias", [(56, 56, (80, 80), 2, True), (64, 64, (40, 48), 3, False), (56, 56, (37, 45), 2, False),
                                              (56, 56, (160, 160), 3, True)])
def test_conv_tc_tail_projection_fp16_sixteen_epilogue_warps(ref, cin, cq, hw, n, bias):
    """the dominant layer's configuration: fp16 activations, CTA pairs, tail projection with one sub-pixel per epilogue
    warp (16 epilogue warps) - against the plain conv of the same fp16 input values"""
    tc_ops = K.CudaOps(use_tc=True)
    (h, w), r = hw, 2
    g = torch.Generator().manual_seed(cin * 3 + cq)
    wt = (torch.rand(cq * r * r, cin, 3, 3, generator=g) - 0.5) * (2.0 / (cin * 9) ** 0.5)
    b = (torch.rand(cq * r * r, generator=g) - 0.5) if bias else None
    pc = K.pack_conv(wt, b, pad=(1, 1), device=DEV, tc=True, tc16=True, tc_shuffle=(r, r, 0))
    head = (torch.rand(1, cq, 3, 3, generator=g) - 0.5) * 0.2
    tw = torch.zeros(cq, 12)
    tw[:, :9] = head[0].reshape(cq, 9)
    tw = tw.to(DEV)
    x16 = K.alloc_nhwc16(n, h, w, cin, DEV)
    x16.copy_(nhwc(n, h, w, cin, seed=3))
    ta, tb = nhwc(n, h * r, w * r, 9, seed=4), nhwc(n, h * r, w * r, 9, seed=4)
    kw = dict(act=2, slope=0.1, shuffle=(r, r, 0), tail=(tw, 9, cq))
    l0 = tc_ops.lib.lfsr_launch_count()
    tc_ops.conv(x16, pc, ta, **kw)
    assert tc_ops.lib.lfsr_launch_count() == l0 + 1
    ref.conv(x16.float(), pc, tb, **kw)
    assert (ta - tb).abs().max().item() <= 2e-3


@pytest.mark.parametrize("cq,r,k,mode,hw", [(64, 4, 1, 1, (32, 32)), (64, 4, 1, 1, (21, 45)), (32, 4, 3, 0, (40, 40))])
def test_conv_tc_tail_projection_many_cout_chunks(ref, cq, r, k, mode, hw):
    """tail projection when cq*r^2 needs several 256-column cout chunks (EPIT.py:45-48: 1x1 64->1024, PixelShuffle(4),
    LReLU(0.2), 3x3 64->1): every chunk holds whole sub-pixel channel runs and projects them independently"""
    tc_ops = K.CudaOps(use_tc=True)
    n, (h, w), cin = 2, hw, 64
    g = torch.Generator().manual_seed(cq * r + k)
    wt = (torch.rand(cq * r * r, cin, k, k, generator=g) - 0.5) * (2.0 / (cin * k * k) ** 0.5)
    pc = K.pack_conv(wt, None, pad=(k // 2, k // 2), device=DEV, tc=True, tc_shuffle=(r, r, mode))
    head = (torch.rand(1, cq, 3, 3, generator=g) - 0.5) * 0.2
    tw = torch.zeros(cq, 12)
    tw[:, :9] = head[0].reshape(cq, 9)
    tw = tw.to(DEV)
    x = nhwc(n, h, w, cin, seed=3)
    assert tc_ops.tail_supported(pc, cq, (r, r, mode))
    ta, tb = nhwc(n, h * r, w * r, 9, seed=4), nhwc(n, h * r, w * r, 9, seed=4)
    kw = dict(act=2, slope=0.2, shuffle=(r, r, mode), tail=(tw, 9, cq))
    l0 = tc_ops.lib.lfsr_launch_count()
    tc_ops.conv(x, pc, ta, **kw)
    assert tc_ops.lib.lfsr_launch_count() == l0 + 1
    ref.conv(x, pc, tb, **kw)
    assert (ta - tb).abs().max().item() <= 2e-3
    ya = rnd(n, h * r, w * r, 1, seed=5)
    tc_ops.tap_gather(ta, 3, 3, None, ya, ya)
    full = nhwc(n, h * r, w * r, cq, seed=6)
    ref.conv(x, pc, full, act=2, slope=0.2, shuffle=(r, r, mode))
    y2 = rnd(n, h * r, w * r, 1, seed=5)
    ref.conv(full, K.pack_conv(head, None, pad=(1, 1), device=DEV), y2, res=y2.clone())
    assert (ya - y2).abs().max().item() <= 2e-3


@pytest.mark.parametrize("cin,k,dil,hw,bias,act", [(18, 3, 5, (160, 160), True, 2), (18, 3, 5, (37, 45), False, 0), (20, 3, 1, (40, 40), True, 1),
                                                   (16, 1, 1, (40, 40), False, 0)])
def test_conv_thin(ops, ref, cin, k, dil, hw, bias, act):
    """18 -> 20 channel slices of the grouped trunk on the FFMA2 kernel (fp32-exact), pads of the output slot written"""
    n, (h, w) = 2, hw
    g = torch.Generator().manual_seed(cin * 7 + k)
    wt = (torch.rand(20, cin, k, k, generator=g) - 0.5) * (2.0 / (cin * k * k) ** 0.5)
    b = (torch.rand(20, generator=g) - 0.5) if bias else None
    p = dil * (k // 2)
    pc = K.pack_conv(wt, b, dil=(dil, dil), pad=(p, p), device=DEV)
    trunk = nhwc(n, h, w, 60, seed=1)
    x = trunk[..., 20:20 + cin]
    fa, fb = nhwc(n, h, w, 60, seed=2), nhwc(n, h, w, 60, seed=2)
    l0 = ops.lib.lfsr_launch_count()
    ops.conv(x, pc, fa[..., 40:60], act=act, slope=0.1)
    assert ops.lib.lfsr_launch_count() == l0 + 1
    ref.conv(x, pc, fb[..., 40:60], act=act, slope=0.1)
    assert (fa - fb).abs().max().item() <= 2e-5


def test_imresize_vs_reference_golden_and_oracle(golden_dir):
    """SURVEY 8f-3: utils/imresize.py on the GPU against outputs of the unmodified reference (oracle/make_golden.py) and
    against the oracle on other shapes; uint8 results must match exactly, float64 to 1e-12"""
    g = np.load(f"{golden_dir}/imresize.npz")
    kws = {"y_down4": dict(scalar_scale=0.25), "cbcr_up4": dict(scalar_scale=4), "tri_down2": dict(scalar_scale=0.5, method="bilinear"),
           "shape": dict(output_shape=(45, 20)), "u8_down3": dict(scalar_scale=1.0 / 3)}
    for key, kw in kws.items():
        out = lfsr_b200.lfutils.imresize(g[key + "_in"], **kw)
        ref_out = g[key + "_out"]
        assert isinstance(out, np.ndarray) and out.shape == ref_out.shape and out.dtype == ref_out.dtype, key
        if out.dtype == np.uint8:
            assert np.array_equal(out, ref_out), key
        else:
            assert np.abs(out - ref_out).max() <= 1e-12, key
    rs = np.random.RandomState(3)
    for shape, kw in (((160, 160), dict(scalar_scale=0.5)), ((33, 47, 3), dict(scalar_scale=2)), ((64, 64), dict(output_shape=(17, 90)))):
        a = rs.random_sample(shape)
        assert np.abs(lfsr_b200.lfutils.imresize(a, **kw) - lf_oracle.imresize(a, **kw)).max() <= 1e-12
    t = torch.from_numpy(g["y_down4_in"]).to(DEV)
    out_t = lfsr_b200.lfutils.imresize(t, scalar_scale=0.25)
    assert out_t.is_cuda and out_t.dtype == torch.float64 and np.abs(out_t.cpu().numpy() - g["y_down4_out"]).max() <= 1e-12


def test_colour_tail_and_bmp_vs_reference_golden(golden_dir, tmp_path):
    """SURVEY 8f-4: Y + CbCr mosaics -> uint8 RGB views on the device, bit-exact to the reference's fp64 numpy tail
    (oracle/make_golden.py), and BMP files byte-identical to Pillow's (the writer behind imageio.imwrite)"""
    g = np.load(f"{golden_dir}/colour_tail.npz")
    sy, sc = torch.from_numpy(g["sr_y"]), torch.from_numpy(g["sr_cbcr"])
    v = lfsr_b200.lfutils.sai_to_rgb8_views(sy.to(DEV), sc, 5)
    assert v.is_cuda and v.dtype == torch.uint8 and np.array_equal(v.cpu().numpy(), g["views"])
    rs = np.random.RandomState(2)
    y2 = (rs.random_sample((5 * 37, 5 * 29)) * 1.4 - 0.2).astype(np.float32)
    c2 = rs.random_sample((2, 5 * 37, 5 * 29)).astype(np.float32)
    v2 = lfsr_b200.lfutils.sai_to_rgb8_views(torch.from_numpy(y2), torch.from_numpy(c2), 5)
    assert np.array_equal(v2.cpu().numpy(), lf_oracle.sai_to_rgb8_views(y2, c2, 5))
    p = tmp_path / "View_1_3.bmp"
    lfsr_b200.lfutils.write_bmp(str(p), v[1, 3])
    assert np.array_equal(np.frombuffer(p.read_bytes(), dtype=np.uint8), g["bmp_view_1_3"])


@pytest.mark.parametrize("tail", [False, True])
def test_conv_tc_twin_tiles_odd_count(ref, tail):
    """wide streamed-weight layers walk M-tile pairs (one weight stage feeds two tiles / both accumulator stages): an odd
    number of 128-pixel tiles leaves a dummy partner whose stores must be suppressed"""
    tc_ops = K.CudaOps(use_tc=True)
    n, h, w, cin, cq, r = 3, 20, 32, 64, 64, 2          # 3 * 5 * 1 = 15 tiles, weights 590 KB -> streamed
    g = torch.Generator().manual_seed(5)
    wt = (torch.rand(cq * r * r, cin, 3, 3, generator=g) - 0.5) * (2.0 / (cin * 9) ** 0.5)
    pc = K.pack_conv(wt, None, pad=(1, 1), device=DEV, tc=True, tc_shuffle=(r, r, 0))
    x = nhwc(n, h, w, cin, seed=3)
    kw = dict(act=2, slope=0.1, shuffle=(r, r, 0))
    if tail:
        tw = torch.zeros(cq, 12)
        tw[:, :9] = (torch.rand(cq, 9, generator=g) - 0.5) * 0.2
        kw["tail"] = (tw.to(DEV), 9, cq)
        a, b = nhwc(n, h * r, w * r, 9, seed=4), nhwc(n, h * r, w * r, 9, seed=4)
    else:
        a, b = nhwc(n, h * r, w * r, cq, seed=4), nhwc(n, h * r, w * r, cq, seed=4)
    guard = a.clone()
    tc_ops.conv(x, pc, a, **kw)
    ref.conv(x, pc, b, **kw)
    assert (a - b).abs().max().item() <= 2e-3
    assert not torch.equal(a, guard)
