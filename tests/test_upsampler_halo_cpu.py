"""Block plan of the halo-block CTA-pair kernel (lfsr_conv_tc_halo_plan): runs without a GPU. Restates in numpy how the
kernel walks its blocks (cluster pairs, dummy block of an odd tail) and which flattened MMA rows it stores, and checks that
every output pixel is written exactly once and that the shared-memory plan fits."""
import ctypes as C

import numpy as np
import pytest

from lfsr_b200 import _native as N

SMEM_MAX = 227 * 1024
SMS = 148


def _plan(h, w, cout=224):
    geom = (C.c_int * 8)()
    ok = N.load().lfsr_conv_tc_halo_plan(h, w, cout, geom)
    return ok, list(geom)


def _coverage(n, h, w, g):
    two, rout, p, nt, sx, by = g[:6]
    total = n * by * sx
    hits = np.zeros((n, h, w), np.int32)
    pos = np.arange(nt * 128)
    ty, tx = pos // p, pos % p
    keep = (ty < rout) & (tx < two)
    clusters = min((total + 1) // 2, SMS // 2)
    for cl in range(clusters):
        for rank in range(2):
            pr = cl
            while 2 * pr < total:
                b = 2 * pr + rank
                if b < total:           # (b >= total: the dummy block of an odd tail, nothing stored)
                    x0, u = (b % sx) * two, b // sx
                    img, y0 = u // by, (u % by) * rout
                    Y, X = y0 + ty[keep], x0 + tx[keep]
                    inside = (Y < h) & (X < w)
                    np.add.at(hits, (img, Y[inside], X[inside]), 1)
                pr += clusters
    return hits


@pytest.mark.parametrize("h,w", [(160, 160), (320, 320), (161, 173), (330, 100), (40, 300)])
@pytest.mark.parametrize("n", [1, 3, 64])
def test_halo_plan_covers_every_pixel_once(n, h, w):
    ok, g = _plan(h, w)
    assert ok
    two, rout, p, nt, sx, by, a_buf, smem = g
    assert p == two + 2 and sx == -(-w // two) and by == -(-h // rout)
    assert rout * p <= nt * 128 and rout * p > (nt - 1) * 128
    # an input buffer holds the haloed box and every row the last tile's bottom-right tap reads
    assert a_buf % 1024 == 0 and a_buf >= 128 * max((rout + 2) * p, nt * 128 + 2 * p + 2)
    assert smem <= SMEM_MAX and smem >= 2 * a_buf + 9 * 112 * 128
    if n == 64 and max(h, w) > 200:
        n = 4               # (the walk is the same per image; keep the restatement quick)
    assert (_coverage(n, h, w, g) == 1).all()


def test_halo_plan_for_the_upsampler_convs():
    # the x4 model's up.3 (320^2, tail) and up.0 (160^2, fp16 out): at least 90 % of the MMA rows are output pixels
    for h in (320, 160):
        ok, g = _plan(h, h)
        two, rout, p, nt, sx, by = g[:6]
        assert ok and h * h / (sx * by * nt * 128) >= 0.9, g


def test_halo_plan_rejects_what_the_kernel_cannot_run():
    assert _plan(320, 320, cout=600)[0] == 0          # more than one 256-column chunk
    assert _plan(0, 320)[0] == 0
