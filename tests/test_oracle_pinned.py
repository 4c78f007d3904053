"""The oracle pinned against outputs of the UNMODIFIED reference (tests/golden/*.npz, written in the build container by
oracle/make_golden.py from /root/reference; nothing here reads the reference at run time) and against the
size-independent properties of the patch pipeline (SURVEY 8c). CPU only: this is what makes the GPU parity tests mean
"equals the reference" rather than "equals our restatement"."""
import numpy as np
import pytest
import torch

from oracle import lf_oracle, nets as onets, weights

GOLD = weights.GOLDEN_DIR
SIZES = ((32, 32), (47, 61), (64, 40))


@pytest.mark.parametrize("h0,w0", SIZES)
def test_lfdivide_lfintegrate_equal_reference_outputs(h0, w0):
    """utils/utils.py:152-178 through the reference itself -> pipeline.npz, pipeline_tail.npz; bit-exact (pure indexing)"""
    g = weights.load_pipeline_golden()
    scene = g[f"div_{h0}x{w0}_scene"]
    sub = lf_oracle.lfdivide(scene, 5, 32, 16)
    assert sub.shape == tuple(g[f"div_{h0}x{w0}_shape"])
    assert np.array_equal(sub[0, min(1, sub.shape[1] - 1)], g[f"div_{h0}x{w0}_sub_u0v1"])
    assert np.array_equal(sub[-1, -1], g[f"div_{h0}x{w0}_sub_last"])
    assert float(sub.astype(np.float64).sum()) == float(g[f"div_{h0}x{w0}_sum"])
    up = np.repeat(np.repeat(sub, 2, axis=2), 2, axis=3).reshape(sub.shape[0], sub.shape[1], 5, 32, 2, 5, 32, 2)
    up = np.ascontiguousarray(up).reshape(sub.shape[0], sub.shape[1], 5 * 64, 5 * 64)
    assert np.array_equal(lf_oracle.lfintegrate(up, 5, 64, 32, h0 * 2, w0 * 2), g[f"int_{h0}x{w0}_out"])


def test_cal_metrics_equal_reference_outputs():
    """utils/utils.py:91-134 (skimage restated on scipy): PSNR / SSIM of the reference run on the same pair"""
    g = weights.load_pipeline_golden()
    p, s, pv, sv = lf_oracle.cal_metrics(g["met_label"][0, 0], g["met_out"][0, 0], 5)
    assert abs(p - float(g["met_psnr"])) < 1e-6 and abs(s - float(g["met_ssim"])) < 1e-7
    assert pv.shape == (5, 5) and sv.shape == (5, 5)
    assert abs(pv[pv > 0].mean() - p) < 1e-9           # the ">0" averaging rule of utils.py:131-132


@pytest.mark.parametrize("ang,h0,w0,patch,stride,s", [(5, 32, 32, 32, 16, 4), (5, 33, 47, 32, 16, 2), (3, 20, 75, 32, 16, 4),
                                                     (7, 23, 23, 32, 16, 2), (2, 40, 56, 64, 32, 2), (5, 128, 128, 32, 16, 1),
                                                     (2, 12, 30, 16, 8, 3)])
def test_divide_integrate_round_trip_any_size(ang, h0, w0, patch, stride, s):
    """integrate(upsample_nearest(divide(x))) == upsample_nearest(x) for ragged sizes, other angular resolutions and views
    smaller than a patch: every output sample comes from exactly one patch interior"""
    scene = np.random.RandomState(h0 * 131 + w0).random_sample((ang * h0, ang * w0)).astype(np.float32)
    sub = lf_oracle.lfdivide(scene, ang, patch, stride)
    bdr, nu, nv = lf_oracle.divide_geometry(h0, w0, patch, stride)
    assert sub.shape == (nu, nv, ang * patch, ang * patch)
    up = sub.reshape(nu, nv, ang, patch, 1, ang, patch, 1)
    up = np.broadcast_to(up, (nu, nv, ang, patch, s, ang, patch, s)).reshape(nu, nv, ang * patch * s, ang * patch * s)
    lf = lf_oracle.lfintegrate(np.ascontiguousarray(up), ang, patch * s, stride * s, h0 * s, w0 * s)
    views = scene.reshape(ang, h0, ang, w0).transpose(0, 2, 1, 3)
    assert np.array_equal(lf, np.repeat(np.repeat(views, s, axis=2), s, axis=3))
    assert np.array_equal(lf_oracle.to_sai(views), scene)
    # mirror padding: the first patch's top-left border is the reflected interior (utils.py:137-149)
    p0 = sub[0, 0].reshape(ang, patch, ang, patch)
    assert np.array_equal(p0[:, :bdr, :, bdr:bdr + 4], p0[:, 2 * bdr - 1:bdr - 1:-1, :, bdr:bdr + 4])


@pytest.mark.parametrize("h0,w0,patch,stride", [(40, 40, 16, 16), (17, 16, 32, 16), (64, 64, 32, 8), (64, 64, 48, 16), (4, 40, 32, 24),
                                                (32, 7, 32, 16)])
def test_divide_rejects_what_the_reference_cannot_tile(h0, w0, patch, stride):
    """the reference's unfold / rearrange pair (utils.py:160-164) raises for non-overlapping patches, patch != 2 * stride in
    general and views much smaller than a patch; oracle/make_golden.py sweeps 2580 geometries against the reference:
    same accept / reject decision everywhere, identical values where it accepts"""
    assert not lf_oracle.divide_supported(h0, w0, patch, stride)
    with pytest.raises(ValueError):
        lf_oracle.lfdivide(np.zeros((5 * h0, 5 * w0), np.float32), 5, patch, stride)
    import lfsr_b200
    with pytest.raises(ValueError):
        lfsr_b200.lfutils.check_divide_geometry(h0, w0, patch, stride)
    for ok in ((32, 32, 32, 16), (20, 75, 32, 16), (12, 30, 16, 8), (40, 56, 64, 32)):
        assert lf_oracle.divide_supported(*ok)
        lfsr_b200.lfutils.check_divide_geometry(*ok)


def test_metrics_properties():
    rs = np.random.RandomState(3)
    a = rs.random_sample((5 * 24, 5 * 20)).astype(np.float32)
    p, s, pv, sv = lf_oracle.cal_metrics(a, a, 5)
    assert np.isinf(pv).all() or (pv > 100).all()      # identical views
    assert np.allclose(sv, 1.0)
    b = np.clip(a + 0.1, 0, 1)
    p2, s2, _, _ = lf_oracle.cal_metrics(a, b, 5)
    mse = float(((a.astype(np.float64) - b.astype(np.float64)) ** 2).reshape(5, 24, 5, 20).mean(axis=(1, 3)).mean())
    assert 0 < s2 < 1 and abs(p2 - 10 * np.log10(1.0 / mse)) < 0.2   # mean of per-view PSNRs ~ PSNR of the mean MSE


@pytest.mark.parametrize("name,scale", [("MyEfficientLFNet", 4), ("MyEfficientLFNet", 2), ("EPIT", 4), ("DistgSSR", 4),
                                        ("DistgSSR", 2), ("LF_InterNet", 4), ("MyEfficientLFNetV4_5", 4)])
def test_network_oracles_equal_reference_outputs(name, scale):
    """the functional restatements in oracle/nets.py vs the reference nn.Modules (same seeded state_dict and input):
    8x8-view patches in full, one 32x32-view patch through a subsampled grid and its sum"""
    g = np.load(f"{GOLD}/{name}_x{scale}.npz")
    sd = weights.make_state_dict(name, scale, 1234)
    assert sum(v.numel() for k, v in sd.items() if "running_" not in k and "num_batches" not in k) >= int(g["nparams"])
    x8 = weights.synthetic_patches(2, 5, 8, seed=7)
    y8 = onets.forward(name, x8, sd, 5, scale).numpy()
    assert y8.shape == g["p8_out"].shape and np.abs(y8 - g["p8_out"]).max() <= 1e-5
    if name in ("MyEfficientLFNet", "LF_InterNet"):            # the cheap ones also at the real patch size
        torch.set_num_threads(max(1, torch.get_num_threads()))
        x32 = weights.synthetic_patches(3, 5, 32, seed=0)[:1]
        y32 = onets.forward(name, x32, sd, 5, scale).numpy()
        assert np.abs(y32[0, 0, ::8, ::8] - g["p32_sub"][0, 0]).max() <= 1e-5
        assert abs(float(y32.astype(np.float64).sum()) - float(g["p32_sum"])) <= 1e-2


def test_reference_test_loop_golden_is_consistent():
    """test_loop.npz (reference train.test() on a synthetic scene): the stored PSNR / SSIM are reproducible from the stored
    super-resolved mosaic only through the full pipeline (checked on the GPU); here: its geometry and value ranges"""
    g = np.load(f"{GOLD}/test_loop.npz")
    h0, w0 = int(g["h0"]), int(g["w0"])
    assert g["sr_sub"].shape == (5 * h0 * 4 // 4, 5 * w0 * 4 // 4)
    assert 0 < float(g["psnr"]) < 60 and 0 < float(g["ssim"]) <= 1
