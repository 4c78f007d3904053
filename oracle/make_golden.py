"""ORACLE tooling, build-container only: generate tests/golden/* from the UNMODIFIED reference.

    python oracle/make_golden.py            # writes tests/golden/*.npz + *.spec.json
    python oracle/make_golden.py --stats    # also prints activation statistics (gain tuning)

For every model named by BASELINE.json's configs it (1) dumps the reference module's state_dict
spec, (2) loads oracle.weights.make_state_dict() into the reference module (strict), (3) runs the
reference forward on seeded inputs and stores the outputs, and (4) asserts that the functional
restatement in oracle/nets.py reproduces the reference to <= 2e-5 - i.e. this script is also the
proof that the oracle is pinned. It also stores LFdivide / LFintegrate / cal_metrics / test()
outputs of the reference's utils/utils.py and train.py.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)
from oracle import ref_shim  # noqa: E402

MODELS = [("MyEfficientLFNet", 4), ("MyEfficientLFNet", 2), ("EPIT", 4), ("DistgSSR", 4), ("DistgSSR", 2),
          ("LF_InterNet", 4), ("MyEfficientLFNetV4_5", 4)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stats", action="store_true")
    ap.add_argument("--only", default="")
    opts = ap.parse_args()
    ref_shim.install()
    from oracle import weights, nets, lf_oracle  # after install(): repo is at the END of sys.path
    gold = weights.GOLDEN_DIR
    os.makedirs(gold, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)

    for name, scale in MODELS:
        if opts.only and opts.only != name:
            continue
        mod, net = ref_shim.ref_model(name, 5, scale)
        net.eval()
        spec = [(k, list(v.shape), str(v.dtype).replace("torch.", "")) for k, v in net.state_dict().items()]
        with open(weights.spec_path(name, scale), "w") as f:
            json.dump(spec, f)
        sd = weights.make_state_dict(name, scale, 1234, [(n, tuple(s), d) for n, s, d in spec])
        net.load_state_dict(sd, strict=True)
        nparams = sum(p.numel() for p in net.parameters())
        out = {"nparams": np.int64(nparams)}
        for tag, patch, batch in (("p8", 8, 2), ("p32", 32, 1)):
            x = weights.synthetic_patches(batch, 5, patch, seed=7 if patch == 8 else 0)
            with torch.no_grad():
                y_ref = net(x, [5, 5])
            y_orc = nets.forward(name, x, sd, 5, scale)
            err = (y_ref - y_orc).abs().max().item()
            print(f"{name} x{scale} {tag}: out {tuple(y_ref.shape)} range [{y_ref.min():.3f},{y_ref.max():.3f}] "
                  f"oracle-vs-reference max|d| = {err:.3e}")
            assert err <= 2e-5, "oracle restatement diverges from the reference"
            if opts.stats:
                import torch.nn.functional as F
                base = F.interpolate(x, scale_factor=scale, mode="bicubic", align_corners=False)
                print(f"    |y - bicubic| mean {(y_ref - base).abs().mean():.4f} max {(y_ref - base).abs().max():.4f}")
            y = y_ref.numpy()
            if patch == 8:
                out[f"{tag}_out"] = y.astype(np.float32)
            else:
                out[f"{tag}_sub"] = y[..., ::8, ::8].astype(np.float32).copy()
                out[f"{tag}_sum"] = np.float64(y.astype(np.float64).sum())
                out[f"{tag}_sumsq"] = np.float64((y.astype(np.float64) ** 2).sum())
        np.savez_compressed(os.path.join(gold, f"{name}_x{scale}.npz"), **out)

    if opts.only and opts.only != "imresize":
        return
    # ---- patch pipeline goldens from the reference's utils/utils.py ------------------------------
    import utils.utils as U  # the reference's
    from einops import rearrange
    # domain of LFdivide: the oracle must accept exactly the geometries the reference can tile (its unfold / rearrange pair
    # raises for the others) and agree bit for bit where it accepts; 2580 geometries
    n_geo = 0
    for A_ in (2, 5):
        for (P_, S_) in ((32, 16), (16, 16), (64, 32), (32, 8), (48, 16), (32, 24), (16, 8), (64, 16), (128, 64), (8, 4)):
            for h0 in list(range(1, 40)) + [63, 64, 65, 100]:
                for w0 in (max(h0, 33), h0, 2 * h0 + 1):
                    scene = np.random.RandomState(1).random_sample((A_ * h0, A_ * w0)).astype(np.float32)
                    try:
                        sub = U.LFdivide(torch.from_numpy(scene), A_, P_, S_).numpy()
                    except Exception:
                        sub = None
                    assert (sub is not None) == lf_oracle.divide_supported(h0, w0, P_, S_), (A_, P_, S_, h0, w0)
                    if sub is not None:
                        assert np.array_equal(sub, lf_oracle.lfdivide(scene, A_, P_, S_)), (A_, P_, S_, h0, w0)
                    n_geo += 1
    print(f"LFdivide domain: oracle == reference on {n_geo} geometries")
    pipe = {}
    rs = np.random.RandomState(3)
    for (h0, w0) in ((32, 32), (47, 61), (64, 40)):
        scene = rs.random_sample((5 * h0, 5 * w0)).astype(np.float32)
        sub = U.LFdivide(torch.from_numpy(scene), 5, 32, 16).numpy()
        mine = lf_oracle.lfdivide(scene, 5, 32, 16)
        assert sub.shape == mine.shape and np.array_equal(sub, mine), "lfdivide oracle != reference"
        pipe[f"div_{h0}x{w0}_scene"] = scene
        pipe[f"div_{h0}x{w0}_shape"] = np.array(sub.shape)
        pipe[f"div_{h0}x{w0}_sub_u0v1"] = sub[0, min(1, sub.shape[1] - 1)]
        pipe[f"div_{h0}x{w0}_sub_last"] = sub[-1, -1]
        pipe[f"div_{h0}x{w0}_sum"] = np.float64(sub.astype(np.float64).sum())
        # integrate at x2 on a nearest-upsampled version of the patches (SURVEY 8c identity)
        up = np.repeat(np.repeat(sub, 2, axis=2), 2, axis=3)
        up = up.reshape(sub.shape[0], sub.shape[1], 5, 32, 2, 5, 32, 2)
        up = np.ascontiguousarray(up).reshape(sub.shape[0], sub.shape[1], 5 * 64, 5 * 64)
        integ = U.LFintegrate(torch.from_numpy(up), 5, 64, 32, h0 * 2, w0 * 2).numpy()
        mine_i = lf_oracle.lfintegrate(up, 5, 64, 32, h0 * 2, w0 * 2)
        assert np.array_equal(integ, mine_i), "lfintegrate oracle != reference"
        pipe[f"int_{h0}x{w0}_out"] = integ
    # cal_metrics control flow (>0 rule, per-view loop) through the reference function
    class MA:
        angRes_in = 5
        angRes_out = 5
        task = "SR"
    lab = rs.random_sample((1, 1, 5 * 24, 5 * 20)).astype(np.float32)
    noisy = np.clip(lab + rs.normal(0, 0.05, lab.shape).astype(np.float32), 0, 1).astype(np.float32)
    p_ref, s_ref = U.cal_metrics(MA, torch.from_numpy(lab), torch.from_numpy(noisy))
    p_or, s_or, _, _ = lf_oracle.cal_metrics(lab[0, 0], noisy[0, 0], 5)
    assert abs(p_ref - p_or) < 1e-6 and abs(s_ref - s_or) < 1e-7
    pipe["met_label"], pipe["met_out"] = lab, noisy
    pipe["met_psnr"], pipe["met_ssim"] = np.float64(p_ref), np.float64(s_ref)
    weights.save_pipeline_golden(pipe)

    # ---- utils/imresize.py (SURVEY 8f-3): the reference function on seeded arrays ---------------------
    import utils.imresize as RI  # the reference's
    assert os.path.abspath(RI.__file__).startswith(os.path.abspath(ref_shim.REF_ROOT)), RI.__file__
    rr = np.random.RandomState(31)
    res = {}
    cases = {"y_down4": (rr.random_sample((64, 80)), dict(scalar_scale=0.25)),
             "cbcr_up4": (rr.random_sample((24, 20, 2)), dict(scalar_scale=4)),
             "tri_down2": (rr.random_sample((37, 45)), dict(scalar_scale=0.5, method="bilinear")),
             "shape": (rr.random_sample((30, 50, 3)), dict(output_shape=(45, 20))),
             "u8_down3": ((rr.random_sample((48, 39, 3)) * 255).astype(np.uint8), dict(scalar_scale=1.0 / 3))}
    for key, (arr, kw) in cases.items():
        ref_out = RI.imresize(arr, **kw)
        mine_out = lf_oracle.imresize(arr, **kw)
        d = np.abs(ref_out.astype(np.float64) - mine_out.astype(np.float64)).max()
        print(f"imresize {key}: {arr.shape} {arr.dtype} -> {ref_out.shape} {ref_out.dtype}, oracle-vs-reference max|d| = {d:.3e}")
        assert ref_out.shape == mine_out.shape and ref_out.dtype == mine_out.dtype
        assert d <= (0 if arr.dtype == np.uint8 else 1e-13), key
        res[key + "_in"], res[key + "_out"] = arr, ref_out
    np.savez_compressed(os.path.join(gold, "imresize.npz"), **res)

    # ---- colour / BMP tail (SURVEY 8f-4): the reference's ycbcr2rgb + train.py:332-335, and Pillow's BMP bytes ----------
    import utils.utils as RU  # the reference's
    assert os.path.abspath(RU.__file__).startswith(os.path.abspath(ref_shim.REF_ROOT)), RU.__file__
    from einops import rearrange as _re
    rc = np.random.RandomState(41)
    sy = (rc.random_sample((1, 1, 5 * 12, 5 * 14)) * 1.2 - 0.1).astype(np.float32)          # some values outside [0, 1]
    scbcr = (rc.random_sample((1, 2, 5 * 12, 5 * 14))).astype(np.float32)
    ycbcr = torch.cat((torch.from_numpy(sy), torch.from_numpy(scbcr)), dim=1)
    rgb = (RU.ycbcr2rgb(ycbcr.squeeze().permute(1, 2, 0).numpy()).clip(0, 1) * 255).astype("uint8")
    views = _re(rgb, "(a1 h) (a2 w) c -> a1 a2 h w c", a1=5, a2=5)
    mine_v = lf_oracle.sai_to_rgb8_views(sy[0, 0], scbcr[0], 5)
    assert np.array_equal(views, mine_v), "colour tail oracle != reference"
    import io
    from PIL import Image          # imageio.imwrite of the reference writes .bmp through Pillow's BmpImagePlugin
    bio = io.BytesIO()
    Image.fromarray(views[1, 3]).save(bio, format="BMP")
    np.savez_compressed(os.path.join(gold, "colour_tail.npz"), sr_y=sy, sr_cbcr=scbcr, views=views,
                        bmp_view_1_3=np.frombuffer(bio.getvalue(), dtype=np.uint8))
    print("colour tail: oracle == reference on", views.shape, "; BMP golden", len(bio.getvalue()), "bytes")

    # ---- the reference's train.test() end to end on a synthetic scene (row L of SURVEY 8a) --------
    import train as T  # the reference's
    name, scale = "MyEfficientLFNet", 4
    mod, net = ref_shim.ref_model(name, 5, scale)
    net.load_state_dict(weights.make_state_dict(name, scale, 1234), strict=True)
    net.eval()
    h0, w0 = 40, 48
    # inputs are regenerated from these seeds by the tests (numpy RandomState is platform-stable)
    lr = np.random.RandomState(21).random_sample((1, 1, 5 * h0, 5 * w0)).astype(np.float32)
    hr = np.random.RandomState(22).random_sample((1, 1, 5 * h0 * scale, 5 * w0 * scale)).astype(np.float32)
    cbcr = np.zeros((1, 2, 5 * h0 * scale, 5 * w0 * scale), np.float32)
    loader = [(torch.from_numpy(lr), torch.from_numpy(hr), torch.from_numpy(cbcr),
               [torch.tensor([5]), torch.tensor([5])], ["scene0"])]
    from option import args as ref_args
    torch.cuda.empty_cache = lambda: None
    # capture the stitched SR mosaic by wrapping the reference's own cal_metrics
    captured = {}
    orig = T.cal_metrics
    def spy(a, label, out):
        captured["sr"] = out.numpy().copy()
        return orig(a, label, out)
    T.cal_metrics = spy
    psnr, ssim, names = T.test(loader, torch.device("cpu"), net, ref_args, None)
    T.cal_metrics = orig
    sr = captured["sr"][0, 0]
    np.savez_compressed(os.path.join(gold, "test_loop.npz"), lr_seed=np.int64(21), hr_seed=np.int64(22),
                        h0=np.int64(h0), w0=np.int64(w0), psnr=np.float64(psnr[0]), ssim=np.float64(ssim[0]),
                        sr_sub=sr[::4, ::4].copy(), sr_sum=np.float64(sr.astype(np.float64).sum()))
    print("test(): psnr %.6f ssim %.6f" % (psnr[0], ssim[0]))


if __name__ == "__main__":
    main()
