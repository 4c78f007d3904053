"""x8 geometric self-ensemble on the B200: the two gathers (lfsr_divide_rows_d8 / lfsr_integrate_rows_d8) bit-exact against
their torch composition over the plain divide / integrate kernels, the ensemble scene against the CPU oracle composition,
the pipelined driver, and the test.py flag."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import lfsr_b200
from lfsr_b200 import kernels as K
from lfsr_b200 import lfutils as U
from oracle import lf_oracle, weights
from test_self_ensemble_cpu import oracle_ensemble_scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ops():
    return K.CudaOps()


def t_d8(x, t):
    """T_t on the last two dims"""
    if t & 1:
        x = x.flip(-2)
    if t & 2:
        x = x.flip(-1)
    if t & 4:
        x = x.transpose(-1, -2)
    return x


def t_d8_inv(z, t):
    if t & 4:
        z = z.transpose(-1, -2)
    if t & 2:
        z = z.flip(-1)
    if t & 1:
        z = z.flip(-2)
    return z


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A,h0,w0,P,S,rows", [
    (5, 32, 32, 32, 16, None), (5, 37, 45, 32, 16, None), (3, 20, 75, 32, 16, None), (5, 47, 61, 32, 16, (1, 3)),
    (3, 40, 24, 16, 8, (2, 4)), (5, 64, 40, 32, 16, (3, 4))])
def test_divide_rows_d8_bit_exact(ops, A, h0, w0, P, S, rows):
    scene = torch.from_numpy(np.random.RandomState(h0 * 7 + w0).random_sample((A * h0, A * w0)).astype(np.float32)).to(DEV)
    _, nu, nv = U.divide_geometry(h0, w0, P, S)
    u0, u1 = rows or (0, nu)
    L = A * P
    plain = torch.empty(((u1 - u0) * nv, 1, L, L), device=DEV)
    ops.divide_rows(scene, plain, A, h0, w0, P, S, u0, u1)
    got = torch.full(((u1 - u0) * nv * 8, 1, L, L), -1.0, device=DEV)
    ops.divide_rows_d8(scene, got, A, h0, w0, P, S, u0, u1)
    want = torch.stack([t_d8(plain[:, 0], t) for t in range(8)], 1)
    assert torch.equal(got.view(-1, 8, L, L), want)


def test_divide_rows_d8_rejects_what_divide_rejects(ops):
    small = torch.zeros(5 * 10, 5 * 10, device=DEV)
    out = torch.empty(8, 1, 5 * 32, 5 * 32, device=DEV)
    for fn in (ops.divide_rows, ops.divide_rows_d8):
        with pytest.raises(lfsr_b200.LfsrError):
            fn(small, out, 5, 10, 10, 32, 16, 0, 1)
    with pytest.raises(lfsr_b200.LfsrError, match="row shard"):
        ops.divide_rows_d8(torch.zeros(5 * 32, 5 * 32, device=DEV), out, 5, 32, 32, 32, 16, 1, 3)


@pytest.mark.parametrize("A,h0,w0,P,S,s,rows,offset", [
    (5, 32, 32, 32, 16, 2, None, 0),         # float4 path
    (5, 40, 24, 32, 16, 4, (1, 3), 0),       # x4, row shard
    (5, 37, 45, 32, 16, 2, None, 0),         # w = 90: scalar path
    (2, 12, 30, 16, 8, 3, (1, 2), 0),        # x3 (pz 48, bdr 12), w = 90: scalar path, shard
    (5, 32, 32, 32, 16, 4, None, 1),         # unaligned output pointer: scalar path
    (3, 20, 75, 32, 16, 4, (0, 1), 0)])      # a shard whose rows end before the last patch row
def test_integrate_rows_d8_bit_exact(ops, A, h0, w0, P, S, s, rows, offset):
    _, nu, nv = U.divide_geometry(h0, w0, P, S)
    u0, u1 = rows or (0, nu)
    pz, ss, h, w = P * s, S * s, h0 * s, w0 * s
    Lz = A * pz
    g = torch.Generator().manual_seed(h0 * 31 + w0 * s)
    z8 = (torch.rand(((u1 - u0) * nv, 8, Lz, Lz), generator=g) * 2 - 1).to(DEV)
    acc = t_d8_inv(z8[:, 0], 0)
    for t in range(1, 8):
        acc = acc + t_d8_inv(z8[:, t], t)
    y = (acc * 0.125).unsqueeze(1).contiguous()
    want = torch.full((A * h, A * w), -7.0, device=DEV)
    ops.integrate_rows(y, want, A, pz, ss, h, w, nu, nv, u0, u1)
    buf = torch.full((A * h * A * w + offset,), -7.0, device=DEV)
    got = buf[offset:].view(A * h, A * w)
    ops.integrate_rows_d8(z8, got, A, pz, ss, h, w, nu, nv, u0, u1)
    assert torch.equal(got, want)
    if u1 < nu:                                   # rows outside the shard are untouched
        assert bool((got.view(A, h, A * w)[:, min(u1 * ss, h):] == -7.0).all())


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,scale,minibatch", [("MyEfficientLFNet", 4, 8), ("DistgSSR", 2, 16), ("EPIT", 4, 16)])
def test_ensemble_scene_vs_oracle(name, scale, minibatch):
    """non-square 16 x 24 views = 2 patches = 16 network patches; minibatch 8 runs a patch-grid row in two forwards
    (row_sr path), 16 one row per forward"""
    A, P, S, h0, w0 = 5, 32, 16, 16, 24
    net = lfsr_b200.load_net(name, A, scale).eval()
    sd = weights.make_state_dict(name, scale, 1234)
    net.load_state_dict(sd, strict=True)
    net = net.to(DEV)
    rs = np.random.RandomState(11)
    lr = rs.random_sample((A * h0, A * w0)).astype(np.float32)
    hr = rs.random_sample((A * h0 * scale, A * w0 * scale)).astype(np.float32)
    with torch.no_grad():
        psnr, ssim, sr = lfsr_b200.scene.test_scene(net, torch.from_numpy(lr).to(DEV), torch.from_numpy(hr).to(DEV), A, scale,
                                                    P, S, minibatch, self_ensemble=True)
        sr = sr.cpu().numpy()
        plain = lfsr_b200.scene.super_resolve_scene(net, torch.from_numpy(lr).to(DEV), A, scale, P, S, minibatch).cpu().numpy()
    torch.set_num_threads(os.cpu_count() or 1)
    want = oracle_ensemble_scene(name, lr, sd, A, scale, P, S, h0, w0)
    err = float(np.abs(sr - want).max())
    p_or = lf_oracle.cal_metrics(hr, want, A)[0]
    assert err <= TOL and abs(psnr - p_or) <= 0.01, (err, psnr, p_or)
    assert np.abs(sr - plain).max() > 10 * TOL          # the flag takes effect (random weights are not equivariant)


def test_ensemble_submit_result_equals_test_scene():
    net = lfsr_b200.load_net("MyEfficientLFNet", 5, 4).eval()
    net.load_state_dict(weights.make_state_dict("MyEfficientLFNet", 4, 1234), strict=True)
    net = net.to(DEV)
    A, s, h0, w0 = 5, 4, 40, 24
    r = lfsr_b200.scene.SceneRunner(net, A, s, h0, w0, minibatch=16, device=DEV, world=1, rank=0, depth=2, self_ensemble=True)
    scenes = []
    for k in range(3):
        rs = np.random.RandomState(60 + k)
        lr = torch.from_numpy(rs.random_sample((A * h0, A * w0)).astype(np.float32))
        hr = torch.from_numpy(rs.random_sample((A * h0 * s, A * w0 * s)).astype(np.float32))
        scenes.append((lr.pin_memory() if k % 2 == 0 else lr, hr))
    want = []
    with torch.no_grad():
        for lr, hr in scenes:
            p, q, sr = lfsr_b200.scene.test_scene(net, lr.to(DEV), hr.to(DEV), A, s, minibatch=16, self_ensemble=True)
            want.append((p, q, sr.cpu().clone()))
        tickets, got = [], []
        for lr, hr in scenes:
            tickets.append(r.submit(lr, hr))
            if len(tickets) == 2:
                p, q, sr = r.result(tickets.pop(0))
                got.append((p, q, sr.clone()))
        while tickets:
            p, q, sr = r.result(tickets.pop(0))
            got.append((p, q, sr.clone()))
    for (p0, q0, s0), (p1, q1, s1) in zip(want, got):
        assert torch.equal(s0, s1) and abs(p0 - p1) < 1e-9 and abs(q0 - q1) < 1e-9


def test_entry_point_self_ensemble(tmp_path):
    cmd = [sys.executable, "test.py", "--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4",
           "--use_pre_ckpt", "", "--synthetic", "1", "--synthetic_size", "40", "--self_ensemble", "1",
           "--path_log", str(tmp_path) + "/", "--data_name", "Synthetic"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "The mean psnr on testsets" in r.stdout
    out = tmp_path / "SR_5x5_4x" / "Synthetic" / "MyEfficientLFNet" / "results" / "TEST"
    bmps = sorted(out.rglob("View_*_*.bmp"))
    assert len(bmps) == 25, len(bmps)
