"""x8 geometric self-ensemble (include/lfsr.h: lfsr_divide_rows_d8 / lfsr_integrate_rows_d8) without a GPU: the group
itself, the scene driver's ensemble plan on the torch statement of the kernels against the numpy composition over the
oracle forward, and a world-2 gloo run of a row-sharded ensemble scene."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from opref import RefOps
from oracle import lf_oracle, nets as onets, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the definition, in numpy -----------------------------------------------------------------------------------------
def d8(m, t):
    """T_t(M): flip rows if t & 1, flip columns if t & 2, transpose if t & 4 (in that order)"""
    if t & 1:
        m = m[::-1, :]
    if t & 2:
        m = m[:, ::-1]
    if t & 4:
        m = m.T
    return m


def d8_inv(z, t):
    """T_t^-1: the same steps in reverse order"""
    if t & 4:
        z = z.T
    if t & 2:
        z = z[:, ::-1]
    if t & 1:
        z = z[::-1, :]
    return z


def ensemble(z8):
    """z8 [8, L, L] = F(T_t X) -> ((T_0^-1 z0 + T_1^-1 z1) + ... + T_7^-1 z7) * 0.125 in float32"""
    acc = np.ascontiguousarray(d8_inv(z8[0], 0)).astype(np.float32)
    for t in range(1, 8):
        acc = acc + d8_inv(z8[t], t).astype(np.float32)
    return acc * np.float32(0.125)


class D8RefOps(RefOps):
    """RefOps plus the two self-ensemble gathers stated on top of the plain divide / integrate statements"""

    def divide_rows_d8(self, scene, patches, ang, h0, w0, patch, stride, u0, u1):
        sub = lf_oracle.lfdivide(scene.detach().cpu().numpy().reshape(ang * h0, ang * w0), ang, patch, stride)[u0:u1]
        sub = sub.reshape(-1, ang * patch, ang * patch)
        v = np.stack([np.stack([d8(p, t) for t in range(8)]) for p in sub])
        patches.view(-1)[: v.size].copy_(torch.from_numpy(v.reshape(-1)))

    def integrate_rows_d8(self, patches8, out, ang, pz, stride, h, w, num_u, num_v, u0, u1):
        L = ang * pz
        z = patches8.detach().cpu().numpy().reshape(-1)[: (u1 - u0) * num_v * 8 * L * L].reshape(-1, 8, L, L)
        y = np.stack([ensemble(p) for p in z])
        self.integrate_rows(torch.from_numpy(y), out, ang, pz, stride, h, w, num_u, num_v, u0, u1)


def oracle_ensemble_scene(name, lr, sd, A, scale, patch, stride, h0, w0):
    """LFdivide -> per patch: F on its 8 variants, undo, average -> LFintegrate, all on the CPU oracle"""
    sub = lf_oracle.lfdivide(lr, A, patch, stride)
    nu, nv = sub.shape[:2]
    L = A * patch
    x = np.stack([d8(p, t) for p in sub.reshape(-1, L, L) for t in range(8)])
    y = onets.forward(name, torch.from_numpy(np.ascontiguousarray(x)).unsqueeze(1), sd, A, scale).numpy()
    y = y.reshape(nu * nv, 8, L * scale, L * scale)
    ens = np.stack([ensemble(p) for p in y]).reshape(nu, nv, L * scale, L * scale)
    return lf_oracle.to_sai(lf_oracle.lfintegrate(ens, A, patch * scale, stride * scale, h0 * scale, w0 * scale))


# ---- the group ---------------------------------------------------------------------------------------------------------
def test_group_properties():
    A, h, w = 3, 4, 6
    m = np.random.RandomState(0).random_sample((A * h, A * h)).astype(np.float32)
    imgs = [d8(m, t) for t in range(8)]
    for t in range(8):
        assert np.array_equal(d8_inv(imgs[t], t), m)
    assert len({im.tobytes() for im in imgs}) == 8
    # on a [(u h), (v w)] SAI mosaic a row flip reverses u together with h, a column flip v with w, and the transpose swaps
    # (u, h) with (v, w): the epipolar geometry is kept
    r = np.random.RandomState(1).random_sample((A * h, A * w)).astype(np.float32)
    v = r.reshape(A, h, A, w)
    assert np.array_equal(r[::-1, :].reshape(A, h, A, w), v[::-1, ::-1, :, :])
    assert np.array_equal(r[:, ::-1].reshape(A, h, A, w), v[:, :, ::-1, ::-1])
    assert np.array_equal(r.T.reshape(A, w, A, h), v.transpose(2, 3, 0, 1))
    # averaging the un-transformed network outputs of an equivariant "network" (the identity) returns the input
    z = np.stack([d8(m, t) for t in range(8)])
    assert ensemble(z).dtype == np.float32 and np.allclose(ensemble(z), m, rtol=0, atol=1e-6)


def test_ref_gathers_state_the_definition():
    A, P, S, h0, w0 = 5, 8, 4, 12, 8
    ops = D8RefOps()
    lr = np.random.RandomState(3).random_sample((A * h0, A * w0)).astype(np.float32)
    sub = lf_oracle.lfdivide(lr, A, P, S)
    nu, nv = sub.shape[:2]
    L = A * P
    got = torch.empty(((nu - 1) * nv * 8, 1, L, L))
    ops.divide_rows_d8(torch.from_numpy(lr), got, A, h0, w0, P, S, 1, nu)
    got = got.numpy().reshape(nu - 1, nv, 8, L, L)
    for u in range(1, nu):
        for v in range(nv):
            for t in range(8):
                assert np.array_equal(got[u - 1, v, t], d8(sub[u, v], t))
    # integrate: the unchanged patch in all 8 slots (each already un-transformed) -> the plain LFintegrate, since 8 equal
    # float32 summands scaled by 1/8 give the summand back exactly when no addition rounds (small integers)
    s = 2
    Lz = L * s
    up = np.random.RandomState(4).randint(0, 16, (nu, nv, Lz, Lz)).astype(np.float32)
    z8 = np.stack([np.stack([d8(p, t) for t in range(8)]) for p in up.reshape(-1, Lz, Lz)])
    out = torch.full((A * h0 * s, A * w0 * s), -1.0)
    ops.integrate_rows_d8(torch.from_numpy(z8), out, A, P * s, S * s, h0 * s, w0 * s, nu, nv, 0, nu)
    want = lf_oracle.to_sai(lf_oracle.lfintegrate(up, A, P * s, S * s, h0 * s, w0 * s))
    assert np.array_equal(out.numpy(), want)


# ---- the scene driver --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,scale,h0,w0,minibatch", [
    ("MyEfficientLFNet", 4, 12, 8, 16),      # non-square views, one patch-grid row (2 patches x 8 variants) per forward
    ("DistgSSR", 2, 10, 10, 20),             # square views, MacPI network, a row (24) wider than a forward: row_sr path
])
def test_scene_ensemble_matches_oracle(name, scale, h0, w0, minibatch):
    import lfsr_b200
    A, P, S = 5, 8, 4
    sd = weights.make_state_dict(name, scale, 1234)
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(sd, strict=True)
    ops = D8RefOps()
    net.set_backend(ops)
    lr = np.random.RandomState(h0 * 100 + w0).random_sample((A * h0, A * w0)).astype(np.float32)
    runner = lfsr_b200.scene.SceneRunner(net, A, scale, h0, w0, P, S, minibatch=minibatch, device="cpu", ops=ops, world=1,
                                         rank=0, depth=1, with_metrics=False, self_ensemble=True)
    assert runner.sub.shape[0] == 8 * runner.num_u * runner.num_v
    assert (runner.rows_per_mb == 0) == (8 * runner.num_v > minibatch)
    mosaic = torch.empty((runner.H, runner.W))
    with torch.no_grad():
        runner.run_resident(torch.from_numpy(lr), mosaic)
    want = oracle_ensemble_scene(name, lr, sd, A, scale, P, S, h0, w0)
    assert np.abs(mosaic.numpy() - want).max() <= 2e-5
    # the functional API goes through a cached runner of its own and gives the same mosaic
    with torch.no_grad():
        sr = lfsr_b200.scene.super_resolve_scene(net, torch.from_numpy(lr), A, scale, P, S, minibatch, ops=ops,
                                                 self_ensemble=True)
    assert torch.equal(sr, mosaic)
    plain = lfsr_b200.scene.runner_for(net, A, scale, h0, w0, P, S, minibatch, torch.device("cpu"), ops, world=1, rank=0)
    assert not plain.self_ensemble and plain.sub.shape[0] == runner.num_u * runner.num_v


# ---- world-2 gloo: row-sharded ensemble scene == single process -------------------------------------------------------
def _worker(rank, world, port, out_dir):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    import lfsr_b200
    from test_self_ensemble_cpu import D8RefOps
    name, scale, A = "MyEfficientLFNet", 2, 5
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(weights.make_state_dict(name, scale, 1234))
    ops = D8RefOps()
    net.set_backend(ops)
    lr = torch.from_numpy(np.random.RandomState(5).random_sample((A * 12, A * 8)).astype(np.float32))
    with torch.no_grad():
        sr = lfsr_b200.scene.super_resolve_scene(net, lr, A, scale, 8, 4, minibatch=16, ops=ops, self_ensemble=True)
    np.save(os.path.join(out_dir, f"sr_rank{rank}.npy"), sr.numpy())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(900)
def test_two_rank_ensemble_scene_equals_single_process(tmp_path):
    import lfsr_b200
    port = 29500 + ((os.getpid() + 1000) % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a = np.load(tmp_path / "sr_rank0.npy")
    b = np.load(tmp_path / "sr_rank1.npy")
    assert np.array_equal(a, b)
    name, scale, A = "MyEfficientLFNet", 2, 5
    sd = weights.make_state_dict(name, scale, 1234)
    lr = np.random.RandomState(5).random_sample((A * 12, A * 8)).astype(np.float32)
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(sd)
    ops = D8RefOps()
    net.set_backend(ops)
    with torch.no_grad():
        single = lfsr_b200.scene.super_resolve_scene(net, torch.from_numpy(lr), A, scale, 8, 4, minibatch=16, ops=ops,
                                                     self_ensemble=True, group=None)
    assert np.array_equal(a, single.numpy())
    assert np.abs(a - oracle_ensemble_scene(name, lr, sd, A, scale, 8, 4, 12, 8)).max() <= 2e-5
