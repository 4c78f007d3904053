"""Dataset split of train.test under a process group (what test.py / inference.py do under torchrun), checked at world 2
over gloo with the kernels replaced by their torch statements (tests/opref.RefOps): full rounds of scenes run one per
rank, the tail is row-sharded over all ranks, and every rank returns what a single process returns, in dataset order."""
import os
import pickle
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME, SCALE, A, P, S = "LF_InterNet", 4, 5, 8, 4
# mixed view sizes; with 2 ranks scenes 0-3 are two full rounds and scene 4 (3 patch-grid rows: ragged stripes) the tail
SIZES = [(12, 8), (8, 12), (10, 10), (12, 8), (12, 16)]


def _args():
    return SimpleNamespace(scale_factor=SCALE, patch_size_for_test=P, stride_for_test=S, minibatch=4, self_ensemble=0,
                           angRes_out=A)


class CountingSet:
    """indexable test set of batch-1 scenes (the layout utils_datasets yields) that records every index it reads."""

    def __init__(self, sizes):
        self.sizes, self.reads = sizes, []

    def __len__(self):
        return len(self.sizes)

    def __getitem__(self, i):
        self.reads.append(i)
        h0, w0 = self.sizes[i]
        rs = np.random.RandomState(100 + i)
        lr = torch.from_numpy(rs.random_sample((1, 1, A * h0, A * w0)).astype(np.float32))
        hr = torch.from_numpy(rs.random_sample((1, 1, A * h0 * SCALE, A * w0 * SCALE)).astype(np.float32))
        cbcr = torch.full((1, 2, A * h0 * SCALE, A * w0 * SCALE), 0.5)
        return lr, hr, cbcr, [torch.tensor([A]), torch.tensor([A])], ["scene_%d" % i]


class IterOnly:
    """a loader that can only iterate (like torch's DataLoader)."""

    def __init__(self, ds):
        self.ds = ds

    def __len__(self):
        return len(self.ds)

    def __iter__(self):
        for i in range(len(self.ds)):
            yield self.ds[i]


def _net():
    import lfsr_b200
    from opref import RefOps
    from oracle import weights
    net = lfsr_b200.load_net(NAME, A, SCALE).eval()
    net.load_state_dict(weights.make_state_dict(NAME, SCALE, 1234))
    net.set_backend(RefOps())
    return net


def _worker(rank, world, port, out_dir):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    import train
    net, args = _net(), _args()
    out = {}
    ds = CountingSet(SIZES)
    out["five"] = train.test(ds, "cpu", net, args)
    out["five_reads"] = list(ds.reads)
    out["five_iter"] = train.test(IterOnly(CountingSet(SIZES)), "cpu", net, args)
    ds = CountingSet(SIZES[-1:])
    out["one"] = train.test(ds, "cpu", net, args)
    out["one_reads"] = list(ds.reads)
    try:
        train.test(CountingSet(SIZES[: rank + 1]), "cpu", net, args)
        out["mismatch"] = None
    except RuntimeError as e:
        out["mismatch"] = str(e)
    with open(os.path.join(out_dir, f"rank{rank}.pkl"), "wb") as f:
        pickle.dump(out, f)
    dist.barrier()
    dist.destroy_process_group()


def test_assign_scenes_partitions():
    import lfsr_b200
    for n in range(0, 10):
        for world in range(1, 10):
            parts = [lfsr_b200.scene.assign_scenes(n, world, r) for r in range(world)]
            full = world * (n // world)
            owned = sorted(i for own, _ in parts for i in own)
            assert owned == list(range(full))                                 # every full-round scene exactly once
            for r, (own, tail) in enumerate(parts):
                assert len(own) == n // world and all(i % world == r for i in own)
                assert tail == list(range(full, n)) and len(tail) < world   # the same tail on every rank
                assert own + tail == sorted(own + tail)                     # run order is dataset order
    with pytest.raises(ValueError):
        lfsr_b200.scene.assign_scenes(3, 2, 2)


def test_synthetic_test_set_indexing_matches_iteration():
    from utils.utils_datasets import SyntheticTestSet
    ds = SyntheticTestSet(SimpleNamespace(angRes_in=A, angRes_out=A, scale_factor=2), 3, 8)
    for i, it in enumerate(ds):
        got = ds[i]
        assert got[4] == it[4] and all(torch.equal(a, b) for a, b in zip(got[:3], it[:3]))
    with pytest.raises(IndexError):
        ds[3]


@pytest.mark.timeout(900)
def test_two_rank_dataset_split_equals_single_process(tmp_path):
    import train
    port = 29500 + ((os.getpid() + 500) % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    got = []
    for r in range(2):
        with open(tmp_path / f"rank{r}.pkl", "rb") as f:
            got.append(pickle.load(f))
    threads = torch.get_num_threads()
    torch.set_num_threads(2)          # the ranks' thread count: the CPU convolutions give the same bits
    try:
        net, args = _net(), _args()
        want5 = train.test(CountingSet(SIZES), "cpu", net, args)
        want1 = train.test(CountingSet(SIZES[-1:]), "cpu", net, args)
    finally:
        torch.set_num_threads(threads)
    for key, want, n_full in (("five", want5, 4), ("five_iter", want5, 4), ("one", want1, 0)):
        for r in range(2):
            psnr, ssim, names = got[r][key]
            assert names == want[2], (key, r, names)
            # full-round scenes ran as single-GPU runs: exact; tail scenes were row-sharded
            assert psnr[:n_full] == want[0][:n_full] and ssim[:n_full] == want[1][:n_full], key
            assert np.abs(np.subtract(psnr[n_full:], want[0][n_full:])).max() <= 1e-4, key
            assert np.abs(np.subtract(ssim[n_full:], want[1][n_full:])).max() <= 1e-6, key
        assert got[0][key] == got[1][key]
    # a full-round scene is read only by its owner; the tail by every rank
    for r in range(2):
        assert got[r]["five_reads"] == [r, r + 2, 4]
        assert got[r]["one_reads"] == [0]
        assert "disagree" in got[r]["mismatch"]
