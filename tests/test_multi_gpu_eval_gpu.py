"""test.py / inference.py under torchrun on 2 GPUs against a single-process run: the same per-dataset lines and
evaluation values, and every View_i_j.bmp byte-identical and written exactly once. With 3 scenes on 2 ranks, scenes 0 and
1 are one full round (one scene per GPU) and scene 2 is the tail, row-sharded over both GPUs.

Row sharding changes the forwards' batch shapes (a rank runs only its patch-grid rows). The one-device test below runs
each rank's rows on their own and checks that the stitched mosaic equals the single run bit for bit, which is what lets
the torchrun comparison ask for byte-identical BMPs of the tail scene too."""
import csv
import os
import re
import signal
import subprocess
import sys

import numpy as np
import pytest
import torch

import lfsr_b200
from oracle import weights

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"

# runs an entry point with lfutils.write_bmp wrapped to log every file it writes (one log per rank). Ranks other than 0
# get their own torch seed, so a random initialisation that did not reach them from rank 0 would show in their scenes.
WRAPPER = r"""
import os, runpy, sys
root, log_dir, script = sys.argv[1:4]
sys.path.insert(0, root)
import torch
rank = int(os.environ.get("RANK", "0"))
if rank:
    torch.manual_seed(1000 + rank)
from lfsr_b200 import lfutils
_write = lfutils.write_bmp
def write_bmp(path, img):
    with open(os.path.join(log_dir, "writes_%d.txt" % rank), "a") as f:
        f.write(os.path.abspath(path) + "\n")
    _write(path, img)
lfutils.write_bmp = write_bmp
sys.argv = [script] + sys.argv[4:]
runpy.run_path(os.path.join(root, script), run_name="__main__")
"""


@pytest.mark.parametrize("name,scale,h0,w0,world,ens", [
    ("MyEfficientLFNet", 4, 32, 32, 2, False), ("MyEfficientLFNet", 4, 64, 48, 8, False), ("DistgSSR", 2, 32, 32, 2, False),
    ("DistgSSR", 2, 32, 32, 2, True)])
def test_row_shards_equal_single_run(name, scale, h0, w0, world, ens):
    A = 5
    net = lfsr_b200.load_net(name, A, scale).eval()
    net.load_state_dict(weights.make_state_dict(name, scale, 1234), strict=True)
    net = net.to(DEV)
    lr = torch.from_numpy(np.random.RandomState(3).random_sample((A * h0, A * w0)).astype(np.float32)).to(DEV)
    with torch.no_grad():
        single = lfsr_b200.scene.super_resolve_scene(net, lr, A, scale, world=1, rank=0, self_ensemble=ens).clone()
        got = torch.full_like(single, -1.0)
        for rank in range(world):
            r = lfsr_b200.scene.SceneRunner(net, A, scale, h0, w0, device=DEV, world=world, rank=rank, depth=1,
                                            with_metrics=False, self_ensemble=ens)
            part = torch.full_like(single, -1.0)
            r.run_resident(lr, part, gather=False)
            a, b = r.spans[rank]
            got.view(A, r.hs, r.W)[:, a:b] = part.view(A, r.hs, r.W)[:, a:b]
    torch.cuda.synchronize()
    assert torch.equal(got, single), float((got - single).abs().max())


def _run(tmp_path, tag, script, flags, nproc):
    log_dir = tmp_path / tag
    log_dir.mkdir()
    wrapper = tmp_path / "wrap_entry.py"
    wrapper.write_text(WRAPPER)
    launch = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(nproc)] if nproc > 1 \
        else [sys.executable]
    cmd = launch + [str(wrapper), ROOT, str(log_dir), script] + flags + ["--path_log", str(log_dir / "log") + "/"]
    # a new session, so that a timeout can take the launcher and every rank down together
    p = subprocess.Popen(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = p.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        p.communicate()
        raise
    assert p.returncode == 0, err[-4000:]
    writes = []
    for fn in sorted(log_dir.glob("writes_*.txt")):
        writes += [os.path.relpath(w, log_dir) for w in fn.read_text().split()]
    bmps = {os.path.relpath(str(b), log_dir): b.read_bytes() for b in (log_dir / "log").rglob("View_*_*.bmp")}
    evals = list((log_dir / "log").rglob("evaluation.*"))
    return out, writes, bmps, evals


def _eval_values(files):
    assert len(files) == 1, files
    f = files[0]
    if f.suffix == ".csv":
        rows = list(csv.reader(open(f)))
    else:
        xlrd = pytest.importorskip("xlrd")
        sh = xlrd.open_workbook(str(f)).sheet_by_index(0)
        rows = [sh.row_values(i) for i in range(sh.nrows)]
    return [(r[0], r[1], float(r[2]), float(r[3])) for r in rows[1:]]


def _numbers(line):
    return [float(x) for x in re.findall(r"\d+\.\d+", line)]


def _compare(single, multi, n_scenes, metric_lines):
    out1, writes1, bmps1, ev1 = single
    out2, writes2, bmps2, ev2 = multi
    assert len(bmps1) == 25 * n_scenes and set(bmps2) == set(bmps1)
    bad = [k for k in bmps1 if bmps1[k] != bmps2[k]]
    assert not bad, bad[:5]
    assert sorted(writes2) == sorted(writes1) == sorted(bmps1)          # every view written once, by one rank
    if metric_lines:
        for key in ("Test on ", "The mean psnr"):
            l1 = [line for line in out1.splitlines() if line.startswith(key)]
            l2 = [line for line in out2.splitlines() if line.startswith(key)]
            assert len(l1) == len(l2) == 1, (l1, l2)                    # printed by rank 0 only
            np.testing.assert_allclose(_numbers(l2[0]), _numbers(l1[0]), rtol=1e-9)
        v1, v2 = _eval_values(ev1), _eval_values(ev2)
        assert [v[:2] for v in v1] == [v[:2] for v in v2] and len(v1) == n_scenes + 2
        np.testing.assert_allclose([v[2:] for v in v2], [v[2:] for v in v1], rtol=1e-9)


def _need_two():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")


def test_test_py_two_gpus_checkpoint(tmp_path):
    _need_two()
    ckpt = tmp_path / "MyEfficientLFNet_x4.pth"
    torch.save({"state_dict": weights.make_state_dict("MyEfficientLFNet", 4, 1234)}, ckpt)
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--path_pre_pth", str(ckpt),
             "--synthetic", "3", "--synthetic_size", "32", "--data_name", "Synthetic"]
    _compare(_run(tmp_path, "single", "test.py", flags, 1), _run(tmp_path, "multi", "test.py", flags, 2), 3, True)


def test_test_py_two_gpus_random_init(tmp_path):
    """--use_pre_ckpt '': rank 0's random initialisation reaches every rank"""
    _need_two()
    flags = ["--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4", "--use_pre_ckpt", "",
             "--synthetic", "3", "--synthetic_size", "32", "--data_name", "Synthetic"]
    _compare(_run(tmp_path, "single", "test.py", flags, 1), _run(tmp_path, "multi", "test.py", flags, 2), 3, True)


def test_inference_py_two_gpus_self_ensemble(tmp_path):
    _need_two()
    ckpt = tmp_path / "DistgSSR_x2.pth"
    torch.save({"state_dict": weights.make_state_dict("DistgSSR", 2, 1234)}, ckpt)
    flags = ["--model_name", "DistgSSR", "--angRes", "5", "--scale_factor", "2", "--path_pre_pth", str(ckpt),
             "--synthetic", "3", "--synthetic_size", "32", "--self_ensemble", "1", "--data_name", "Synthetic"]
    _compare(_run(tmp_path, "single", "inference.py", flags, 1), _run(tmp_path, "multi", "inference.py", flags, 2), 3,
             False)
