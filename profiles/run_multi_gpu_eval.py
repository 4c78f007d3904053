"""Wall time of a dataset evaluation split across the GPUs of one node (train.test as test.py runs it under torchrun).

  torchrun --standalone --nproc_per_node N profiles/run_multi_gpu_eval.py OUT_DIR  -> OUT_DIR/multi_gpu_eval_n<N>.json
  python profiles/run_multi_gpu_eval.py --table OUT_DIR                            -> markdown table of every N found there,
                                                                                      speedup over N = 1

Workloads: MyEfficientLFNet x4 with seeded weights (oracle.weights, seed 1234) on the seeded synthetic scenes of
utils/utils_datasets.py, which generates each scene when it is read, as an h5 read would. The three sit on either side
of the split rule (scene.assign_scenes):
  (a) 16 scenes of 5x5x64x64: full rounds only at N = 1, 2, 8
  (b) 11 such scenes: at N = 8 one full round and a row-sharded tail of 3
  (c) 3 scenes of 5x5x256x256: at N = 8 tail only (fewer scenes than GPUs)
Each runs with the BMP tail on (25 View_i_j.bmp per scene, into a temporary directory) and off. Wall seconds per dataset:
from before the first scene is read to train.test's return, which comes after the last per-scene result is gathered;
the ranks start together after a barrier. One untimed pass per workload first (runner allocation, CUDA-graph capture),
then the median of 3 timed passes. The GPU names and power limits are read in the same run.
"""
import glob
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = [("a", 16, 64), ("b", 11, 64), ("c", 3, 256)]
REPEATS = 3


def device_info(index):
    import torch
    info = {"index": index, "name": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        pl, mx = [x.strip() for x in q.split(",")]
        info.update(power_limit=pl, clocks_max_sm=mx)
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        info.update(power_limit=None, error=repr(e)[:200])
    return info


def measure(out_dir):
    # the entry points read their options from the command line at import time
    sys.argv = ["test.py", "--model_name", "MyEfficientLFNet", "--angRes", "5", "--scale_factor", "4"]
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import torch.distributed as dist
    import test as entry
    import train
    from option import args
    from oracle import weights
    from utils.utils_datasets import SyntheticTestSet
    import lfsr_b200
    if not torch.cuda.is_available():
        sys.exit("run_multi_gpu_eval.py measures on CUDA devices; none found")
    device, rank = entry.init_distributed(args)
    try:
        world, _ = train.dist_world()
        barrier = dist.barrier if world > 1 else (lambda: None)
        net = lfsr_b200.load_net("MyEfficientLFNet", 5, 4).eval()
        net.load_state_dict(weights.make_state_dict("MyEfficientLFNet", 4, 1234), strict=True)
        net = net.to(device)
        entry.broadcast_weights(net)
        res = {"world": world, "repeats": REPEATS, "workloads": []}
        for tag, n, size in WORKLOADS:
            ds = SyntheticTestSet(args, n, size)
            for bmp in (True, False):
                save_dir = Path(tempfile.mkdtemp(prefix="lfsr_eval_")) if bmp else None
                try:
                    walls, psnr = [], None
                    for k in range(REPEATS + 1):
                        barrier()
                        t0 = time.perf_counter()
                        with torch.no_grad():
                            psnr, _, _ = train.test(ds, device, net, args, save_dir)
                        torch.cuda.synchronize()
                        if k:
                            walls.append(time.perf_counter() - t0)
                finally:
                    if save_dir is not None:
                        shutil.rmtree(save_dir, ignore_errors=True)
                _, tail = lfsr_b200.scene.assign_scenes(n, world, rank)
                wall = float(np.median(walls))
                res["workloads"].append({"workload": tag, "scenes": n, "view": size, "bmp": bmp, "full_rounds": n // world,
                                         "tail": len(tail), "wall_s": wall, "walls_s": walls, "scenes_per_s": n / wall,
                                         "mean_psnr": float(np.mean(psnr))})
        infos = [None] * world
        if world > 1:
            dist.all_gather_object(infos, device_info(device.index))
        else:
            infos = [device_info(device.index)]
        res["devices"] = infos
        if rank == 0:
            os.makedirs(out_dir, exist_ok=True)
            with open(os.path.join(out_dir, "multi_gpu_eval_n%d.json" % world), "w") as f:
                json.dump(res, f, indent=1)
            print(json.dumps(res))
    finally:
        entry.finish_distributed()


def table(out_dir):
    runs = {}
    for fn in glob.glob(os.path.join(out_dir, "multi_gpu_eval_n*.json")):
        with open(fn) as f:
            r = json.load(f)
        runs[r["world"]] = r
    base = {(w["workload"], w["bmp"]): w["wall_s"] for w in runs.get(1, {"workloads": []})["workloads"]}
    print("| workload | BMP | N | full rounds + tail | wall s | scenes/s | speedup over N = 1 |")
    print("|---|---|---|---|---|---|---|")
    for world in sorted(runs):
        for w in runs[world]["workloads"]:
            b = base.get((w["workload"], w["bmp"]))
            sp = "%.2f" % (b / w["wall_s"]) if b else "not measured"
            print("| (%s) %d x 5x5x%d² | %s | %d | %d + %d | %.3f | %.1f | %s |" % (
                w["workload"], w["scenes"], w["view"], "on" if w["bmp"] else "off", world, w["full_rounds"], w["tail"],
                w["wall_s"], w["scenes_per_s"], sp))
    for world in sorted(runs):
        print("N = %d: %s" % (world, "; ".join("%s, power limit %s" % (d["name"], d.get("power_limit"))
                                               for d in runs[world]["devices"])))


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--table":
        table(sys.argv[2])
    elif len(sys.argv) == 2:
        measure(sys.argv[1])
    else:
        sys.exit(__doc__)
