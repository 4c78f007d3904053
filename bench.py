#!/usr/bin/env python
"""bench.py - LF patches/s of the patch-wise LF-SR inference path on N B200s (one rank per GPU).

Headline (BASELINE.json configs[1]): a step = one pass of the hot path over one synthetic scene that LFdivide cuts into
`--batch` (default 64) 5x5x32x32 patches:  LFdivide -> MyEfficientLFNet forward (batch 64) -> LFintegrate -> PSNR/SSIM,
through the product's scene driver (lfsr_b200.scene.SceneRunner - what train.test() calls).
  value     LR + HR scene already in HBM when the timed region starts
  e2e       the same call with HOST buffers: LR and HR label in (H2D inside), stitched SR mosaic and metric sums out (D2H
            inside), two scenes in flight
  parity    max|net(x) - oracle(x)| and |dPSNR| on the first patches AT THE WEIGHTS BEING TIMED (oracle = CPU restatement
            of the reference, pinned bit-exact to it)
  roofline  dominant kernel (tensor-pipe bound) + whole-path per-layer HBM fraction (SURVEY 8d reporting rule)
  configs   the other BASELINE configs: EPIT x4, DistgSSR x2/x4 batch sweep, LF-InterNet x4 with on-GPU PSNR/SSIM, V4_5
  gpu_eager_baseline   the reference algorithm in eager PyTorch fp32 (TF32 off) on the same GPU - the bar of SURVEY 2
  strong_scaling       BASELINE configs[2]: ONE 5x5x512x512 EPIT scene, patch-grid rows sharded over the ranks, stripes
                       all-gathered over NCCL
  cpu_baseline         the reference algorithm on the host cores (oracle port)
N > 1: every rank runs its own scenes for `value` (weak scaling, no data-path collective).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model NAME] [--quick] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed headline step of --impl ours returned (rank 0): sr.npy (float32 SR mosaic),
metric_sums.npy (float64 per-view sums of squared error and SSIM) and psnr_ssim.npy (float64). Inputs and weights are
seeded, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ANG, PATCH, STRIDE = 5, 32, 16

# SURVEY.md 8d: algorithmic work per patch (fp32, "per-layer bytes" = sum over contraction ops of in + out + weights)
PER_PATCH = {
    ("MyEfficientLFNet", 4): dict(flops=38.95e9, layer_bytes=665.6e6),
    ("MyEfficientLFNetV4_5", 4): dict(flops=60.84e9, layer_bytes=1715.3e6),
    ("EPIT", 4): dict(flops=162.61e9, layer_bytes=2372.1e6, basictrans_flops=96.5e9, attn_core_flops=21.0e9),
    ("DistgSSR", 2): dict(flops=127.97e9, layer_bytes=1608.9e6),
    ("DistgSSR", 4): dict(flops=130.52e9, layer_bytes=1767.6e6),
    ("LF_InterNet", 4): dict(flops=107.34e9, layer_bytes=839.6e6),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="MyEfficientLFNet")
    ap.add_argument("--scale", type=int, default=4)
    ap.add_argument("--batch", type=int, default=64, help="patches per step per GPU (must be a square number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + parity + roofline only (no configs / eager / sustained legs)")
    ap.add_argument("--no-tc", action="store_true", help="keep every conv on the fp32 CUDA-core kernels")
    ap.add_argument("--sustained-s", type=float, default=5.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def scene_side(batch: int) -> int:
    """view size h0 such that LFdivide yields sqrt(batch)^2 patches: numU = (h0 + 15)//16."""
    n = int(round(batch ** 0.5))
    assert n * n == batch, "--batch must be a square number"
    return n * STRIDE


def synthetic_scene(h0: int, scale: int, seed: int):
    rs = np.random.RandomState(seed)
    lr = rs.random_sample((ANG * h0, ANG * h0)).astype(np.float32)
    hr = rs.random_sample((ANG * h0 * scale, ANG * h0 * scale)).astype(np.float32)
    return lr, hr


def workload_config(model: str, scale: int, batch: int, world: int):
    """the `config` object of BOTH arms (the reference arm times a bounded sample of exactly this workload)."""
    h0 = scene_side(batch)
    return {"workload": f"{model} 5x5 x{scale}: LFdivide -> forward(batch {batch} patches 5x5x32x32) -> LFintegrate -> "
                        f"PSNR/SSIM, one {h0}x{h0}-view synthetic scene per GPU per step (BASELINE configs[1])",
            "patches_per_step_per_gpu": batch, "parallelism": f"scene-parallel x{world}",
            "l2": "activations per step (>6 GB at batch 64) exceed the 126 MB L2; inputs rotate over 4 scenes",
            "weights": "random init (torch.manual_seed(1234), constructor defaults)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
            if len(f) > 6:
                try:
                    pw.append(float(f[6]))
                except ValueError:
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# -------------------------------------------------------------------------------------------------
def cpu_reference_rate(model: str, scale: int, patches: int, steps: int, warmup: int, minibatch: int = 1, sd=None):
    """The reference algorithm on the host cores (oracle port: numpy divide/integrate/metrics + the
    torch-CPU restatement of the reference forward, == reference bit-exactly). Returns patches/s."""
    from oracle import lf_oracle, nets as onets, weights
    torch.set_num_threads(os.cpu_count() or 1)
    if sd is None:
        sd = weights.make_state_dict(model, scale, 1234)
    n = int(round(patches ** 0.5))
    h0 = n * STRIDE
    lr, hr = synthetic_scene(h0, scale, 0)

    def step():
        sub = lf_oracle.lfdivide(lr, ANG, PATCH, STRIDE)
        nu, nv = sub.shape[:2]
        x = torch.from_numpy(sub.reshape(nu * nv, 1, ANG * PATCH, ANG * PATCH))
        with torch.no_grad():      # minibatch 1: option.py:45
            ys = [onets.forward(model, x[i:i + minibatch], sd, ANG, scale) for i in range(0, nu * nv, minibatch)]
        y = torch.cat(ys).numpy().reshape(nu, nv, ANG * PATCH * scale, ANG * PATCH * scale)
        sr = lf_oracle.to_sai(lf_oracle.lfintegrate(y, ANG, PATCH * scale, STRIDE * scale, h0 * scale, h0 * scale))
        return lf_oracle.cal_metrics(hr, sr, ANG)[:2], nu * nv

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        _, k = step()
        done += k
    dt = time.perf_counter() - t0
    return done / dt, dt / steps * 1e3, done // steps


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.dump_outputs:
        print("[bench] --dump-outputs is ignored with --impl reference (it times a smaller sample of the workload)",
              file=sys.stderr)
    patches = 16           # bounded sample: a 4x4-patch scene per step (~1.5 s of host work on the GPU box)
    import lfsr_b200
    torch.manual_seed(1234)                                  # the product arm's weights: seeded constructor-default init
    sd = {k: v.detach().clone() for k, v in lfsr_b200.load_net(a.model, ANG, a.scale).state_dict().items()}
    rate, ms, per_step = cpu_reference_rate(a.model, a.scale, patches, max(a.steps, 1), a.warmup, 1, sd)
    cores = os.cpu_count() or 1
    sample = (f"{per_step}-patch scene (5x5x32x32 views) per step instead of {a.batch}, minibatch 1 as option.py:45, "
              f"{a.steps} steps; oracle port of the reference (bit-identical to it on CPU), torch {torch.__version__}")
    print(json.dumps({
        "impl": "reference", "metric": "LF patches/sec (5x5x32x32 x%d SR)" % a.scale, "value": rate, "unit": "patches/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a.model, a.scale, a.batch, world),
        "cpu_baseline": {"value": rate, "unit": "patches/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# -------------------------------------------------------------------------------------------------
def cuda_time(fn, iters: int, warmup: int = 1, sync=None):
    """ms per call, CUDA events on the current stream after `warmup` untimed calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


DUMP_BUDGET = 64 * 10 ** 6
DUMP_HEADER = 4096          # room left for each .npy header


def dump_outputs(out_dir: str, arrays: dict):
    """Write each float32 / float64 array as out_dir/<name>.npy, smallest first, within DUMP_BUDGET bytes in all. An array
    larger than what is left is replaced by a fixed sample of its flattened elements (RandomState(0), sorted indices): the
    same arguments give the same sample, so the files of two builds stay comparable."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BUDGET
    written = {}
    for name, arr in sorted(arrays.items(), key=lambda kv: kv[1].nbytes):
        arr = np.ascontiguousarray(arr)
        assert arr.dtype in (np.float32, np.float64), (name, arr.dtype)
        keep = (left - DUMP_HEADER) // arr.itemsize
        if keep <= 0:
            raise ValueError(f"--dump-outputs: no room left for {name}")
        if arr.size > keep:
            idx = np.sort(np.random.RandomState(0).choice(arr.size, keep, replace=False))
            arr = arr.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), arr)
        left -= arr.nbytes + DUMP_HEADER
        written[name] = list(arr.shape)
    return written


def measure_tf32_peak(dev, n: int = 8192):
    """dense TF32 matmul peak with the MEASURED_PEAKS protocol: torch.matmul n^3 (2 n^3 flops), fp32 inputs with
    allow_tf32 (cuBLAS TF32 tensor-core GEMM), best of 10 after warm-up, CUDA events."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b)
        best = 1e30
        for _ in range(10):
            best = min(best, cuda_time(lambda: torch.matmul(a, b), 1, 0))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def oracle_parity(net, model, scale, x_dev, n_check=2):
    """max|net(x) - oracle(x)| and |dPSNR| (against a fixed pseudo ground truth) on the first patches, at the network's OWN
    current weights. The oracle (CPU fp32 restatement of the reference forward) is used as the checker only."""
    from oracle import lf_oracle, nets as onets
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    x = x_dev[:n_check].contiguous()
    y = net(x, [ANG, ANG]).cpu()
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        y_or = onets.forward(model, x.cpu(), sd, ANG, scale)
    err = float((y - y_or).abs().max())
    hr = np.random.RandomState(5).random_sample(tuple(y_or.shape[-2:])).astype(np.float32)
    dps = max(abs(lf_oracle.psnr_view(hr, y[i, 0].numpy()) - lf_oracle.psnr_view(hr, y_or[i, 0].numpy()))
              for i in range(y.shape[0]))
    return {"max_abs": err, "dpsnr_db": float(dps), "tol_max_abs": 1e-3, "tol_dpsnr_db": 0.01, "patches": int(y.shape[0]),
            "out_absmax": float(y_or.abs().max()), "ok": bool(err <= 1e-3 and dps <= 0.01)}


def eager_reference_rate(model, scale, sd_dev, batch, dev, iters=3):
    """the reference algorithm in eager PyTorch on this GPU: fp32, TF32 off (protocol of check_efficiency_official.py:306-330,
    shortened). oracle/nets.forward == the reference forward, bit-exact on CPU."""
    from oracle import nets as onets
    prev = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True          # test.py:59
    try:
        x = torch.rand(batch, 1, ANG * PATCH, ANG * PATCH, device=dev)
        with torch.no_grad():
            ms = cuda_time(lambda: onets.forward(model, x, sd_dev, ANG, scale), iters, 2)
        return {"batch": batch, "ms": ms, "patches_per_s": batch / (ms * 1e-3)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = prev


# -------------------------------------------------------------------------------------------------
def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)

    import lfsr_b200
    from lfsr_b200 import kernels as K, lfutils as U, scene as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    lib = lfsr_b200._native.load()
    if a.no_tc:
        K._default_ops = K.CudaOps(use_tc=False)
    ops = K.default_ops()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"

    def make_net(model, scale):
        torch.manual_seed(1234)                              # seeded constructor-default init (SURVEY 8d)
        return lfsr_b200.load_net(model, ANG, scale).eval().to(dev)

    net = make_net(a.model, a.scale)
    nets = [net]
    launches_of = lambda: lib.lfsr_launch_count() + sum(n.graph_launches for n in nets)

    h0 = scene_side(a.batch)
    s = a.scale
    n_scenes = 4                                              # rotate inputs so no step reuses the previous one
    host_lr, host_hr, dev_lr, dev_hr = [], [], [], []
    for i in range(n_scenes):
        lr, hr = synthetic_scene(h0, s, 100 * rank + i)
        host_lr.append(torch.from_numpy(lr).pin_memory())
        host_hr.append(torch.from_numpy(hr).pin_memory())
        dev_lr.append(torch.from_numpy(lr).to(dev))
        dev_hr.append(torch.from_numpy(hr).to(dev))
    # scene-parallel: every rank drives its OWN scenes (world=1 runner per rank)
    runner = S.SceneRunner(net, ANG, s, h0, h0, PATCH, STRIDE, minibatch=a.batch, device=dev, world=1, rank=0, depth=2)
    assert runner.num_u * runner.num_v == a.batch
    slot0 = runner.device_slot(0)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step, steps, warmup, finish=None):
        for i in range(warmup):
            step(i)
        if finish:
            finish()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = launches_of()
        e0.record()
        for i in range(steps):
            step(warmup + i)
        if finish:
            finish()                                          # drains the pipeline: every copy is inside the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = launches_of() - l0
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    # ---- parity at the weights being timed (rank 0; the other ranks hold the same seeded weights) ----
    parity = None
    if rank == 0:
        ops.divide_rows(dev_lr[0], runner.sub, ANG, h0, h0, PATCH, STRIDE, 0, runner.num_u)
        parity = oracle_parity(net, a.model, s, runner.sub)
        parity["weights"] = "the timed ones: torch.manual_seed(1234), constructor-default init"
        if not parity["ok"]:
            print(f"[bench] PARITY FAILED at the timed weights: {parity}", file=sys.stderr)

    # ---- headline: resident inputs ----
    def step_resident(i):
        runner.run_resident(dev_lr[i % n_scenes], slot0["mosaic"], dev_hr[i % n_scenes], slot0["acc"])

    sampler = ClockSampler(local) if rank == 0 else None
    ms_total, launches = timed(step_resident, a.steps, max(a.warmup, 3))
    clocks = sampler.stop() if sampler else None
    value = a.batch * world * a.steps / (ms_total * 1e-3)
    # slot 0 now holds the last timed step's outputs; the e2e leg below reuses it
    if a.dump_outputs and rank == 0:
        acc = slot0["acc"].cpu().numpy()
        written = dump_outputs(a.dump_outputs, {
            "sr": slot0["mosaic"].cpu().numpy(), "metric_sums": acc,
            "psnr_ssim": np.array(runner.metrics_from_sums(acc), dtype=np.float64)})
        print(f"[bench] outputs of the last timed step -> {a.dump_outputs}: {written}", file=sys.stderr)

    # ---- e2e: host LR + host HR in, host SR mosaic + (psnr, ssim) out, through SceneRunner.submit/result ----
    pending = []
    results = []

    def step_e2e(i):
        pending.append(runner.submit(host_lr[i % n_scenes], host_hr[i % n_scenes]))
        if len(pending) == runner.depth:
            results.append(runner.result(pending.pop(0))[:2])

    def drain_e2e():
        while pending:
            results.append(runner.result(pending.pop(0))[:2])
        torch.cuda.current_stream().wait_stream(runner.d2h)     # the closing event is ordered after the last D2H

    ms_e2e, _ = timed(step_e2e, a.steps, 2, drain_e2e)
    e2e = a.batch * world * a.steps / (ms_e2e * 1e-3)
    h2d_bytes = host_lr[0].numel() * 4 + host_hr[0].numel() * 4
    d2h_bytes = runner.slots[0]["host_sr"].numel() * 4 + runner.slots[0]["host_acc"].numel() * 8

    # ---- sustained: >= a.sustained_s seconds of back-to-back steps with its own clock record ----
    sustained = None
    if not a.quick and a.sustained_s > 0:
        n_sus = max(a.steps, int(a.sustained_s / (ms_total / a.steps * 1e-3)) + 1)
        sampler = ClockSampler(local) if rank == 0 else None
        ms_sus, _ = timed(step_resident, n_sus, 1)
        ck = sampler.stop() if sampler else None
        sustained = {"value": a.batch * world * n_sus / (ms_sus * 1e-3), "unit": "patches/s", "steps": n_sus,
                     "seconds": ms_sus * 1e-3, "clocks": ck}

    tf32_peak = measure_tf32_peak(dev) if rank == 0 else None

    # ---- roofline of the dominant kernel, timed alone with CUDA events on its launch stream ----
    roof = None
    if rank == 0 and hasattr(net, "dominant_kernel"):
        call, info = net.dominant_kernel(a.batch)
        kms = cuda_time(call, 10, 3)
        gbs = info["bytes"] / (kms * 1e-3) / 1e9
        tfl = info["flops"] / (kms * 1e-3) / 1e12
        traffic = tensor_active = None
        try:
            nc = json.load(open(os.path.join(ROOT, "profiles", info.get("ncu_json", "r01_dominant_kernel_ncu.json"))))
            gb = lambda k: float(nc[k]["value"]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[nc[k]["unit"]]
            traffic = (gb("dram__bytes_read.sum") + gb("dram__bytes_write.sum")) * a.batch / 64.0
        except (OSError, KeyError, ValueError):
            pass
        # this kernel moves 0.2x its per-layer bytes through DRAM (the head conv's input never exists) and keeps the tensor
        # pipe busy: it is tensor / shared-memory bound. Its operands are fp16 on the fp16 operand plan (kind::f16 MMAs, fp32
        # accumulate), TF32 otherwise: the yardstick is the measured dense peak of THAT operand type
        f16_dom = bool(net._packed and net._packed.get("f16"))
        peak_t = float(peaks.get("bf16_tflops", 1590.0)) if f16_dom else tf32_peak
        roof = {"bound": "tensor", "achieved": tfl, "peak": peak_t, "unit": "TFLOP/s", "frac": tfl / peak_t,
                "traffic": traffic, "kernel": info["name"], "kernel_ms": kms, "flops_per_launch": info["flops"],
                "operands": "fp16 (kind::f16), fp32 accumulate" if f16_dom else "tf32 (kind::tf32), fp32 accumulate",
                "peak_source": ("MEASURED_PEAKS.json bf16_tflops (16-bit dense tensor peak, burst: kernel timed alone)" if f16_dom else
                                "torch.matmul fp32 inputs, allow_tf32, 8192^3, best of 10, measured in this run (MEASURED_PEAKS "
                                "protocol)") if peaks or not f16_dom else "fallback 1590 TFLOP/s (B200_PROFILING.md)",
                "frac_of_tf32_peak": tfl / tf32_peak, "tf32_peak_tflops": tf32_peak, "fp16_peak_tflops": peaks.get("bf16_tflops"),
                "hbm": {"per_layer_bytes": info["bytes"], "per_layer_gbs": gbs, "per_layer_frac": gbs / hbm_peak,
                        "conv_layer_only_frac": (info["bytes_conv_layer_only"] / (kms * 1e-3) / 1e9 / hbm_peak
                                                 if "bytes_conv_layer_only" in info else None),
                        "dram_traffic_note": "traffic = DRAM bytes of the committed ncu capture of this kernel",
                        "dram_traffic_gbs": traffic / (kms * 1e-3) / 1e9 if traffic else None,
                        "dram_frac": traffic / (kms * 1e-3) / 1e9 / hbm_peak if traffic else None,
                        "peak": hbm_peak, "peak_source": peak_src}}

    def whole_path(model, scale, rate):
        pp = PER_PATCH.get((model, scale))
        if pp is None:
            return None
        w = {"per_layer_bytes_per_patch": pp["layer_bytes"], "achieved_hbm_gbs": rate * pp["layer_bytes"] / 1e9,
             "achieved_hbm_frac": rate * pp["layer_bytes"] / 1e9 / hbm_peak, "hbm_peak_gbs": hbm_peak,
             "achieved_tflops": rate * pp["flops"] / 1e12}
        if tf32_peak:
            w["achieved_tensor_frac_tf32"] = rate * pp["flops"] / 1e12 / tf32_peak
        if "basictrans_flops" in pp and tf32_peak:
            # BasicTrans FLOPs as the reference counts them (dense 160 x 160 attention) over the whole forward's time: a lower
            # bound of the fused kernel's own rate (profiles/run_basictrans.py times it alone)
            w["basictrans_tflops"] = rate * pp["basictrans_flops"] / 1e12
            w["basictrans_tensor_frac_tf32"] = rate * pp["basictrans_flops"] / 1e12 / tf32_peak
            if peaks.get("bf16_tflops"):
                w["basictrans_tensor_frac_fp16"] = rate * pp["basictrans_flops"] / 1e12 / float(peaks["bf16_tflops"])
        return w

    # ---- the other BASELINE configs (rank 0 of a 1-GPU run; multi-GPU runs only add config 5's reduction) ----
    configs, eager = None, None
    if not a.quick and rank == 0 and world == 1:
        configs, eager = {}, {}

        def fwd_rate(nt, B, iters):
            x = torch.rand(B, 1, ANG * PATCH, ANG * PATCH, device=dev)
            ms = cuda_time(lambda: nt.forward_static(x), iters, 2)
            return ms, B / (ms * 1e-3)

        def leg(model, scale, batches, iters=5, with_metrics=False):
            nt = make_net(model, scale)
            nets.append(nt)
            out = {"weights": "random init (seed 1234, constructor defaults)"}
            xs = torch.rand(2, 1, ANG * PATCH, ANG * PATCH, device=dev)
            out["parity"] = oracle_parity(nt, model, scale, xs, 1)
            sweep = {}
            for B in batches:
                ms, rate = fwd_rate(nt, B, iters if B < 256 else 3)
                sweep[str(B)] = {"ms": ms, "patches_per_s": rate}
            out["forward"] = sweep
            best = max(v["patches_per_s"] for v in sweep.values())
            out["roofline"] = whole_path(model, scale, best)
            if with_metrics:      # config 5: batch forward + on-GPU PSNR/SSIM of every patch against its HR patch
                B = batches[-1]
                x = torch.rand(B, 1, ANG * PATCH, ANG * PATCH, device=dev)
                hr = torch.rand(B, 1, ANG * PATCH * scale, ANG * PATCH * scale, device=dev)
                acc = torch.zeros(B * 2 * ANG * ANG, dtype=torch.float64, device=dev)

                def f():
                    y = nt.forward_static(x)
                    acc.zero_()
                    ops.metric_sums_batched(hr, y, B, ANG, PATCH * scale, PATCH * scale, acc)
                ms = cuda_time(f, 3, 1)
                out["forward_plus_metrics"] = {"batch": B, "ms": ms, "patches_per_s": B / (ms * 1e-3)}
            sd_dev = {k: v.detach().to(dev) for k, v in nt.state_dict().items()}
            try:
                eager[f"{model}_x{scale}"] = [eager_reference_rate(model, scale, sd_dev, 64, dev)]
            except Exception as e:  # noqa: BLE001 - the bar is a reported baseline; never lose the bench line over it
                eager[f"{model}_x{scale}"] = {"error": repr(e)[:200]}
            nt.release_workspace()
            nets.remove(nt)
            del nt
            torch.cuda.empty_cache()
            return out

        configs["EPIT_x4"] = leg("EPIT", 4, [64], iters=3)
        configs["DistgSSR_x2"] = leg("DistgSSR", 2, [1, 4, 16, 64, 256])
        configs["DistgSSR_x4"] = leg("DistgSSR", 4, [1, 4, 16, 64, 256])
        configs["LF_InterNet_x4"] = leg("LF_InterNet", 4, [64, 256], with_metrics=True)
        configs["MyEfficientLFNetV4_5_x4"] = leg("MyEfficientLFNetV4_5", 4, [64])
        sd_dev = {k: v.detach().to(dev) for k, v in net.state_dict().items()}
        try:
            eager[f"{a.model}_x{s}"] = [eager_reference_rate(a.model, s, sd_dev, 1, dev, 10),
                                        eager_reference_rate(a.model, s, sd_dev, 64, dev)]
        except Exception as e:  # noqa: BLE001
            eager[f"{a.model}_x{s}"] = {"error": repr(e)[:200]}
        eager["protocol"] = ("oracle/nets.forward (== reference forward) on cuda, fp32, cudnn/matmul allow_tf32=False, "
                             "cudnn.benchmark=True, 2 warm-ups, CUDA events")

    # ---- BASELINE configs[2]: ONE 5x5x512x512 scene, EPIT, rows sharded over the ranks + NCCL all-gather ----
    strong = None
    if not a.quick:
        strong = strong_scaling_leg(S, make_net, dev, dist, world, rank)

    # ---- config 5 across GPUs: LF-InterNet x4, batch 256 per GPU, on-GPU PSNR/SSIM of every patch, and the only
    # collective of scene-level data parallelism: one all-reduce of (sum PSNR, sum SSIM, count) ----
    config5 = None
    if not a.quick and world > 1:
        config5 = config5_multi_gpu(make_net, ops, dev, dist, world, rank)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        sd_cpu = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        rate, ms_cpu, per_step = cpu_reference_rate(a.model, s, 16, 6, 1, 1, sd_cpu)     # ~100 patches, 10-20 s of host work
        rate8, _, _ = cpu_reference_rate(a.model, s, 16, 3, 1, 8, sd_cpu)
        cpu = {"value": rate, "unit": "patches/s", "cores": os.cpu_count() or 1, "kind": "port",
               "sample": f"6 steps of a {per_step}-patch scene (same pipeline, minibatch 1 as option.py:45), torch-CPU oracle "
                         f"port of the reference at the timed weights",
               "minibatch8_value": rate8}

    if rank == 0:
        cfg = workload_config(a.model, s, a.batch, world)
        print(json.dumps({
            "metric": "LF patches/sec (5x5x32x32 x%d SR)" % s, "value": value, "unit": "patches/s", "n_gpus": world,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_total / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": ("f16/tf32" if (net._packed and net._packed.get("f16")) else "tf32") if ops.use_tc else "f32",
            "dtype_note": "tensor-core operands: fp16 between tensor-core layers (10-bit mantissa = TF32's), TF32 where a layer is fed "
                          "fp32; fp32 accumulation, fp32 residual trunks / CUDA-core kernels; outputs within 1e-3 of the fp32 reference "
                          "(parity object)",
            "data": "synthetic", "config": cfg,
            "e2e": {"value": e2e, "unit": "patches/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": ms_e2e / a.steps, "ratio_to_value": e2e / value,
                    "api": "lfsr_b200.scene.SceneRunner.submit(lr_host, hr_host) / result() - the driver train.test() runs on",
                    "copies_declared": {"h2d": ["LR mosaic", "HR label mosaic"], "d2h": ["SR mosaic", "per-view metric sums"]},
                    "pipeline": "2 scenes in flight: H2D / D2H on copy streams under the kernels of the neighbouring scene; "
                                "the closing event waits for the last D2H",
                    "last_psnr_ssim": [float(results[-1][0]), float(results[-1][1])] if results else None},
            "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "roofline": roof,
            "whole_path": whole_path(a.model, s, value / world), "sustained": sustained,
            "tf32_peak_tflops": tf32_peak, "configs": configs, "gpu_eager_baseline": eager, "strong_scaling": strong,
            "config5_multi_gpu": config5, "cpu_baseline": cpu,
        }))
    if dist is not None:
        dist.destroy_process_group()


def config5_multi_gpu(make_net, ops, dev, dist, world, rank, model="LF_InterNet", scale=4, B=256):
    net = make_net(model, scale)
    torch.manual_seed(1000 + rank)
    x = torch.rand(B, 1, ANG * PATCH, ANG * PATCH, device=dev)
    hr = torch.rand(B, 1, ANG * PATCH * scale, ANG * PATCH * scale, device=dev)
    acc = torch.zeros(B * 2 * ANG * ANG, dtype=torch.float64, device=dev)
    hs = PATCH * scale
    tot = torch.zeros(3, dtype=torch.float64, device=dev)

    def f():
        y = net.forward_static(x)
        acc.zero_()
        ops.metric_sums_batched(hr, y, B, ANG, hs, hs, acc)
        v = acc.view(-1, 2)
        psnr = 10.0 * torch.log10(float(hs * hs) / v[:, 0])
        ssim = v[:, 1] / float((hs - 10) * (hs - 10))
        tot[0], tot[1], tot[2] = psnr.sum(), ssim.sum(), float(v.shape[0])
        dist.all_reduce(tot)

    f()
    dist.barrier(); torch.cuda.synchronize()
    ms = cuda_time(f, 3, 1)
    t = torch.tensor([ms], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {"workload": f"{model} x{scale}, batch {B} per GPU + PSNR/SSIM of every patch on the GPU + one 3-scalar all-reduce "
                       "(BASELINE configs[4])", "n_gpus": world, "ms": float(t.item()),
           "patches_per_s": B * world / (float(t.item()) * 1e-3),
           "mean_psnr": float(tot[0] / tot[2]), "mean_ssim": float(tot[1] / tot[2])}
    net.release_workspace()
    del net
    torch.cuda.empty_cache()
    return out


def strong_scaling_leg(S, make_net, dev, dist, world, rank, side=512, model="EPIT", scale=4, minibatch=64):
    """BASELINE configs[2] / SURVEY 8e (ii): one 5x5xside^2 scene, patch-grid rows sharded over the ranks, each rank's
    stitched stripes all-gathered in place (NCCL). Times scene = divide + forwards + integrate + gather (max over ranks,
    CUDA events), the gather alone, and checks the gathered mosaic against locally recomputed rows of another rank."""
    net = make_net(model, scale)
    lr = torch.from_numpy(np.random.RandomState(7).random_sample((ANG * side, ANG * side)).astype(np.float32)).to(dev)
    r = S.SceneRunner(net, ANG, scale, side, side, PATCH, STRIDE, minibatch=minibatch, device=dev, world=world, rank=rank,
                      depth=1, with_metrics=False)
    mosaic = r.slots[0]["mosaic"]
    patches = r.num_u * r.num_v

    def sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    r.run_resident(lr, mosaic)                      # warm-up: graph capture, workspace, NCCL channels
    sync()
    reps = 2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * reps)]
    for i in range(reps):
        ev[3 * i].record()
        r.run_resident(lr, mosaic, gather=False)
        ev[3 * i + 1].record()
        if world > 1:
            r.gather_stripes(mosaic)
        ev[3 * i + 2].record()
    sync()
    scene_ms = sum(ev[3 * i].elapsed_time(ev[3 * i + 2]) for i in range(reps)) / reps
    gather_ms = sum(ev[3 * i + 1].elapsed_time(ev[3 * i + 2]) for i in range(reps)) / reps
    if dist is not None:
        t = torch.tensor([scene_ms, gather_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        scene_ms, gather_ms = float(t[0]), float(t[1])
    # check: rows owned by the LAST rank, recomputed locally on this rank, must equal what the gather delivered
    err = 0.0
    if world > 1:
        chk = S.SceneRunner(net, ANG, scale, side, side, PATCH, STRIDE, minibatch=minibatch, device=dev, world=world,
                            rank=(rank + 1) % world, depth=1, with_metrics=False)
        ref = torch.zeros_like(mosaic)
        chk.run_resident(lr, ref, gather=False)
        a_, b_ = chk.spans[chk.rank]
        v0, v1 = mosaic.view(ANG, r.hs, r.W), ref.view(ANG, r.hs, r.W)
        e = (v0[:, a_:b_] - v1[:, a_:b_]).abs().max().reshape(1)
        dist.all_reduce(e, op=dist.ReduceOp.MAX)
        err = float(e.item())
        del chk, ref
    out = {"workload": f"{model} x{scale}, one 5x5x{side}x{side} scene = {patches} patches, minibatch {minibatch}, "
                       f"rows sharded x{world} + in-place all_gather_into_tensor per view row (BASELINE configs[2])",
           "n_gpus": world, "scene_ms": scene_ms, "gather_ms": gather_ms, "gather_share": gather_ms / scene_ms,
           "patches_per_s": patches / (scene_ms * 1e-3), "rows_per_rank": r.u1 - r.u0,
           "equal_stripes_in_place": bool(r.equal_stripes), "max_abs_gathered_vs_local": err,
           "gathered_bytes_per_rank": int(mosaic.numel() * 4 * (world - 1) / max(world, 1))}
    net.release_workspace()
    del r, net
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
