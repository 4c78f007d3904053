"""On-device scene driver: the hot loop of train.test() (train.py:286-322) without its per-patch
host round trips. LFdivide -> batched forward -> LFintegrate (-> PSNR/SSIM) all stay in HBM; with
torch.distributed initialised, one scene is split by patch-grid rows across the ranks and the
stitched stripes are all-gathered over NCCL (SURVEY.md 8e) - there is no other exchange step.

`SceneRunner` owns everything a scene of one geometry needs (patch buffer, stitched mosaics, metric
accumulators, pinned host staging, copy streams), allocated once: per scene there is no allocation,
no memset of the mosaic (LFintegrate writes every pixel of it), no copy of the network output (each
minibatch's static CUDA-graph output is consumed in place by LFintegrate) and no host sync other
than the one the caller asks for with `result()`. `submit()` / `result()` pipeline scenes: the H2D
of scene i+1 and the D2H of scene i-1 run on copy streams under the kernels of scene i.
The functional API (`super_resolve_scene`, `test_scene`, ...) is what train.test() calls; it runs on
a runner cached on the network.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import kernels as K
from . import lfutils as U


def shard_rows(num_u: int, world: int, rank: int):
    """contiguous, balanced split of the patch-grid rows: rank r owns [lo, hi)."""
    base, extra = divmod(num_u, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def assign_scenes(n: int, world: int, rank: int):
    """(own, tail) of a dataset of n scenes on `world` ranks. `own`: the scenes rank runs alone as single-GPU runs, i in
    [0, world * (n // world)) with i % world == rank (full rounds, no communication). `tail`: the remaining n % world
    scenes, each row-sharded over all ranks; rank i % world keeps its result. Both lists ascend and every tail index is
    above every full-round index, so own + tail is the rank's run order and follows dataset order."""
    if n < 0 or world < 1 or not 0 <= rank < world:
        raise ValueError(f"assign_scenes: n={n}, world={world}, rank={rank}")
    full = world * (n // world)
    return list(range(rank, full, world)), list(range(full, n))


def _dist_state(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


class SceneRunner:
    """LFdivide -> forward -> LFintegrate (-> all-gather) (-> PSNR/SSIM) for scenes of ONE geometry.

    net        a `get_model(args)` module of this package (already on its device)
    h0, w0     LR view size; the LR mosaic is [(ang h0), (ang w0)], the SR mosaic [(ang h0 s), (ang w0 s)]
    minibatch  patches per forward (rounded down to whole patch-grid rows when a row fits, so that LFintegrate reads the
               forward's output buffer directly)
    world/rank row sharding of the patch grid (defaults: torch.distributed state); `group` is the process group of the
               all-gather
    depth      scenes in flight through submit()/result()
    self_ensemble  x8 geometric self-ensemble per patch (include/lfsr.h, lfsr_divide_rows_d8): the network runs on the 8
               flips / transposes of every patch mosaic, the un-transformed outputs are averaged before LFintegrate. Each
               forward covers the 8 variants of whole patch-grid rows; `minibatch` still counts network patches
    """

    def __init__(self, net, ang: int, scale: int, h0: int, w0: int, patch: int = 32, stride: int = 16, minibatch: int = 64,
                 device=None, ops=None, world: Optional[int] = None, rank: Optional[int] = None, group=None,
                 depth: int = 2, with_metrics: bool = True, self_ensemble: bool = False):
        self.net, self.ang, self.scale, self.h0, self.w0 = net, int(ang), int(scale), int(h0), int(w0)
        self.patch, self.stride = int(patch), int(stride)
        self.ops = ops or getattr(net, "_ops", None) or K.default_ops()
        if device is None:
            try:
                device = next(net.parameters()).device
            except StopIteration:
                device = torch.device("cpu")
        self.dev = torch.device(device)
        self.cuda = self.dev.type == "cuda"
        U.check_divide_geometry(h0, w0, patch, stride)
        _, self.num_u, self.num_v = U.divide_geometry(h0, w0, patch, stride)
        w_, r_ = _dist_state(group)
        self.world = w_ if world is None else int(world)
        self.rank = r_ if rank is None else int(rank)
        self.group = group
        self.u0, self.u1 = shard_rows(self.num_u, self.world, self.rank)
        self.pz, self.ss = patch * scale, stride * scale
        self.H, self.W = ang * h0 * scale, ang * w0 * scale         # SR mosaic
        self.hs, self.ws = h0 * scale, w0 * scale
        # the reference slices [0:h, 0:w] out of numU*stride x numV*stride stitched views (utils.py:176-178)
        self.hs_cov, self.ws_cov = min(self.hs, self.num_u * self.ss), min(self.ws, self.num_v * self.ss)
        if (self.hs_cov, self.ws_cov) != (self.hs, self.ws):
            raise ValueError("SceneRunner: the patch grid does not cover the scene (non-overlapping patches)")
        self.self_ensemble = bool(self_ensemble)
        self.nvar = 8 if self.self_ensemble else 1            # network patches per source patch
        row = self.nvar * self.num_v                          # network patches per patch-grid row
        n_own = (self.u1 - self.u0) * row
        self.rows_per_mb = max(1, int(minibatch) // row) if row <= int(minibatch) else 0
        self.minibatch = int(minibatch)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.sub = torch.empty((max(n_own, 1), 1, ang * patch, ang * patch), **f32)
        # a patch-grid row wider than the minibatch is super-resolved in pieces into this row buffer
        self.row_sr = torch.empty((row, 1, ang * self.pz, ang * self.pz), **f32) if self.rows_per_mb == 0 else None
        self.depth = max(1, int(depth))
        self.with_metrics = with_metrics
        self.slots = []
        pin = self.cuda
        for _ in range(self.depth):
            s = dict(
                lr=torch.empty((ang * h0, ang * w0), **f32),
                mosaic=torch.empty((self.H, self.W), **f32),
                acc=torch.zeros(2 * ang * ang, dtype=torch.float64, device=self.dev),
                hr=None, host_lr=None, host_hr=None,
                host_sr=torch.empty((self.H, self.W), dtype=torch.float32, pin_memory=pin),
                host_acc=torch.zeros(2 * ang * ang, dtype=torch.float64, pin_memory=pin),
                done=None, busy=False, has_hr=False, gather_ms=None)
            self.slots.append(s)
        self._n = 0
        if self.cuda:
            self.h2d = torch.cuda.Stream(device=self.dev)
            self.d2h = torch.cuda.Stream(device=self.dev)
        # equal stripes: all-gather in place inside the mosaic, one call per view row a1 (each rank's rows of a view are
        # one contiguous [rows, A*w] block at offset rank * rows) - no staging buffer, no unpack pass
        spans = [shard_rows(self.num_u, self.world, r) for r in range(self.world)]
        self.spans = [(min(lo * self.ss, self.hs), min(hi * self.ss, self.hs)) for lo, hi in spans]
        sizes = {b - a for a, b in self.spans}
        self.equal_stripes = self.world > 1 and len(sizes) == 1 and self.spans[0][0] == 0 and \
            all(self.spans[r][0] == r * (self.spans[0][1]) for r in range(self.world))
        self._pad = None
        if self.world > 1 and not self.equal_stripes:
            mr = max(b - a for a, b in self.spans)
            self._pad = torch.empty((self.world, ang, mr, self.W), **f32)

    # -- device-side pipeline ---------------------------------------------------------------------------------------
    def _forward(self, x):
        fs = getattr(self.net, "forward_static", None)
        return fs(x) if fs is not None else self.net(x, [self.ang, self.ang])

    def run_resident(self, lr_dev: torch.Tensor, mosaic: torch.Tensor, hr_dev: Optional[torch.Tensor] = None,
                     acc: Optional[torch.Tensor] = None, gather: bool = True):
        """the hot path on tensors already in HBM; everything is enqueued on the current stream, nothing syncs."""
        ops, A = self.ops, self.ang
        u0, u1 = self.u0, self.u1
        if self.self_ensemble:
            divide, integrate = ops.divide_rows_d8, ops.integrate_rows_d8
        else:
            divide, integrate = ops.divide_rows, ops.integrate_rows
        row = self.nvar * self.num_v
        if u1 > u0:
            divide(lr_dev, self.sub, A, self.h0, self.w0, self.patch, self.stride, u0, u1)
            if self.rows_per_mb:
                for r in range(u0, u1, self.rows_per_mb):
                    r1 = min(r + self.rows_per_mb, u1)
                    x = self.sub[(r - u0) * row:(r1 - u0) * row]
                    y = self._forward(x)
                    integrate(y, mosaic, A, self.pz, self.ss, self.hs, self.ws, self.num_u, self.num_v, r, r1)
            else:
                for r in range(u0, u1):
                    for c in range(0, row, self.minibatch):
                        c1 = min(c + self.minibatch, row)
                        self.row_sr[c:c1] = self.net(self.sub[(r - u0) * row + c:(r - u0) * row + c1], [A, A])
                    integrate(self.row_sr, mosaic, A, self.pz, self.ss, self.hs, self.ws, self.num_u, self.num_v, r, r + 1)
        if gather and self.world > 1:
            self.gather_stripes(mosaic)
        if hr_dev is not None and acc is not None:
            acc.zero_()
            ops.metric_sums(hr_dev, mosaic, A, self.hs, self.ws, acc)
        return mosaic

    def gather_stripes(self, mosaic: torch.Tensor):
        """all-gather of the per-rank stripes of the stitched mosaic [(a1 h), (a2 w)]: rank r owns rows spans[r] of every
        view row a1. Equal stripes: `ang` in-place all_gather_into_tensor calls (send = the rank's own slice of the receive
        buffer). Ragged stripes: one all_gather_into_tensor through a padded [G, A, max_rows, A*w] buffer + unpack."""
        import torch.distributed as dist
        view = mosaic.view(self.ang, self.hs, self.W)
        if self.equal_stripes:
            a, b = self.spans[self.rank]
            for a1 in range(self.ang):
                dist.all_gather_into_tensor(view[a1], view[a1, a:b], group=self.group)
            return mosaic
        a, b = self.spans[self.rank]
        pad = self._pad
        if b > a:
            pad[self.rank, :, : b - a] = view[:, a:b]
        dist.all_gather_into_tensor(pad.view(-1), pad[self.rank].reshape(-1), group=self.group)
        for r, (a, b) in enumerate(self.spans):
            if r != self.rank and b > a:
                view[:, a:b] = pad[r, :, : b - a]
        return mosaic

    # -- host-facing pipeline -----------------------------------------------------------------------------------------
    def _stage(self, slot, key, src: torch.Tensor, shape):
        """host tensor -> the slot's device tensor (async when the source is pinned; pageable sources go through the
        slot's pinned staging buffer first). Device tensors are used as they are."""
        if src.is_cuda or not self.cuda:
            t = src.to(device=self.dev, dtype=torch.float32).reshape(shape)
            return t.contiguous()
        src = src.reshape(shape)
        dst = slot[key]
        if dst is None:
            dst = slot[key] = torch.empty(shape, dtype=torch.float32, device=self.dev)
        if not src.is_pinned() or src.dtype != torch.float32 or not src.is_contiguous():
            hk = "host_" + key
            if slot[hk] is None:
                slot[hk] = torch.empty(shape, dtype=torch.float32, pin_memory=True)
            slot[hk].copy_(src)
            src = slot[hk]
        with torch.cuda.stream(self.h2d):
            dst.copy_(src, non_blocking=True)
        return dst

    def submit(self, lr: torch.Tensor, hr: Optional[torch.Tensor] = None, readback: bool = True) -> int:
        """enqueue one scene: lr [(a h0), (a w0)] and (optionally) the HR label [(a h0 s), (a w0 s)], host or device tensors.
        Returns a ticket for result(). At most `depth` scenes may be in flight."""
        k = self._n % self.depth
        s = self.slots[k]
        if s["busy"]:
            raise RuntimeError("SceneRunner.submit: all slots are in flight - call result() first")
        self._n += 1
        ctx = torch.cuda.device(self.dev) if self.cuda else _NullCtx()
        with ctx:
            if self.cuda:
                # (no wait before the H2D: the slot's previous scene was consumed by result(), which synchronised on it, so
                # these copies run under whatever the main stream is still computing for the scene before)
                main = torch.cuda.current_stream(self.dev)
            lr_dev = self._stage(s, "lr", lr, (self.ang * self.h0, self.ang * self.w0))
            hr_dev = None
            if hr is not None and self.with_metrics:
                if tuple(hr.shape[-2:]) != (self.H, self.W):
                    raise ValueError(f"HR label {tuple(hr.shape)} does not match the SR mosaic {(self.H, self.W)}")
                hr_dev = self._stage(s, "hr", hr, (self.H, self.W))
            if self.cuda:
                main.wait_stream(self.h2d)
            self.run_resident(lr_dev, s["mosaic"], hr_dev, s["acc"])
            s["has_hr"] = hr_dev is not None
            if self.cuda:
                self.d2h.wait_stream(main)
                with torch.cuda.stream(self.d2h):
                    if readback:
                        s["host_sr"].copy_(s["mosaic"], non_blocking=True)
                    if s["has_hr"]:
                        s["host_acc"].copy_(s["acc"], non_blocking=True)
                    s["done"] = torch.cuda.Event()
                    s["done"].record(self.d2h)
            else:
                if readback:
                    s["host_sr"].copy_(s["mosaic"])
                s["host_acc"].copy_(s["acc"])
        s["busy"], s["readback"] = True, readback
        return self._n - 1

    def result(self, ticket: int):
        """(psnr, ssim, sr) of a submitted scene; sr is the slot's pinned host mosaic (valid until the slot is reused, i.e.
        until `depth` more scenes have been submitted) - or the device mosaic when readback=False. psnr/ssim are None
        without a label. Means over views with value > 0, as utils/utils.py:121-134."""
        s = self.slots[ticket % self.depth]
        if not s["busy"]:
            raise RuntimeError("SceneRunner.result: this ticket is not in flight")
        if s["done"] is not None:
            s["done"].synchronize()
        s["busy"] = False
        psnr = ssim = None
        if s["has_hr"]:
            psnr, ssim = self.metrics_from_sums(s["host_acc"].numpy())
        return psnr, ssim, (s["host_sr"] if s["readback"] else s["mosaic"])

    def metrics_from_sums(self, acc):
        return metrics_from_sums(acc, self.ang, self.hs, self.ws)

    def device_slot(self, k: int = 0):
        return self.slots[k % self.depth]


def metrics_from_sums(acc, ang, hs: int, ws: int):
    """(psnr, ssim) from the per-view sums of lfsr_metric_sums over an ang x ang mosaic of hs x ws views (an
    ang_u x ang_v one for ang = (ang_u, ang_v)): means over views with value > 0, as utils/utils.py:121-134."""
    a = np.asarray(acc, dtype=np.float64).reshape(*U.ang_pair(ang), 2)
    mse = a[..., 0] / float(hs * ws)
    with np.errstate(divide="ignore"):
        P = (10.0 * np.log10(1.0 / mse)).astype(np.float32)
    S = (a[..., 1] / float((hs - 10) * (ws - 10))).astype(np.float32)
    vp, vs = np.sum(P > 0), np.sum(S > 0)
    return (P.sum() / vp if vp > 0 else 0.0), (S.sum() / vs if vs > 0 else 0.0)


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def runner_for(net, ang, scale, h0, w0, patch=32, stride=16, minibatch=64, device=None, ops=None, group=None,
               world=None, rank=None, self_ensemble=False) -> SceneRunner:
    """the SceneRunner of this geometry, cached on the network (dropped with the network)."""
    w_, r_ = _dist_state(group)
    world = w_ if world is None else world
    rank = r_ if rank is None else rank
    cache = net.__dict__.setdefault("_scene_runners", {})
    key = (ang, scale, h0, w0, patch, stride, minibatch, str(device), id(ops), world, rank, id(group), bool(self_ensemble))
    r = cache.get(key)
    if r is None:
        if len(cache) >= 4:                    # scenes of a dataset come in a few sizes; do not hoard HBM
            cache.pop(next(iter(cache)))
        r = cache[key] = SceneRunner(net, ang, scale, h0, w0, patch, stride, minibatch, device, ops, world, rank, group,
                                     self_ensemble=bool(self_ensemble))
    return r


def super_resolve_rows(net, lr_sai: torch.Tensor, ang: int, scale: int, patch: int = 32, stride: int = 16,
                       minibatch: int = 64, rows=None, out_mosaic: torch.Tensor = None, ops=None,
                       self_ensemble: bool = False) -> torch.Tensor:
    """SR of the patch-grid rows `rows` of one scene; returns the full-size SAI mosaic
    [(a1 h s), (a2 w s)] with only the owned stripes written. self_ensemble: see SceneRunner."""
    H, W = lr_sai.shape
    h0, w0 = H // ang, W // ang
    dev = lr_sai.device
    _, num_u, _ = U.divide_geometry(h0, w0, patch, stride)
    r = runner_for(net, ang, scale, h0, w0, patch, stride, minibatch, dev, ops, world=1, rank=0, self_ensemble=self_ensemble)
    if out_mosaic is None:
        out_mosaic = torch.zeros((ang * h0 * scale, ang * w0 * scale), dtype=torch.float32, device=dev)
    saved = (r.u0, r.u1)
    r.u0, r.u1 = (0, num_u) if rows is None else rows
    if (r.u1 - r.u0) * r.nvar * r.num_v > r.sub.shape[0]:
        r.sub = torch.empty(((r.u1 - r.u0) * r.nvar * r.num_v,) + tuple(r.sub.shape[1:]), dtype=torch.float32, device=dev)
    try:
        r.run_resident(lr_sai.to(torch.float32).contiguous(), out_mosaic, gather=False)
    finally:
        r.u0, r.u1 = saved
    return out_mosaic


def super_resolve_scene(net, lr_sai: torch.Tensor, ang: int, scale: int, patch: int = 32, stride: int = 16,
                        minibatch: int = 64, group=None, ops=None, self_ensemble: bool = False, world: Optional[int] = None,
                        rank: Optional[int] = None) -> torch.Tensor:
    """Full scene; when a process group is given (or torch.distributed is initialised with
    world_size > 1) each rank computes its row band and the bands are all-gathered. Returns a device mosaic owned by the
    caller. world/rank override the group's (world=1, rank=0: the whole scene on this rank, no exchange).
    self_ensemble: see SceneRunner."""
    H, W = lr_sai.shape
    h0, w0 = H // ang, W // ang
    dev = lr_sai.device
    r = runner_for(net, ang, scale, h0, w0, patch, stride, minibatch, dev, ops, group, world, rank,
                   self_ensemble=self_ensemble)
    mosaic = torch.empty((r.H, r.W), dtype=torch.float32, device=dev)
    ctx = torch.cuda.device(dev) if dev.type == "cuda" else _NullCtx()
    with ctx:
        return r.run_resident(lr_sai.to(torch.float32).contiguous(), mosaic)


def gather_stripes(mosaic: torch.Tensor, ang: int, h: int, w: int, ss: int, num_u: int, world: int, group=None):
    """all-gather of the per-rank stripes of a stitched mosaic (see SceneRunner.gather_stripes)."""
    import torch.distributed as dist
    r = SceneRunner.__new__(SceneRunner)
    r.ang, r.hs, r.W, r.world, r.rank, r.group = ang, h, ang * w, world, dist.get_rank(group), group
    spans = [shard_rows(num_u, world, k) for k in range(world)]
    r.spans = [(min(lo * ss, h), min(hi * ss, h)) for lo, hi in spans]
    sizes = {b - a for a, b in r.spans}
    r.equal_stripes = len(sizes) == 1 and all(r.spans[k][0] == k * r.spans[0][1] for k in range(world))
    r._pad = None
    if not r.equal_stripes:
        mr = max(b - a for a, b in r.spans)
        r._pad = torch.empty((world, ang, mr, ang * w), dtype=mosaic.dtype, device=mosaic.device)
    return r.gather_stripes(mosaic)


def test_scene(net, lr_sai, hr_sai, ang: int, scale: int, patch: int = 32, stride: int = 16, minibatch: int = 64,
               ops=None, self_ensemble: bool = False, world: Optional[int] = None, rank: Optional[int] = None):
    """(psnr, ssim, sr_mosaic) for one scene - the body of train.test()'s loop on the device. lr/hr may be host or device
    tensors; sr_mosaic is a device tensor that stays valid until the next scene of the same geometry is submitted twice.
    world/rank: see super_resolve_scene. self_ensemble: see SceneRunner."""
    lr_sai = lr_sai.reshape(lr_sai.shape[-2:])
    hr_sai = hr_sai.reshape(hr_sai.shape[-2:])
    H, W = lr_sai.shape
    h0, w0 = H // ang, W // ang
    try:
        dev = next(net.parameters()).device
    except StopIteration:
        dev = lr_sai.device
    if lr_sai.is_cuda:
        dev = lr_sai.device
    r = runner_for(net, ang, scale, h0, w0, patch, stride, minibatch, dev, ops, world=world, rank=rank,
                   self_ensemble=self_ensemble)
    psnr, ssim, sr = r.result(r.submit(lr_sai, hr_sai, readback=False))
    return psnr, ssim, sr


# -- angular window tiling (include/lfsr.h, "Angular window tiling"; DESIGN.md row f-8) ---------------------------------------
def window_origins(n: int, ang: int, stride: Optional[int] = None):
    """origins of the A x A windows along one angular axis of an N-view grid: 0, t, 2t, ... while < N - A, then N - A.
    stride t in [1, A - 1] (None or 0: A - 1, the fewest windows that cover the grid); N = A gives the one origin 0."""
    n, ang = int(n), int(ang)
    if ang < 1 or n < ang:
        raise ValueError(f"window_origins: a {n}-view axis has no {ang}-view window")
    if n == ang:
        return [0]
    t = ang - 1 if not stride else int(stride)
    if not 1 <= t <= ang - 1:
        raise ValueError(f"window_origins: angular stride {t} outside [1, {ang - 1}] (neighbouring windows of {ang} views "
                         f"share at least one view)")
    return list(range(0, n - ang, t)) + [n - ang]


def window_plan(n, ang: int, stride: Optional[int] = None):
    """[(o_u, o_v, modes)] in window order (row-major in (o_u, o_v)) for an N x N grid, or an N_u x N_v one for
    n = (N_u, N_v) (origins per axis, one stride); modes[a1 * ang + a2] is the lfsr_window_accumulate step for window view
    (a1, a2): 0 = store (first window over the view), 1 = add, c >= 2 = add then divide by the view's window count
    c = c_u * c_v (last window over it)."""
    n_u, n_v = U.ang_pair(n)
    orig_u, orig_v = window_origins(n_u, ang, stride), window_origins(n_v, ang, stride)
    cover_u = [[i for i, o in enumerate(orig_u) if o <= x < o + ang] for x in range(n_u)]
    cover_v = [[j for j, o in enumerate(orig_v) if o <= x < o + ang] for x in range(n_v)]
    plan = []
    for i, ou in enumerate(orig_u):
        for j, ov in enumerate(orig_v):
            modes = []
            for a1 in range(ang):
                cu = cover_u[ou + a1]
                for a2 in range(ang):
                    cv = cover_v[ov + a2]
                    if (i, j) == (cu[0], cv[0]):
                        modes.append(0)
                    elif (i, j) == (cu[-1], cv[-1]):
                        modes.append(len(cu) * len(cv))
                    else:
                        modes.append(1)
            plan.append((ou, ov, modes))
    return plan


def _grid_run(net, lr_sai, n, ang, scale, patch, stride, minibatch, group, ops, ang_stride, self_ensemble, world, rank):
    """(runner, N_u x N_v SR mosaic): every window through the scene pipeline of one runner, merged as it completes."""
    lr = lr_sai.reshape(lr_sai.shape[-2:])
    n_u, n_v = U.ang_pair(n)
    ang = int(ang)
    H, W = lr.shape
    if H % n_u or W % n_v:
        raise ValueError(f"super_resolve_grid: LR mosaic {H}x{W} is not a {n_u}x{n_v} grid of views")
    h0, w0 = H // n_u, W // n_v
    plan = window_plan((n_u, n_v), ang, ang_stride)
    dev = lr.device
    if not lr.is_cuda:
        try:
            dev = next(net.parameters()).device
        except StopIteration:
            pass
    r = runner_for(net, ang, scale, h0, w0, patch, stride, minibatch, dev, ops, group, world, rank,
                   self_ensemble=self_ensemble)
    # the windows go through one slot of the runner, taken in turn like a submitted scene (so a test_scene mosaic stays
    # valid as long as documented there)
    s = r.slots[r._n % r.depth]
    if s["busy"]:
        raise RuntimeError("super_resolve_grid: the runner's next slot is in flight - call result() first")
    r._n += 1
    out = torch.empty((n_u * r.hs, n_v * r.ws), dtype=torch.float32, device=dev)
    ctx = torch.cuda.device(dev) if dev.type == "cuda" else _NullCtx()
    with ctx:
        views = lr.to(device=dev, dtype=torch.float32).contiguous().view(n_u, h0, n_v, w0)
        win_lr = s["lr"].view(ang, h0, ang, w0)
        for ou, ov, modes in plan:
            win_lr.copy_(views[ou:ou + ang, :, ov:ov + ang, :])
            r.run_resident(s["lr"], s["mosaic"])
            if n_u == n_v:                    # square grids keep the square entry points (and backends with only those)
                r.ops.window_accumulate(s["mosaic"], out, ang, n_u, r.hs, r.ws, ou, ov, modes)
            else:
                r.ops.window_accumulate_uv(s["mosaic"], out, ang, n_u, n_v, r.hs, r.ws, ou, ov, modes)
    return r, out


def super_resolve_grid(net, lr_sai: torch.Tensor, n, ang: int, scale: int, patch: int = 32, stride: int = 16,
                       minibatch: int = 64, group=None, ops=None, ang_stride: Optional[int] = None,
                       self_ensemble: bool = False, world: Optional[int] = None, rank: Optional[int] = None) -> torch.Tensor:
    """Every view of an N x N light field with a network for A x A inputs (A = ang): lr_sai [(N h0), (N w0)] -> the device
    SR mosaic [(N h0 s), (N w0 s)] owned by the caller; n = (N_u, N_v) for an N_u x N_v light field
    [(N_u h0), (N_v w0)]. The A x A windows of window_plan(n, A, ang_stride) each run exactly
    what super_resolve_scene runs (row-sharded and all-gathered like a scene under a process group, so the result is the
    same on every rank); lfsr_window_accumulate averages the views several windows produce. N = A is super_resolve_scene."""
    return _grid_run(net, lr_sai, n, ang, scale, patch, stride, minibatch, group, ops, ang_stride, self_ensemble, world,
                     rank)[1]


def test_grid(net, lr_sai, hr_sai, n, ang: int, scale: int, patch: int = 32, stride: int = 16, minibatch: int = 64,
              ops=None, ang_stride: Optional[int] = None, self_ensemble: bool = False, world: Optional[int] = None,
              rank: Optional[int] = None):
    """(psnr, ssim, sr_mosaic) of super_resolve_grid against the N x N (or N_u x N_v) HR mosaic: means over all the
    grid's views with value > 0, as test_scene's over A^2."""
    r, sr = _grid_run(net, lr_sai, n, ang, scale, patch, stride, minibatch, None, ops, ang_stride, self_ensemble, world,
                      rank)
    hr = hr_sai.reshape(hr_sai.shape[-2:])
    if tuple(hr.shape) != tuple(sr.shape):
        raise ValueError(f"HR label {tuple(hr.shape)} does not match the SR mosaic {tuple(sr.shape)}")
    n_u, n_v = U.ang_pair(n)
    acc = torch.zeros(2 * n_u * n_v, dtype=torch.float64, device=sr.device)
    ctx = torch.cuda.device(sr.device) if sr.is_cuda else _NullCtx()
    with ctx:
        label = hr.to(device=sr.device, dtype=torch.float32).contiguous()
        if n_u == n_v:
            r.ops.metric_sums(label, sr, n_u, r.hs, r.ws, acc)
        else:
            r.ops.metric_sums_uv(label, sr, n_u, n_v, r.hs, r.ws, acc)
    psnr, ssim = metrics_from_sums(acc.cpu().numpy(), (n_u, n_v), r.hs, r.ws)
    return psnr, ssim, sr
