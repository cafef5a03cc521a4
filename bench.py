#!/usr/bin/env python
"""bench.py -- headline benchmark of the OpenGaussian hot path on B200.

Metric (BASELINE.json): fwd+bwd frames/sec @ 1 M Gaussians, 1920x1080, SH degree 3, gradients
w.r.t. all rasterizer inputs (SURVEY.md section 8d: "frame" = one GaussianRasterizer forward +
backward).  One process per GPU; every rank renders its own camera views against a full replica of
the Gaussians (views split across ranks, weak scaling) and the parameter gradients are summed
with NCCL all-reduce when N > 1.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

Prints ONE JSON line (rank 0).  `--dump-outputs DIR` also writes what the resident step returned in its last timed
step as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output.
`value` is device-timed with inputs resident in HBM; `e2e` goes
through the public Python API with the per-step inputs -- every view's camera and fp32 [3,H,W]
ground-truth image, what the reference moves per step at train.py:377 -- copied from pinned host
memory, an L1 loss against that image (train.py:384) and the loss scalar read back, inside the timed region.  `--impl reference` times the CPU restatement of the reference
path (oracle/, OpenMP over all host threads) on the same workload.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "fwd+bwd frames/sec @1M Gaussians 1080p"
UNIT = "frames/s"
WORKLOAD = "lerf_1m_1080p"
N_VIEWS = 8


_REAL_STDOUT = None


def quiet_stdout():
    """NCCL (and friends) print banners such as 'NCCL version ...' on the C-level stdout; the contract is
    ONE JSON line there.  Point fd 1 at stderr for the run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, line)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=WORKLOAD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kmeans", action="store_true")
    ap.add_argument("--views-per-step", type=int, default=4,
                    help="views each rank renders per step (gradients accumulate; ONE gradient all-reduce per step)")
    ap.add_argument("--streams", type=int, default=1,
                    help="side streams the views of a step are spread over (dist.render_views_backward)")
    ap.add_argument("--no-profile", action="store_true", help="do not record per-kernel events in the timed region")
    ap.add_argument("--repeats", type=int, default=5, help="timed regions of `steps` steps each; the median is reported")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 2 and 4 legs")
    ap.add_argument("--grad-allreduce", default="auto", choices=["auto", "nvls", "nccl"],
                    help="N > 1: sum the gradients with the library's in-switch kernel (GradArena), with NCCL, or "
                         "(auto) time both and keep the faster")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the resident step returned in its last timed step (images, radii and parameter "
                         "gradients at a fixed, seeded sample of pixels and Gaussians) as DIR/<name>.npy, float32")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    return a


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm = []
        self.reasons = set()
        self.max_mhz = None
        self.ok = False

    def prepare(self):
        """NVML initialisation takes driver locks for ~100 ms: do it BEFORE the timed region, never inside."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# --------------------------------------------------------------------------------------------
def algorithmic_bytes(P, P_vis, N, H, W, C, deg, tile_bits):
    """SURVEY.md section 8d per-frame algorithmic HBM bytes, split per kernel family."""
    b_in = 12 + 12 + 16 + 4 + 4 * 3 * (deg + 1) ** 2
    HW = H * W
    d = {}
    d["preprocess_fwd"] = P * b_in + P_vis * 48
    d["depth_sort_scan"] = P * 16 * 4 + P * 8
    d["emit"] = N * 6 + P * 40
    d["tile_sort"] = N * 12 * ((tile_bits + 7) // 8)
    d["tile_ranges"] = N * 2
    d["blend_fwd"] = N * (4 + 28 + 4 * C + 4) + HW * 4 * (C + 2) + HW * 8
    d["blend_bwd"] = HW * 4 * (C + 2) + HW * 8 + N * (4 + 28 + 4 * C + 4) + P_vis * 4 * (C + 7) * 2
    d["preprocess_bwd"] = P_vis * (40 + b_in) + P * b_in
    return d


def load_traffic():
    """DRAM bytes per launch of each kernel family from the committed ncu summary (profiles/traffic.json)."""
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get("families", {})
    except Exception:
        return None


def median(xs):
    s = sorted(xs)
    n = len(s)
    return s[n // 2] if n % 2 else 0.5 * (s[n // 2 - 1] + s[n // 2])


class Ctx:
    """Process-wide state of one bench run: rank/world, device, barrier, and max-over-ranks timing."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)

    def timed_repeats(self, step, first, K, R, wall=False):
        """R repeats of a timed region of EXACTLY K steps (step(i) for consecutive i), each bracketed by a
        barrier + synchronize on both sides and timed with CUDA events on the launching stream; every repeat's
        time is the max over ranks (and, with wall=True, over the host clock as well).  Returns R times in ms."""
        out, i = [], first
        for _ in range(R):
            self.barrier()
            t0 = time.perf_counter()
            self.e0.record()
            for _k in range(K):
                step(i)
                i += 1
            self.e1.record()
            self.torch.cuda.synchronize()
            ms = self.e0.elapsed_time(self.e1)
            if wall:
                ms = max(ms, (time.perf_counter() - t0) * 1000.0)
            self.barrier()
            out.append(self.max_over_ranks(ms))
        return out, i

    def settle(self, step, first, max_iters=24):
        """Untimed iterations until torch's caching allocator has stopped growing for 4 consecutive steps (the
        binning buffers are sized from a running estimate of num_rendered, so the first frames of a new view set
        still allocate); returns the next step index."""
        torch = self.torch
        i, quiet, last = first, 0, -1
        while i - first < max_iters and quiet < 4:
            step(i)
            i += 1
            torch.cuda.synchronize()
            now = torch.cuda.memory_reserved(self.dev)
            quiet = quiet + 1 if now == last else 0
            last = now
        return i


class RasterWorkload:
    """fwd + bwd of V views per rank per step through opengaussian_b200.dist.render_views_backward on a synthetic
    scene of synth.SCENES; gradients to every rasterizer input (`fused_feat`: the 6 ins_feat channels are composited
    in the same pass and get gradients too).  Resident step: inputs live in HBM.  End-to-end step: every view's camera
    and ground-truth image (fp32 [3,H,W], train.py:377) come from pinned host memory (double-buffered copy stream),
    the loss is L1 against that image (+ the fixed weightings of depth / alpha), and the step's loss scalar is copied
    back and read by the host."""

    def __init__(self, cx, workload, V, streams=1, fused_feat=False, n_views=N_VIEWS):
        import torch
        from opengaussian_b200 import synth
        from opengaussian_b200.rasterizer import GaussianRasterizationSettings
        self.cx, self.V, self.S = cx, V, max(1, min(streams, V))
        self.workload, self.fused_feat = workload, fused_feat
        dev = cx.dev
        kind, P0, W, H, fovx, rad, height, scale_mult = synth.SCENES[workload]
        gs = synth.make_gaussians(P0, kind, 0, scale_mult=scale_mult)
        self.cams = [c.to(dev) for c in synth.orbit_cameras(n_views * cx.world, rad, W, H, fovx, height)][cx.rank::cx.world]
        self.P, self.W, self.H = P0, W, H
        names = ("means3D", "opacities", "shs", "scales", "rotations")
        self.params = {k: gs[k].to(dev).requires_grad_(True) for k in names}
        self.extra = gs["ins_feat"].to(dev).requires_grad_(True) if fused_feat else None
        self.means2D = torch.zeros(P0, 3, device=dev, requires_grad=True)
        self.bg = torch.zeros(3, device=dev)
        self.C = 9 if fused_feat else 3
        gen = torch.Generator().manual_seed(1234 + cx.rank)
        self.G = torch.randn(self.C + 2, H, W, generator=gen).to(dev)      # resident step: fixed N(0,1) loss gradients
        # end-to-end step: the per-view host input of the reference's training step is the ground-truth image,
        # fp32 [3,H,W] (`gt_image = viewpoint_cam.original_image.cuda()`, train.py:377), plus the camera
        self.NS = 3          # staging slots: with the step's one-view lookahead two views are in flight
        self.gt_host = [torch.rand(3, H, W, generator=gen).pin_memory() for _ in range(self.NS)]
        self.settings = [GaussianRasterizationSettings(H, W, c.tanfovx, c.tanfovy, self.bg, 1.0, c.world_view_transform,
                                                       c.full_proj_transform, 3, c.camera_center, False, False)
                         for c in self.cams]
        self.reduced = [self.params[k] for k in names] + ([self.extra] if fused_feat else [])   # all-reduced gradients
        self.grads = self.reduced + [self.means2D]
        self.allreduce = True
        self.keep_step, self.kept = None, None
        self._e2e_ready = False
        # N > 1: the step's gradient buffer lives in symmetric memory and is summed by our own in-switch kernel
        self.arena = None
        if cx.world > 1 and getattr(cx, "grad_allreduce", "auto") != "nccl":
            from opengaussian_b200 import dist as ogd
            _, span = ogd._flat_layout(self.reduced)
            self.arena = ogd.GradArena(span)
            if self.arena.buf is None:
                self.arena = None

    def close(self):
        self.zero_grads()
        if self.arena is not None:
            self.arena.close()
            self.arena = None

    def zero_grads(self):
        for t in self.grads:
            t.grad = None

    def _call(self, rs):
        from opengaussian_b200.rasterizer import GaussianRasterizer
        if self.fused_feat:
            color, radii, depth, alpha, feat = GaussianRasterizer(rs)(means2D=self.means2D, extra_feats=self.extra, **self.params)
            return color, feat, depth, alpha, radii
        color, radii, depth, alpha = GaussianRasterizer(rs)(means2D=self.means2D, **self.params)
        return color, None, depth, alpha, radii

    def _grad_outputs(self, outs, Gd):
        color, feat, depth, alpha = outs[:4]
        C = self.C
        if feat is None:
            return (color, depth, alpha), (Gd[0:3], Gd[C:C + 1], Gd[C + 1:C + 2])
        return (color, feat, depth, alpha), (Gd[0:3], Gd[3:C], Gd[C:C + 1], Gd[C + 1:C + 2])

    def step(self, i):
        """Step i renders views (i * V + v) % len(settings).  Step `keep_step` keeps every view's forward outputs in
        `kept` (references only: no copy, nothing synchronised)."""
        from opengaussian_b200.dist import render_views_backward
        self.zero_grads()
        V = self.V
        kept = {} if i == self.keep_step else None

        def view(v):
            outs = self._call(self.settings[(i * V + v) % len(self.settings)])
            if kept is not None:
                kept[v] = outs
            return self._grad_outputs(outs, self.G)

        render_views_backward(view, list(range(V)), self.reduced, already_split=True, streams=self.S,
                              reduce=self.allreduce)
        if kept is not None:
            self.kept = [kept[v] for v in range(V)]

    # ---- end to end ----
    def _e2e_setup(self):
        torch, dev, H, W = self.cx.torch, self.cx.dev, self.H, self.W
        NS = self.NS
        self.cam_host = [torch.cat([c.world_view_transform.reshape(-1), c.full_proj_transform.reshape(-1),
                                    c.camera_center.reshape(-1)]).cpu().pin_memory() for c in self.cams]
        self.copy_stream = torch.cuda.Stream(dev)
        self.gt_dev = [torch.empty(3, H, W, device=dev) for _ in range(NS)]
        self.cam_dev = [torch.empty(35, device=dev) for _ in range(NS)]
        self.ready = [torch.cuda.Event() for _ in range(NS)]
        self.consumed = [torch.cuda.Event() for _ in range(NS)]
        self.loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.loss_ready = [torch.cuda.Event() for _ in range(2)]
        self.losses = []
        for s in range(NS):
            self.consumed[s].record()
        self._staged_upto = -1
        self._e2e_ready = True

    def _stage(self, j):        # async H2D of view j's inputs on the copy stream (NS rotating slots)
        torch = self.cx.torch
        if j <= self._staged_upto:
            return
        self._staged_upto = j
        s = j % self.NS
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[s])
            self.gt_dev[s].copy_(self.gt_host[s], non_blocking=True)
            self.cam_dev[s].copy_(self.cam_host[j % len(self.cam_host)], non_blocking=True)
            self.ready[s].record(self.copy_stream)

    def _e2e_view(self, j):
        """Forward of view j from staged inputs; the backward is issued by render_views_backward (one view later)."""
        from opengaussian_b200.rasterizer import GaussianRasterizationSettings
        torch = self.cx.torch
        s = j % self.NS
        self._stage(j)
        torch.cuda.current_stream().wait_event(self.ready[s])
        self._stage(j + 1)                          # the next view's inputs travel while this one is rendered
        c = self.cams[j % len(self.cams)]
        cd = self.cam_dev[s]
        rs = GaussianRasterizationSettings(self.H, self.W, c.tanfovx, c.tanfovy, self.bg, 1.0, cd[0:16].view(4, 4),
                                           cd[16:32].view(4, 4), 3, cd[32:35], False, False)
        outs, gouts = self._grad_outputs(self._call(rs), self.G)
        # loss = L1(render, staged ground-truth image) (train.py:384 `l1_loss(image, gt_image)`, utils/loss_utils.py:17);
        # the remaining outputs (features / depth / alpha) receive the metric's fixed N(0,1) gradients directly, so
        # that every gradient path of the rasterizer runs; the scalar read back is the L1 loss
        loss = torch.nn.functional.l1_loss(outs[0], self.gt_dev[s])
        return {"outputs": [loss] + list(outs[1:]), "grads": [None] + list(gouts[1:]), "loss": loss.detach(),
                "after": self.consumed[s].record}   # the staged inputs are free again once the backward has used them

    def e2e_step(self, i):
        """V views from pinned host inputs, one gradient all-reduce, and the step's loss copied to pinned host
        memory.  The copy is asynchronous; the host reads it one step later, so that the read-back of step i does
        not drain the GPU before step i+1 is queued -- every step's loss is still read inside the timed region
        (e2e_flush reads the last one)."""
        from opengaussian_b200.dist import render_views_backward
        if not self._e2e_ready:
            self._e2e_setup()
        self.zero_grads()
        V = self.V
        total = render_views_backward(lambda v: self._e2e_view(i * V + v), list(range(V)), self.reduced,
                                      already_split=True, streams=self.S, reduce=self.allreduce)
        self.loss_host[i % 2].copy_(total.reshape(1), non_blocking=True)
        self.loss_ready[i % 2].record()
        if hasattr(self, "_pending"):
            self._read_loss(self._pending)
        self._pending = i

    def _read_loss(self, i):
        self.loss_ready[i % 2].synchronize()
        self.losses.append(float(self.loss_host[i % 2][0]))     # D2H result of step i, on the host

    def e2e_flush(self):
        if hasattr(self, "_pending"):
            self._read_loss(self._pending)
            del self._pending

    def h2d_bytes_per_step(self):
        return self.V * (3 * self.H * self.W * 4 + 35 * 4)

    def stats(self):
        """Realised workload statistics of view 0 (untimed): N, visible P, list lengths, interaction counts."""
        torch = self.cx.torch
        from opengaussian_b200 import debug
        with torch.no_grad():
            p = self.params
            st = debug.forward_with_state(self.settings[0], p["means3D"].detach(), p["opacities"].detach(),
                                          shs=p["shs"].detach(), scales=p["scales"].detach(),
                                          rotations=p["rotations"].detach(), export=True)
            N_r = int(st["N"])
            P_vis = int((st["radii"] > 0).sum())
            nc = st["n_contrib"].long()
            lens = (st["ranges"][:, 1].long() - st["ranges"][:, 0].long())
            out = {"num_rendered": N_r, "visible": P_vis, "mean_tile_list": N_r / lens.numel(),
                   "mean_n_contrib": float(nc.float().mean()),
                   # pixel-entry interactions (SURVEY.md 8d): every pixel of a tile against the tile's whole list
                   # (what a kernel without early exit walks) and up to each pixel's last contributor (what the
                   # backward walks; the forward stops within one 32-entry batch after it)
                   "interactions_listed": int((lens * 256).sum()), "interactions_to_last_contributor": int(nc.sum())}
            del st
        return out


DUMP_BYTES = 60_000_000      # --dump-outputs: at most this much in all, half for the pixel arrays, half per Gaussian


def dump_outputs(wl, out_dir):
    """Writes what the kept step returned to its caller as float32 DIR/<name>.npy: per view `color` [V,3,S], `feat`
    [V,F,S] (fused feature channels only), `depth` and `alpha` [V,1,S] at S pixels, per view `radii` [V,G], and
    `grad_<input>` [G,...] of every rasterizer input at G Gaussians.  The pixels and Gaussians are a seeded sample
    (all of them when they fit DUMP_BYTES): a function of the workload and --views-per-step only."""
    import numpy as np
    torch = wl.cx.torch
    outs = [tuple(None if t is None else t.detach() for t in o) for o in wl.kept]   # the images are autograd outputs
    images = {nm: torch.stack([o[k] for o in outs]).flatten(2)
              for k, nm in enumerate(("color", "feat", "depth", "alpha")) if outs[0][k] is not None}
    inputs = dict(wl.params, means2D=wl.means2D, **({"ins_feat": wl.extra} if wl.extra is not None else {}))
    grads = {nm: t.grad for nm, t in inputs.items() if t.grad is not None}
    rng = np.random.default_rng(0)

    def sample(n, floats_per_item):
        m = min(n, DUMP_BYTES // 2 // (4 * floats_per_item))
        idx = np.arange(n) if m == n else np.sort(rng.choice(n, m, replace=False))
        return torch.from_numpy(idx).to(wl.cx.dev)

    px = sample(wl.H * wl.W, sum(t.shape[0] * t.shape[1] for t in images.values()))
    gs = sample(wl.P, len(outs) + sum(t[0].numel() for t in grads.values()))
    arrays = {nm: t[:, :, px] for nm, t in images.items()}
    arrays["radii"] = torch.stack([o[4] for o in outs])[:, gs]
    arrays.update({"grad_" + nm: t[gs] for nm, t in grads.items()})
    os.makedirs(out_dir, exist_ok=True)
    for nm, t in arrays.items():
        np.save(os.path.join(out_dir, nm + ".npy"), t.float().cpu().numpy())


def raster_headline(cx, a):
    """The BASELINE metric: fwd+bwd frames/s at 1 M Gaussians, 1080p -- resident, end to end, roofline, breakdown."""
    import gc
    torch = cx.torch
    from opengaussian_b200 import _lib
    wl = RasterWorkload(cx, a.workload, max(1, a.views_per_step), a.streams)
    V, K, R = wl.V, a.steps, max(1, a.repeats)
    stats = wl.stats()
    sampler = ClockSampler(physical_gpu_index(cx.local))
    sampler.prepare()
    i = 0
    for _ in range(a.warmup):
        wl.step(i)
        i += 1
    i = cx.settle(wl.step, i)
    gc.collect()
    gc.disable()                      # no cyclic-GC pause inside the timed regions
    sampler.start()
    # per-kernel events ride along in the timed region (a.no_profile: separate pass)
    alt = None
    if wl.arena is not None and a.grad_allreduce == "auto":
        # both gradient collectives on the same box: the in-switch kernel (arena installed) and NCCL; keep the faster
        for _ in range(2):
            wl.step(i)
            i += 1
        t_nvls, i = cx.timed_repeats(wl.step, i, K, max(2, R // 2))
        wl.zero_grads()
        wl.arena.enable(False)
        for _ in range(2):
            wl.step(i)
            i += 1
        t_nccl, i = cx.timed_repeats(wl.step, i, K, max(2, R // 2))
        use_nvls = median(t_nvls) <= median(t_nccl)
        alt = {"in_switch_kernel_ms_per_step": median(t_nvls) / K, "nccl_ms_per_step": median(t_nccl) / K,
               "used": "in-switch kernel" if use_nvls else "nccl"}
        wl.zero_grads()
        wl.arena.enable(use_nvls)
        cx.prefer_nvls = use_nvls
        if not use_nvls:
            wl.arena_kind_override = "NCCL all_reduce of the flat gradient buffer (faster than the in-switch kernel here)"
        for _ in range(2):
            wl.step(i)
            i += 1
    # the timed region starts on the first camera however many settle steps the allocator took, so that its last
    # step renders the same views in every run
    i += -i % len(wl.settings)
    if a.dump_outputs:
        wl.keep_step = i + R * K - 1
    _lib.profile_enable(not a.no_profile)
    _lib.profile_read()
    times, i = cx.timed_repeats(wl.step, i, K, R)
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    if a.dump_outputs:
        if cx.rank == 0:
            dump_outputs(wl, a.dump_outputs)
        wl.keep_step, wl.kept = None, None
    if a.no_profile:
        _lib.profile_enable(True)
        for _ in range(K):
            wl.step(i)
            i += 1
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile_enable(False)
    exposed = None
    if cx.world > 1:                  # the same region without the gradient all-reduce: the difference is what the
        wl.allreduce = False          # collective costs the step (it is not overlapped with anything it could hide behind)
        t_no, i = cx.timed_repeats(wl.step, i, K, R)
        wl.allreduce = True
        exposed = (median(times) - median(t_no)) / K
    # ---- end to end ----
    j = 0
    for _ in range(3):
        wl.e2e_step(j)
        j += 1
    wl.e2e_flush()

    e2e_times = []
    for _ in range(R):
        cx.barrier()
        t0 = time.perf_counter()
        cx.e0.record()
        for _k in range(K):
            wl.e2e_step(j)
            j += 1
        wl.e2e_flush()               # the last step's loss is read inside the timed region too
        cx.e1.record()
        torch.cuda.synchronize()
        ms = max(cx.e0.elapsed_time(cx.e1), (time.perf_counter() - t0) * 1000.0)
        cx.barrier()
        e2e_times.append(cx.max_over_ranks(ms))
    sampler.stop_flag = True
    sampler.join(timeout=2)
    gc.enable()
    assert len(wl.losses) == 3 + R * K and all(x == x for x in wl.losses)    # every step's loss arrived, none is NaN
    frames = cx.world * V * K
    ms = median(times)
    value = frames / (ms / 1e3)
    e2e_value = frames / (median(e2e_times) / 1e3)
    if value < e2e_value * 0.98:
        msg = (f"inconsistent timing: resident {value:.1f} frames/s below end-to-end {e2e_value:.1f} "
               f"(repeats {times} vs {e2e_times})")
        if frames >= 40 * cx.world and R >= 3:       # a real measurement: refuse to print a line that contradicts itself
            raise RuntimeError(msg)
        print("bench.py: " + msg + " -- region too short to judge", file=sys.stderr)
    rep = {"repeats": R, "resident_ms": [round(t, 3) for t in times], "e2e_ms": [round(t, 3) for t in e2e_times],
           "value_min": frames / (max(times) / 1e3), "value_max": frames / (min(times) / 1e3),
           "rule": "value and e2e are the MEDIAN of the repeats; every repeat times exactly `steps` steps"}
    if alt is not None:
        rep["gradient_collective_choice"] = alt
    return wl, stats, prof, sampler.result(), ms, value, e2e_value, rep, exposed


def issue_roofline(stats, fam_ms, traffic, sm_mhz):
    """SURVEY.md 8d's second bound for the blend kernels: pixel-entry interactions, warp instructions per
    interaction (ncu `smsp__inst_executed.sum` of the committed capture of the same workload) and the fraction
    of the warp-issue peak (148 SMs x 4 schedulers x clock) the kernel sustains inside the timed region."""
    out = {}
    peak_issue = 148 * 4 * (sm_mhz or 1965) * 1e6          # warp instructions per second
    # both kernels walk a pixel's list up to (fwd: one 32-entry batch past) its last contributor
    for fam, inter_key in (("blend_fwd", "interactions_to_last_contributor"), ("blend_bwd", "interactions_to_last_contributor")):
        t = (traffic or {}).get(fam, {})
        wi = t.get("warp_insts_per_frame")
        if fam not in fam_ms or not wi:
            continue
        I = stats[inter_key]
        out[fam] = {"interactions": I, "interactions_kind": inter_key, "warp_insts_per_launch": wi,
                    "warp_insts_per_32_interactions": wi / (I / 32.0), "issue_frac_of_peak": wi / (fam_ms[fam] / 1e3) / peak_issue,
                    # SURVEY.md 8d: I * (22 + 2C) flop forward, 3x that backward, against the 74.4 TFLOP/s non-tensor FP32 peak
                    "fp32_floor_ms": I * (22 + 2 * 3) * (1 if fam == "blend_fwd" else 3) / 74.4e12 * 1e3}
        out[fam]["frac_of_fp32_floor"] = out[fam]["fp32_floor_ms"] / fam_ms[fam]
    return out


def kmeans_leg(cx, a):
    """BASELINE config 5: two-level codebook over 5 M points sharded over the ranks.  Coarse level: k = 64 over
    [ins_feat | xyz] (D = 9); fine level: k = 10 per coarse cluster over ins_feat (D = 6), ALL coarse clusters in one
    segmented launch.  One pass = one Lloyd iteration = ONE kernel launch: assign + fused centroid sums + (N > 1) the
    all-reduce of the partials over NVLink peer memory by the kernel's last CTA + the centre update."""
    torch, dev, world, rank = cx.torch, cx.dev, cx.world, cx.rank
    from opengaussian_b200 import dist as ogd
    from opengaussian_b200.kmeans_quantize import LloydWorkspace, kmeans_assign, lloyd_pass, lloyd_pass_segmented
    Nk = 5_000_000 // world
    g2 = torch.Generator(device=dev).manual_seed(7 + rank)
    fa = torch.rand(Nk, 6, device=dev, generator=g2)
    fb = (torch.rand(Nk, 3, device=dev, generator=g2) - 0.5) * 8
    cen = torch.cat([fa[:64], fb[:64]], 1).contiguous()
    if world > 1:
        cx.dist.broadcast(cen, 0)
    cen0 = cen.clone()
    ids = torch.empty(Nk, dtype=torch.int64, device=dev)
    red = ogd.PeerReducer(64 * 10 * 8 * 8 + 4096) if world > 1 else None
    comm = red.comm if red is not None else None
    if world > 1 and comm is None:
        raise RuntimeError("k-means leg: NVLink peer memory could not be mapped (" + red.kind + ")")
    k1, k2 = 64, 10
    ws_c = LloydWorkspace(dev, k=64, D=9)
    ws_f = LloydWorkspace(dev, k1=k1, k2=k2, D=6)
    state_c = torch.full((64,), 1e-6, device=dev)
    n_eps = (Nk * world) // 10000 + 1

    def coarse_pass():        # ONE launch: assign + sums + [peer all-reduce] + centre update
        lloyd_pass(fa, fb, 1.0, cen, state_c, n_eps * 1e-6, ids, ws_c, comm)

    # fine level on the coarse ids of one assign pass
    kmeans_assign(fa, fb, 1.0, cen0, ids_out=ids)
    coarse_ids = ids.clone()
    leaf_c = fa[:k1 * k2 + 1].contiguous().clone()
    if world > 1:
        cx.dist.broadcast(leaf_c, 0)
    seg_k = torch.full((k1,), k2, dtype=torch.int32, device=dev)
    leaf_ids = torch.empty(Nk, dtype=torch.int64, device=dev)
    state_f = torch.full((k1 * k2,), 1e-6, device=dev)

    def fine_pass():          # ONE launch for all 64 coarse clusters' fine levels
        lloyd_pass_segmented(fa, coarse_ids, leaf_c, seg_k, k2, state_f, leaf_ids, 30, ws_f, comm)

    out = {}
    for name, fn, bytes_pt in (("coarse", coarse_pass, 44), ("fine", fine_pass, 40)):
        for _ in range(3):
            fn()
        ts, _ = cx.timed_repeats(lambda _i: fn(), 0, 20, 3)
        ms = median(ts) / 20
        out[name] = {"ms_per_pass": ms, "gpts_per_s": Nk * world / ms / 1e6,
                     "hbm_frac": (Nk * bytes_pt / (ms / 1e3) / 1e9) / load_peaks()[0], "algorithmic_bytes_per_point": bytes_pt}
    out["coarse"]["k"], out["coarse"]["D"], out["fine"]["k"], out["fine"]["D"] = 64, 9, "10 per coarse cluster (640 rows)", 6
    km = {"metric": "kmeans assign + centroid-sum pass (BASELINE config 5: 5 M points, coarse k=64 D=9; fine k=10 per cluster D=6)",
          "points": Nk * world, "sharding": f"points sharded x{world}" if world > 1 else "single GPU",
          "collective": (red.kind + ", inside the assign kernel's last CTA" if red is not None else None),
          "launches_per_pass": 1, "coarse": out["coarse"], "fine": out["fine"],
          # kept at the top level for continuity with round 1
          "ms_per_pass": out["coarse"]["ms_per_pass"], "gpts_per_s": out["coarse"]["gpts_per_s"], "hbm_frac": out["coarse"]["hbm_frac"]}
    if world > 1:
        # the same passes with 5 M points PER RANK (weak scaling): the strong-scaling figures above leave each rank
        # ~30 us of work per pass, where launch + NVLink round trip are a fixed ~25 us
        del fa, fb, ids, coarse_ids, leaf_ids
        torch.cuda.empty_cache()
        Nw = 5_000_000
        fa = torch.rand(Nw, 6, device=dev, generator=g2)
        fb = (torch.rand(Nw, 3, device=dev, generator=g2) - 0.5) * 8
        ids = torch.empty(Nw, dtype=torch.int64, device=dev)
        kmeans_assign(fa, fb, 1.0, cen0, ids_out=ids)
        coarse_ids = ids.clone()
        leaf_ids = torch.empty(Nw, dtype=torch.int64, device=dev)
        n_eps = (Nw * world) // 10000 + 1
        weak = {}
        for name, fn in (("coarse", coarse_pass), ("fine", fine_pass)):
            for _ in range(3):
                fn()
            ts, _ = cx.timed_repeats(lambda _i: fn(), 0, 20, 3)
            ms = median(ts) / 20
            weak[name] = {"ms_per_pass": ms, "gpts_per_s": Nw * world / ms / 1e6}
        km["weak_scaling"] = dict(weak, points=Nw * world, points_per_rank=Nw)
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        # CPU port (oracle/kmeans_oracle.c, scalar C, 1 thread) on BASELINE config 1's 200 k points.  The reference
        # file itself (scene/kmeans_quantize.py under torch CPU) is not on the GPU box; in the build container it
        # takes 1.45 s for its 6 passes over these 200 k points (BASELINE.md section 3).
        from oracle import kmeans as okm
        n_s = 200_000
        ca, cb, cc = fa[:n_s].cpu().numpy(), fb[:n_s].cpu().numpy(), cen.cpu().numpy()
        okm.assign(ca[:1000], cb[:1000], 1.0, cc)
        t0 = time.perf_counter()
        ids_cpu = okm.assign(ca, cb, 1.0, cc)
        okm.accumulate(ca, cb, 1.0, 64, ids_cpu)
        dt = time.perf_counter() - t0
        km["cpu_baseline"] = {"gpts_per_s": n_s / dt / 1e9, "cores": 1, "kind": "port",
                              "sample": f"{n_s} points, one assign + centroid-sum pass through oracle/kmeans_oracle.c "
                                        "(the reference file needs the reference tree, absent on the GPU box)", "seconds": dt}
    if red is not None:
        red.close()
    return km


def stage1_leg(cx, iters=10, view_cache=False, graph=False):
    """BASELINE config 3 -- OpenGaussian's own training step (stage 1, train.py:352-456) on the synthetic ScanNet-like
    scene, one view per rank per step: ONE fused render (RGB + 6 feature channels + depth + alpha, raw parameters),
    the view's 120 SAM masks built from its id map (get_SAM_mask_and_feat), per-mask feature means, cohesion + separation losses, backward to `_ins_feat`, and on
    N > 1 GPUs the all-reduce of the 24 MB ins_feat gradient.
    view_cache=False: every step projects, duplicates and sorts its view again, as the reference does.
    view_cache=True: the geometry is frozen in this stage (train.py:431-436), so after a camera's first visit its
    records and tile lists stay resident in HBM (rasterizer.ViewCache) and a step runs the feature activation, the
    blend kernels, the mask statistics and the colour-only backward; every view is resident when the timing starts.
    graph=True (needs view_cache): each camera's step is additionally captured as ONE CUDA graph on its second visit
    (graphs.GraphedViewStep) and replayed afterwards -- the ~1 ms of Python / ctypes / autograd per step no longer bounds
    it; the gradient all-reduce of N > 1 stays an ordinary call after the replay."""
    import types
    torch, dev = cx.torch, cx.dev
    from opengaussian_b200 import dist as ogd, rasterizer as rz, synth
    from opengaussian_b200.mask_stats import cohesion_loss, get_SAM_mask_and_feat, mask_feature_mean, separation_loss
    from opengaussian_b200.renderer import render
    name = "scannet_1m_1296x968"
    gs, cams = synth.make_scene(name, n_views=4 * cx.world)
    cams = cams[cx.rank::cx.world]
    pc = synth.SynthModel(gs, dev, stage0=False)
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    cam_ns = [types.SimpleNamespace(FoVx=c.FoVx, FoVy=c.FoVy, image_height=c.image_height, image_width=c.image_width,
                                    world_view_transform=c.world_view_transform.to(dev),
                                    full_proj_transform=c.full_proj_transform.to(dev),
                                    camera_center=c.camera_center.to(dev), bClusterOccur=None) for c in cams]
    H, W = cams[0].image_height, cams[0].image_width
    # every view's own 4-level SAM id map, resident like view.original_sam_mask.cuda() (train.py:686)
    sam_maps = [synth.sam_like_id_map(120, H, W, 4 + v).to(dev) for v in range(len(cam_ns))]
    bg = torch.zeros(3, device=dev)

    def view_loss(i):
        out = render(cam_ns[i % len(cam_ns)], pc, pipe, bg, 1000, rescale=False)
        # train.py:441 -- the [120,H,W] masks are rebuilt from the id map every step, the mask count known from load time
        _, masks, _ = get_SAM_mask_and_feat(sam_maps[i % len(cam_ns)], level=0, num_mask=120)
        mean = mask_feature_mean(out["ins_feat"], masks, image_mask=out["silhouette"])
        return separation_loss(mean, 1000) + 0.1 * cohesion_loss(out["ins_feat"], masks, mean)

    def step(i):
        pc._ins_feat.grad = None
        ogd.render_views_backward(view_loss, [i], [pc._ins_feat], already_split=True)

    gstep = None
    if graph:
        from opengaussian_b200.graphs import GraphedViewStep, geometry_guard
        gstep = GraphedViewStep(view_loss, [pc._ins_feat], guard=geometry_guard(pc), key=lambda i: i % len(cam_ns))

        def step(i):       # noqa: F811
            gstep(i)
            if cx.world > 1:
                ogd.allreduce_gradients([pc._ins_feat])

    rz.view_cache.clear()
    rz.view_cache.enabled = bool(view_cache)
    n_warm = (3 if graph else 1) * len(cam_ns) + 2
    try:
        for i in range(n_warm):
            step(i)
        ts, _ = cx.timed_repeats(step, n_warm, iters, 3)
        vc = rz.view_cache.stats()
    finally:
        rz.view_cache.enabled = False
        rz.view_cache.clear()
    ms = median(ts) / iters
    res = {"metric": "Stage-1 training steps/s (fused render + mask means + cohesion/separation losses, fwd+bwd"
                     + (", ins_feat gradient all-reduce)" if cx.world > 1 else ")"),
           "workload": name, "masks": 120, "views_per_step": cx.world, "ms_per_step": ms,
           "steps_per_s": 1000.0 / ms, "views_per_s": cx.world * 1000.0 / ms,
           "note": "the reference does 4 forward + 2 backward rasterizations and [M,6,H,W] mask tensors per step"}
    if view_cache:
        res["view_cache"] = {"resident_views": vc["entries"], "bytes_per_view": vc["bytes"] // max(vc["entries"], 1),
                             "hits": vc["hits"], "misses": vc["misses"],
                             "what": "frozen geometry: per-camera records + depth-sorted tile lists kept in HBM after the "
                                     "first visit; a step = feature activation + blend fwd + mask statistics + colour-only "
                                     "bwd.  Images bit-identical to the uncached step (tests/test_view_cache_gpu.py)"}
    if gstep is not None:
        res["cuda_graph"] = dict(gstep.stats(), what="one captured graph per camera (fwd + losses + bwd), replayed with one launch; "
                                                     "tests/test_graphs_gpu.py compares replay with the eager step")
    return res


def named_config_leg(cx, workload, V, fused_feat, K=8, R=3, label=""):
    """One BASELINE config as a view-parallel fwd+bwd run: frames/s resident, with the exposed collective on N > 1."""
    torch = cx.torch
    wl = RasterWorkload(cx, workload, V, fused_feat=fused_feat, n_views=4)
    if wl.arena is not None and not getattr(cx, "prefer_nvls", True):
        wl.arena.enable(False)           # the headline leg found NCCL faster on this box
    i = 0
    for _ in range(3):
        wl.step(i)
        i += 1
    i = cx.settle(wl.step, i, 12)
    ts, i = cx.timed_repeats(wl.step, i, K, R)
    ms = median(ts) / K
    res = {"config": label, "workload": workload, "gaussians": wl.P, "image": [wl.W, wl.H], "channels": wl.C,
           "views_per_step_per_rank": V, "ms_per_step": ms, "frames_per_s": cx.world * V / (ms / 1e3)}
    if cx.world > 1:
        wl.allreduce = False
        t_no, i = cx.timed_repeats(wl.step, i, K, R)
        wl.allreduce = True
        res["collective_exposed_ms_per_step"] = ms - median(t_no) / K
        res["allreduce_bytes"] = sum(t.numel() for t in wl.reduced) * 4
        res["collective_kind"] = (wl.arena.kind if (wl.arena is not None and getattr(cx, "prefer_nvls", True))
                                  else "NCCL all_reduce of the flat gradient buffer")
    wl.close()
    del wl
    torch.cuda.empty_cache()
    return res


def sweep_leg(cx, n_views_per_rank=4):
    """Forward-only sweep (construct_pseudo_ins_feat / Stage-3 association, train.py:676-681,755-760,846-856): the
    views are split over the ranks, every rank renders its views (no gradients, no collective for the images) and
    fills its columns of a per-view table `match_info [k1*k2, V, 3]`; the columns are merged once at the end
    (dist.merge_view_columns) and the per-cluster object counts with one all-reduce(max)."""
    import types
    torch, dev = cx.torch, cx.dev
    from opengaussian_b200 import dist as ogd, synth
    from opengaussian_b200.renderer import render
    gs, cams = synth.make_scene("scannet_1m_1296x968", n_views=n_views_per_rank * cx.world)
    Vt = len(cams)
    pc = synth.SynthModel(gs, dev, stage0=False)
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    bg = torch.zeros(3, device=dev)
    mine = ogd.view_indices(Vt)
    cam_ns = {v: types.SimpleNamespace(FoVx=cams[v].FoVx, FoVy=cams[v].FoVy, image_height=cams[v].image_height,
                                       image_width=cams[v].image_width,
                                       world_view_transform=cams[v].world_view_transform.to(dev),
                                       full_proj_transform=cams[v].full_proj_transform.to(dev),
                                       camera_center=cams[v].camera_center.to(dev), bClusterOccur=None) for v in mine}
    table = torch.zeros(640, Vt, 3, device=dev)
    sub = torch.zeros(64, dtype=torch.int32, device=dev)

    def sweep(_i):
        with torch.no_grad():
            for v in mine:
                out = render(cam_ns[v], pc, pipe, bg, 1000, rescale=False)
                table[:, v, 0] = out["ins_feat"].mean()          # stand-in for the per-view association statistics
                sub[v % 64] = max(int(v), 1)
            merged = ogd.merge_view_columns(table)
            ogd.allreduce_max(sub)
        return merged

    sweep(0)
    ts, _ = cx.timed_repeats(sweep, 0, 2, 3)
    ms = median(ts) / 2
    return {"metric": "forward-only sweep views/s (fused render per view, views split over ranks, one merge of the per-view table)",
            "workload": "scannet_1m_1296x968", "views": Vt, "ms_per_sweep": ms, "views_per_s": Vt / (ms / 1e3)}


def comparator_leg(cx, a):
    """>= 10x target of BASELINE.json: the product against the upstream-STRUCTURE restatement of the reference CUDA
    rasterizer (baseline/upstream_structure.cu) on the metric's workload and on the Stage-1 step's rasterizer work."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import comparator as cmp
    from opengaussian_b200 import synth
    if not os.path.exists(cmp.COMPARATOR):
        return {"unavailable": "baseline/_build/libogs_upstream_structure.so not built (python baseline/build_comparator.py)"}
    gs, cams = synth.make_scene(a.workload, n_views=2)
    frame = cmp.frame_comparison(gs, cams[0], cx.dev, iters=10, warmup=3)
    gs, cams = synth.make_scene("scannet_1m_1296x968", n_views=2)
    st1 = cmp.stage1_comparison(gs, cams[0], cx.dev, iters=8, warmup=2)
    return {"frames_per_s": frame["upstream_structure"]["frames_per_s"], "product_frames_per_s_same_driver": frame["product"]["frames_per_s"],
            "ratio": frame["speedup"], "workload": a.workload,
            "stage1_step_rasterizer_work": dict(st1, workload="scannet_1m_1296x968",
                                                what="reference: 4 forward + 2 backward 3-channel passes; product: 1 fused 9-channel forward + colour-only backward"),
            "parity": "tests/test_comparator_gpu.py checks the comparator against the CPU oracle (images 1e-5, gradients 1e-3 per element)",
            "note": cmp.NOTE}


def run_ours(a):
    quiet_stdout()
    cx = Ctx()
    cx.grad_allreduce = a.grad_allreduce
    torch, world, rank = cx.torch, cx.world, cx.rank
    from opengaussian_b200 import _lib, dist as ogd
    _lib.lib()   # fails loudly if the CUDA library is missing
    from opengaussian_b200 import rasterizer as _rz
    _rz.view_cache.enabled = False   # every leg re-derives its views' geometry unless it says otherwise (stage1_step_view_cache)
    ogd.bind_to_gpu_numa_node(cx.local)      # pinned host buffers on the GPU's own NUMA node (8 ranks share the host)

    wl, stats, prof, clocks, ms, value, e2e_value, rep, exposed = raster_headline(cx, a)
    P, W, H, V = wl.P, wl.W, wl.H, wl.V
    N_r, P_vis = stats["num_rendered"], stats["visible"]
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    tile_bits = max(1, (tiles - 1).bit_length())
    h2d, d2h = wl.h2d_bytes_per_step(), 4
    n_cams = len(wl.cams)
    coll_kind = getattr(wl, "arena_kind_override", None) or \
        (wl.arena.kind if wl.arena is not None else "NCCL all_reduce of the flat gradient buffer")
    wl.close()
    del wl
    torch.cuda.empty_cache()

    extras = {}
    if not a.no_kmeans:
        extras["kmeans"] = kmeans_leg(cx, a)
        extras["stage1_step"] = stage1_leg(cx)
        extras["stage1_step_view_cache"] = stage1_leg(cx, view_cache=True)
        extras["stage1_step_view_cache_graph"] = stage1_leg(cx, iters=20, view_cache=True, graph=True)
    if not a.no_configs:
        cfgs = {}
        cfgs["2_blender_300k_800"] = named_config_leg(cx, "blender_300k_800", 4, True, label="config 2: 300 k Gaussians, SH deg 3, 800x800, fwd+bwd RGB+ins_feat")
        cfgs["4_lerf_3m_1080p"] = named_config_leg(cx, "lerf_3m_1080p", 2, False, K=6, label="config 4: 3 M Gaussians, 1920x1080, view-parallel render + gradient all-reduce")
        cfgs["3_scannet_stage1"] = "see stage1_step"
        cfgs["5_two_level_codebook"] = "see kmeans"
        if world > 1:
            cfgs["forward_only_sweep"] = sweep_leg(cx)
        extras["configs"] = cfgs

    # ---- roofline of the dominant kernel ----
    peak, peak_src = load_peaks()
    alg = algorithmic_bytes(P, P_vis, N_r, H, W, 3, 3, tile_bits)
    fam_ms = {k: (v[0] / max(v[1], 1)) for k, v in prof.items() if v[1] > 0}
    dom = max((k for k in fam_ms if k in alg), key=lambda k: prof[k][0])
    ach = alg[dom] / (fam_ms[dom] / 1e3) / 1e9
    traffic = load_traffic()
    issue = issue_roofline(stats, fam_ms, traffic, clocks.get("sm_mhz"))
    blend = dom in ("blend_fwd", "blend_bwd")
    roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": (traffic.get(dom, {}).get("dram_bytes_per_frame") if traffic else None),
                "traffic_source": "profiles/traffic.json (ncu --set full dram__bytes_read+write per launch)" if traffic else None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom],
                "ms_per_launch": fam_ms[dom],
                "issue": issue,
                "note": ("the contract's HBM fraction; this kernel is bound by FP32 instruction issue, not HBM (SURVEY 8d): "
                         "see `issue` for interactions, warp instructions per 32 interactions and the fraction of the "
                         "148 x 4 x clock issue peak") if blend else "HBM-bound kernel"}
    breakdown = {k: {"ms_per_launch": fam_ms[k], "launches": prof[k][1],
                     "algorithmic_bytes": alg.get(k),
                     "dram_bytes_ncu": (traffic.get(k, {}).get("dram_bytes_per_frame") if traffic else None),
                     "hbm_frac": (alg[k] / (fam_ms[k] / 1e3) / 1e9 / peak) if k in alg else None} for k in fam_ms}
    own = ("preprocess_fwd", "emit", "tile_ranges", "blend_fwd", "blend_bwd", "preprocess_bwd")
    gpu_launches = sum(prof[k][1] for k in own if k in prof) // max(1, a.repeats if not a.no_profile else 1)
    frame_bytes = sum(alg.values())
    ms_step = ms / a.steps

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": a.workload, "gaussians": P, "image": [W, H], "sh_degree": 3, "views_per_rank": n_cams,
                   "views_per_step_per_rank": V, "streams": max(1, min(a.streams, V)),
                   "gradients": "all inputs (means3D, means2D, opacities, shs, scales, rotations)",
                   "parallelism": f"view-parallel x{world}" + (" + one NCCL grad allreduce per step" if world > 1 else ""),
                   "l2": "inputs larger than L2 (236 MB parameters + 8 rotating views per rank)",
                   **stats},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": gpu_launches,
        "roofline": roofline,
        "repeat": rep,
        "frame_hbm": {"algorithmic_bytes": frame_bytes, "frames_per_step": V,
                      "frac_of_peak": V * frame_bytes / (ms_step / 1e3) / 1e9 / peak},
        "breakdown": breakdown,
    }
    if exposed is not None:
        out["collective"] = {"exposed_ms_per_step": exposed, "bytes": (P * 59 + 64 * 5) * 4, "kind": coll_kind,
                             "how": "median step time with minus without the gradient all-reduce"}
    out.update(extras)
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        out["gpu_comparator"] = comparator_leg(cx, a)
        out["cpu_baseline"] = cpu_frame_baseline(a.workload, steps=1, warmup=0)
    if rank == 0:
        emit(out)
    if world > 1:
        cx.dist.destroy_process_group()


# --------------------------------------------------------------------------------------------
def cpu_frame_baseline(workload, steps, warmup):
    """Times the CPU oracle (the restated reference path, OpenMP) on full frames of the workload."""
    from opengaussian_b200 import synth
    from oracle import lib
    from oracle import raster as orc
    import numpy as np
    kind, P0, W, H, fovx, rad, height, scale_mult = synth.SCENES[workload]
    gs = synth.make_gaussians(P0, kind, 0, scale_mult=scale_mult)
    cams = synth.orbit_cameras(N_VIEWS, rad, W, H, fovx, height)
    g = {k: (v.numpy() if hasattr(v, "numpy") else v) for k, v in gs.items()}
    # every host thread this process may run on (torchrun exports OMP_NUM_THREADS=1: override it)
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cores = int(lib().ogs_oracle_set_threads(avail))
    rng = np.random.default_rng(0)
    gc = rng.standard_normal((3, H, W)).astype(np.float32)
    gd = rng.standard_normal((H, W)).astype(np.float32)
    ga = rng.standard_normal((H, W)).astype(np.float32)

    def frame(i):
        c = cams[i % len(cams)]
        oc = orc.Camera(W=W, H=H, tanfovx=c.tanfovx, tanfovy=c.tanfovy, view=c.world_view_transform.numpy().reshape(-1),
                        proj=c.full_proj_transform.numpy().reshape(-1), campos=c.camera_center.numpy())
        st = orc.forward(oc, g["means3D"], g["opacities"], g["scales"], g["rotations"], shs=g["shs"])
        orc.backward(st, gc, gd, ga)

    for i in range(warmup):
        frame(i)
    t0 = time.perf_counter()
    for i in range(steps):
        frame(warmup + i)
    dt = time.perf_counter() - t0
    return {"value": steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} full fwd+bwd frame(s) of {workload} through oracle/raster_oracle.c (C, OpenMP)",
            "seconds": dt}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from opengaussian_b200 import synth
    _, synth_P, synth_W, synth_H = synth.SCENES[a.workload][:4]
    steps = max(1, a.steps)
    warm = max(0, a.warmup)
    # bounded: a full CPU frame costs seconds; keep the whole run within a few minutes
    t0 = time.perf_counter()
    probe = cpu_frame_baseline(a.workload, steps=1, warmup=0)
    per = probe["seconds"]
    budget = 150.0
    if per * (steps + warm) > budget:
        warm = min(warm, 1)
        steps_run = max(1, int((budget - per * warm) / per))
    else:
        steps_run = steps
    base = cpu_frame_baseline(a.workload, steps=steps_run, warmup=warm)
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": a.gpus,
           "steps": steps_run, "warmup": warm, "ms_per_step": 1000.0 / base["value"], "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": a.workload, "gaussians": synth_P, "image": [synth_W, synth_H], "sh_degree": 3,
                      "gradients": "all inputs (means3D, means2D, opacities, shs, scales, rotations)",
                      "note": "CPU restatement of the reference rasterizer path (the upstream CUDA source is absent "
                              "from the reference tree); each step is one full fwd+bwd frame; steps capped to keep "
                              "the run within minutes" if steps_run != steps else
                              "CPU restatement of the reference rasterizer path; each step is one full fwd+bwd frame"},
           "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": time.perf_counter() - t0}
    emit(out)


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
