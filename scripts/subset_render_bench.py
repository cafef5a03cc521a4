"""render()'s cluster / leaf passes: the per-subset loop against the batched path (one forward_subsets call for all
subsets of a view), in one process, alternating, under torch.no_grad().

Scene scannet_1m_1296x968 (1 M Gaussians, 1296 x 968); coarse and fine clusters from the library's own
Quantize_kMeans (k1 = 64 on [ins_feat, xyz], then cluster_assign_all_leaves with k2 = 10), so that the subsets have
the sizes and screen footprints of real clusters.  Workloads (the reference's no-grad sweeps):
  coarse_sweep     render(render_cluster=True, better_vis=True)          construct_pseudo_ins_feat, train.py:755-760
  per_root_leaves  render(selected_root_id=r) for r in 0..63             train.py:846-856
  all_leaves       render(leaf_cluster_idx=..., selected_root_id=None)   render.py / render_lerf_by_text.py
Per workload and path: ms per view from CUDA events and from the host clock, host waits and library launches per view,
the library's kernel-family breakdown (a separate profiled pass), and whether the two paths return equal dicts.

  python scripts/subset_render_bench.py --views 3 --reps 3 --out profiles/r3_subset_render.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opengaussian_b200 import _lib, renderer, synth  # noqa: E402
from opengaussian_b200.kmeans_quantize import Quantize_kMeans  # noqa: E402

PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
K1, K2 = 64, 10
BG = None     # background, set by main() on the device


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:       # noqa: BLE001
        pl = f"unknown ({e})"
    return name, pl


class Counter:
    """Counts library entry points (C-ABI calls) and the ones that wait on the host for the frame's duplicate count."""

    WAITS = ("ogs_raster_forward", "ogs_raster_forward_subsets")

    def __init__(self):
        self.calls = 0
        self.waits = 0
        self.real = _lib.launch

    def __enter__(self):
        def launch(name, device, *args):
            self.calls += 1
            self.waits += name in self.WAITS
            return self.real(name, device, *args)
        _lib.launch = launch
        return self

    def __exit__(self, *exc):
        _lib.launch = self.real
        return False


def run(cams, model, calls, batched):
    """render() of every call on every camera; returns the last camera's outputs."""
    pipe = types.SimpleNamespace(batched_subsets=batched, **vars(PIPE))
    out = None
    with torch.no_grad():
        for cam in cams:
            out = [renderer.render(cam, model, pipe, BG, 1000, **kw) for kw in calls]
    return out


def same(a, b):
    if isinstance(a, list):
        return isinstance(b, list) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.shape == b.shape and torch.equal(a, b)
    return a == b


def main():
    global BG
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions per path (alternating)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda")
    BG = torch.zeros(3, device=dev)
    gs, cams_s = synth.make_scene("scannet_1m_1296x968", n_views=a.views)
    model = synth.SynthModel(gs, dev)
    q = Quantize_kMeans(num_clusters=K1, num_leaf_clusters=K2, num_iters=10, dim=9)
    q.forward(model, 1, assign=True, mode="root")
    q.iLeafSubNum = torch.full((K1,), K2, dtype=torch.int64)
    q.cluster_assign_all_leaves(model)
    model._ins_feat_q = model._ins_feat_q.detach()
    cluster_idx, leaf_idx = q.cls_ids.clone(), q.leaf_cls_ids.clone()
    cams = [types.SimpleNamespace(FoVx=c.FoVx, FoVy=c.FoVy, image_height=c.image_height, image_width=c.image_width,
                                  world_view_transform=c.world_view_transform.to(dev),
                                  full_proj_transform=c.full_proj_transform.to(dev),
                                  camera_center=c.camera_center.to(dev), bClusterOccur=None) for c in cams_s]
    common = dict(cluster_idx=cluster_idx, root_num=K1, leaf_num=K2, rescale=False)
    workloads = {
        "coarse_sweep": [dict(common, render_cluster=True, better_vis=True)],
        "per_root_leaves": [dict(common, leaf_cluster_idx=leaf_idx, selected_root_id=r) for r in range(K1)],
        "all_leaves": [dict(common, leaf_cluster_idx=leaf_idx)],
    }
    sizes = torch.bincount(cluster_idx, minlength=K1)
    result = {"scene": "scannet_1m_1296x968", "views": a.views, "reps": a.reps, "k1": K1, "k2": K2,
              "coarse_cluster_sizes": {"min": int(sizes.min()), "median": int(sizes.median()), "max": int(sizes.max())},
              "card": None, "workloads": {}}
    result["card"] = dict(zip(("name", "power_limit"), card()))
    for name, calls in workloads.items():
        r = {}
        # warm-up of both paths (module loads, allocator, view cache), then the equality check on the last view
        outs = {b: run(cams, model, calls, b) for b in (False, True)}
        r["outputs_equal"] = all(same(x[k], y[k]) for x, y in zip(outs[False], outs[True]) for k in x)
        r["subsets_rendered_last_view"] = sum(len(o["cluster_imgs"] or []) + len(o["leaf_clusters_imgs"] or [])
                                              for o in outs[True])
        del outs
        times = {False: [], True: []}
        walls = {False: [], True: []}
        for _ in range(a.reps):
            for b in (False, True):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                run(cams, model, calls, b)
                e1.record()
                torch.cuda.synchronize()
                walls[b].append((time.perf_counter() - t0) * 1e3 / a.views)
                times[b].append(e0.elapsed_time(e1) / a.views)
        for b, label in ((False, "loop"), (True, "batched")):
            with Counter() as c:
                torch.cuda.synchronize()
                _lib.profile_enable(True)
                _lib.profile_read()
                run(cams, model, calls, b)
                prof = _lib.profile_read()
                _lib.profile_enable(False)
            r[label] = {
                "ms_per_view_events": statistics.median(times[b]),
                "ms_per_view_wall": statistics.median(walls[b]),
                "ms_per_view_events_all": times[b],
                "library_calls_per_view": c.calls / a.views,
                "library_host_waits_per_view": c.waits / a.views,
                "kernel_families_per_view": {k: {"ms": v[0] / a.views, "launches": v[1] / a.views}
                                             for k, v in prof.items() if v[1]},
            }
        r["speedup_events"] = r["loop"]["ms_per_view_events"] / r["batched"]["ms_per_view_events"]
        r["speedup_wall"] = r["loop"]["ms_per_view_wall"] / r["batched"]["ms_per_view_wall"]
        result["workloads"][name] = r
        print(name, json.dumps({k: v for k, v in r.items() if k not in ("loop", "batched")}),
              {p: (round(r[p]["ms_per_view_events"], 3), round(r[p]["ms_per_view_wall"], 3)) for p in ("loop", "batched")},
              flush=True)
    txt = json.dumps(result, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
