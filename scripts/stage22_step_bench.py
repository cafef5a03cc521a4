"""A Stage 2.2-shaped training step: the per-subset loop against the batched path (one forward_subsets_grad call per
cluster / leaf pass), in one process, alternating (pipe.batched_subsets = False / True).

Scene scannet_1m_1296x968 (1 M Gaussians, 1296 x 968) with k-means clusters from the library's Quantize_kMeans
(k1 = 64, k2 = 10), as scripts/subset_render_bench.py builds them.  Only the instance features train (`_ins_feat_q`
is a leaf that requires grad; the geometry is frozen, train.py:431-436).  One step, for root r:
  render(render_cluster=True, selected_root_id=r, leaf_cluster_idx=..., rescale=True)      train.py:352-358
  a masked L2 on cluster_imgs[0] against a fixed random target -- a STAND-IN for the loss of train.py:475-489
  backward()
The sweep runs one step per root (all 64) per view.  Reported per path: ms per step (CUDA events and host clock), library
calls and library host waits per step (the boolean-index gathers of the loop add host syncs of their own that are not
counted), the kernel-family breakdown from ogs_profile_read (a separate profiled pass), and the two halves of the step
measured on their own: the root pass (render(render_cluster=True, selected_root_id=r) + loss + backward; one slot) and
the leaf pass (render(leaf_cluster_idx=..., selected_root_id=r) with grad enabled; its images are not in the loss, as in
train.py:367).  Both halves include the view's main image, which both paths render the same way.

  python scripts/stage22_step_bench.py --views 2 --reps 3 --out profiles/r4_stage22_step.json
"""
import argparse
import json
import os
import statistics
import sys
import time
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from opengaussian_b200 import _lib, renderer, synth  # noqa: E402
from opengaussian_b200.kmeans_quantize import Quantize_kMeans  # noqa: E402
from subset_render_bench import Counter, card  # noqa: E402

K1, K2 = 64, 10


class StepCounter(Counter):
    WAITS = Counter.WAITS + ("ogs_raster_forward_subsets_state",)


def pipe(batched):
    return types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False,
                                 batched_subsets=batched)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions per path (alternating)")
    ap.add_argument("--roots", type=int, default=K1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda")
    bg = torch.zeros(3, device=dev)
    gs, cams_s = synth.make_scene("scannet_1m_1296x968", n_views=a.views)
    model = synth.SynthModel(gs, dev)
    q = Quantize_kMeans(num_clusters=K1, num_leaf_clusters=K2, num_iters=10, dim=9)
    q.forward(model, 1, assign=True, mode="root")
    q.iLeafSubNum = torch.full((K1,), K2, dtype=torch.int64)
    q.cluster_assign_all_leaves(model)
    model._ins_feat_q = model._ins_feat_q.detach().requires_grad_(True)
    cluster_idx, leaf_idx = q.cls_ids.clone(), q.leaf_cls_ids.clone()
    cams = [types.SimpleNamespace(FoVx=c.FoVx, FoVy=c.FoVy, image_height=c.image_height, image_width=c.image_width,
                                  world_view_transform=c.world_view_transform.to(dev),
                                  full_proj_transform=c.full_proj_transform.to(dev),
                                  camera_center=c.camera_center.to(dev), bClusterOccur=None) for c in cams_s]
    H, W = int(cams[0].image_height), int(cams[0].image_width)
    gen = torch.Generator(device=dev).manual_seed(0)
    target = torch.rand(6, H, W, device=dev, generator=gen)
    mask = (torch.rand(H, W, device=dev, generator=gen) > 0.5).float()
    common = dict(cluster_idx=cluster_idx, root_num=K1, leaf_num=K2, rescale=True)
    roots = list(range(a.roots))

    def step(batched, cam, r, part):
        torch.manual_seed(r)                    # the same rescale draw on both paths
        kw = dict(common, selected_root_id=r)
        if part in ("step", "root"):
            kw["render_cluster"] = True
        if part in ("step", "leaves"):
            kw["leaf_cluster_idx"] = leaf_idx
        out = renderer.render(cam, model, pipe(batched), bg, 1000, **kw)
        if part != "leaves" and out["cluster_imgs"]:
            loss = ((out["cluster_imgs"][0] - target) ** 2 * mask).mean()
            loss.backward()
        return out

    def sweep(batched, part):
        out = None
        for cam in cams:
            for r in roots:
                out = step(batched, cam, r, part)
        model._ins_feat_q.grad = None
        return out

    result = {"scene": "scannet_1m_1296x968", "views": a.views, "reps": a.reps, "roots": len(roots), "k1": K1, "k2": K2,
              "loss": "masked L2 on cluster_imgs[0] (stand-in for train.py:475-489)",
              "card": dict(zip(("name", "power_limit"), card())), "parts": {}}
    n_steps = len(cams) * len(roots)
    # equality of one step's images and gradients between the paths (last view, every root)
    diffs, slots = [], {"root": 0, "leaves": 0}
    for r in roots:
        g = {}
        for b in (False, True):
            model._ins_feat_q.grad = None
            out = step(b, cams[-1], r, "step")
            g[b] = (out, None if model._ins_feat_q.grad is None else model._ins_feat_q.grad.clone())
        same = all(torch.equal(x.detach(), y.detach()) for k in ("cluster_imgs", "leaf_clusters_imgs")
                   for x, y in zip(g[False][0][k] or [], g[True][0][k] or []))
        slots["root"] += len(g[True][0]["cluster_imgs"] or [])
        slots["leaves"] += len(g[True][0]["leaf_clusters_imgs"] or [])
        if g[False][1] is not None:
            d = (g[False][1] - g[True][1]).abs().max() / g[False][1].abs().max().clamp_min(1e-30)
            diffs.append(float(d))
        result.setdefault("images_equal", True)
        result["images_equal"] &= same
    model._ins_feat_q.grad = None
    result["grad_max_rel_diff"] = max(diffs) if diffs else None
    result["slots_per_step_last_view"] = {k: v / len(roots) for k, v in slots.items()}
    for part in ("step", "root", "leaves"):
        r = {}
        for b in (False, True):          # warm-up
            sweep(b, part)
        times = {False: [], True: []}
        walls = {False: [], True: []}
        for _ in range(a.reps):
            for b in (False, True):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                sweep(b, part)
                e1.record()
                torch.cuda.synchronize()
                walls[b].append((time.perf_counter() - t0) * 1e3 / n_steps)
                times[b].append(e0.elapsed_time(e1) / n_steps)
        for b, label in ((False, "loop"), (True, "batched")):
            with StepCounter() as c:
                torch.cuda.synchronize()
                _lib.profile_enable(True)
                _lib.profile_read()
                sweep(b, part)
                prof = _lib.profile_read()
                _lib.profile_enable(False)
            r[label] = {
                "ms_per_step_events": statistics.median(times[b]),
                "ms_per_step_wall": statistics.median(walls[b]),
                "ms_per_step_events_all": times[b],
                "library_calls_per_step": c.calls / n_steps,
                "library_host_waits_per_step": c.waits / n_steps,
                "kernel_families_per_step": {k: {"ms": v[0] / n_steps, "launches": v[1] / n_steps}
                                             for k, v in prof.items() if v[1]},
            }
        r["speedup_events"] = r["loop"]["ms_per_step_events"] / r["batched"]["ms_per_step_events"]
        r["speedup_wall"] = r["loop"]["ms_per_step_wall"] / r["batched"]["ms_per_step_wall"]
        result["parts"][part] = r
        print(part, {p: (round(r[p]["ms_per_step_events"], 3), round(r[p]["ms_per_step_wall"], 3))
                     for p in ("loop", "batched")}, flush=True)
    txt = json.dumps(result, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
