"""Segmented kNN (csrc/knn.cu) against what it replaces, in one process, alternating old and new, medians of --reps.

(a) render()'s post_process for all leaves of a view on scannet_1m_1296x968 (1 M Gaussians, 1296 x 968; coarse and
    fine clusters from the library's Quantize_kMeans as in scripts/subset_render_bench.py):
    render(leaf_cluster_idx=..., post_process=True, better_vis=True), the leaf plan alone (_plan_leaves) and the whole
    call, with the per-leaf _post_process loop (one cdist + topk and two host reads per leaf) against the segmented
    pass (_post_process_slots).  better_vis=True because the per-leaf loop fails on a leaf the view does not see.
(b) knn_points(x, x, K) against chunked cdist + topk (renderer._knn_mean_dists) for n in {1e4, 1e5, 4e5}, K = sqrt(n),
    with the pair count (n^2) and the kernel's time per pair.
Times: host clock around work that ends in a device synchronise ((a): the plan ends in a host read anyway) and CUDA
events ((b)).  The card's name and power limit are read in the same run.

  python scripts/knn_bench.py --out profiles/knn_bench.json
"""
import argparse
import json
import math
import os
import statistics
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opengaussian_b200 import knn, renderer, synth  # noqa: E402
from opengaussian_b200.kmeans_quantize import Quantize_kMeans  # noqa: E402
from subset_render_bench import card  # noqa: E402

PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
K1, K2 = 64, 10


def loop_slots(subset, S, means3D):
    """The per-leaf loop (_plan_leaves before the segmented pass): _post_process once per slot."""
    counts = []
    for k in range(S):
        filt = subset == k
        post = renderer._post_process(filt, means3D)
        subset = torch.where(filt & ~post, -1, subset).to(torch.int32)
        counts.append(int(post.sum()))
    return subset, counts


SEGMENTED = renderer._post_process_slots


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def alternate(paths, reps, timer):
    """{name: median ms}, running the paths in turn reps times after one warm-up each; also the last outputs."""
    times = {k: [] for k in paths}
    outs = {}
    for k, fn in paths.items():
        outs[k] = timer(fn)[1]
    for _ in range(reps):
        for k, fn in paths.items():
            ms, outs[k] = timer(fn)
            times[k].append(ms)
    return {k: statistics.median(v) for k, v in times.items()}, outs


def render_workload(reps, dev):
    gs, cams_s = synth.make_scene("scannet_1m_1296x968", n_views=1)
    model = synth.SynthModel(gs, dev)
    q = Quantize_kMeans(num_clusters=K1, num_leaf_clusters=K2, num_iters=10, dim=9)
    q.forward(model, 1, assign=True, mode="root")
    q.iLeafSubNum = torch.full((K1,), K2, dtype=torch.int64)
    q.cluster_assign_all_leaves(model)
    model._ins_feat_q = model._ins_feat_q.detach()
    c = cams_s[0]
    cam = types.SimpleNamespace(FoVx=c.FoVx, FoVy=c.FoVy, image_height=c.image_height, image_width=c.image_width,
                                world_view_transform=c.world_view_transform.to(dev),
                                full_proj_transform=c.full_proj_transform.to(dev),
                                camera_center=c.camera_center.to(dev), bClusterOccur=None)
    bg = torch.zeros(3, device=dev)
    kw = dict(leaf_cluster_idx=q.leaf_cls_ids.clone(), post_process=True, better_vis=True, rescale=False, root_num=K1,
              leaf_num=K2)
    captured = {}
    plan = renderer._plan_leaves

    def capture(*args):
        captured["args"] = args
        return plan(*args)

    renderer._plan_leaves = capture
    try:
        with torch.no_grad():
            renderer.render(cam, model, PIPE, bg, 1000, **kw)
    finally:
        renderer._plan_leaves = plan
    args = captured["args"]
    sizes = torch.bincount(args[0][args[4] & args[5] & (args[0] >= 0)], minlength=K1 * K2)     # the 100-point rule
    cand = [i for i in range(K1 * K2) if int(sizes[i]) >= 100]
    pairs = sum(int(sizes[i]) ** 2 for i in cand)

    def with_slots(fn, impl):
        def run():
            renderer._post_process_slots = impl
            try:
                return fn()
            finally:
                renderer._post_process_slots = SEGMENTED
        return run

    def do_plan():
        return plan(*args)

    def do_render():
        torch.manual_seed(0)
        with torch.no_grad():
            return renderer.render(cam, model, PIPE, bg, 1000, **kw)

    plan_ms, plan_out = alternate({"loop": with_slots(do_plan, loop_slots), "segmented": with_slots(do_plan, SEGMENTED)},
                                  reps, host_ms)
    render_ms, render_out = alternate({"loop": with_slots(do_render, loop_slots),
                                       "segmented": with_slots(do_render, SEGMENTED)}, reps, host_ms)
    a, b = plan_out["loop"], plan_out["segmented"]
    return {"scene": "scannet_1m_1296x968", "candidate_leaves": len(cand), "candidate_points": int(sizes[cand].sum()),
            "pairs": pairs, "plan_ms": plan_ms, "render_ms": render_ms,
            "plan_same_leaves": a[0] == b[0], "plan_points_differing": int((a[1] != b[1]).sum()),
            "leaves_kept": len(b[0]),
            "render_same_leaf_ids": render_out["loop"]["occured_leaf_id"] == render_out["segmented"]["occured_leaf_id"]}


def knn_workload(reps, dev):
    out = []
    for n in (10_000, 100_000, 400_000):
        K = math.isqrt(n)
        x = (torch.rand(1, n, 3, generator=torch.Generator().manual_seed(n)) * 4 - 2).to(dev)
        ms, res = alternate({"cdist_topk": lambda: renderer._knn_mean_dists(x[0], K),
                             "knn_points": lambda: knn.knn_points(x, x, K=K).dists[0]}, reps, event_ms)
        d_old, d_new = res["cdist_topk"], res["knn_points"]
        out.append({"n": n, "K": K, "pairs": n * n, "ms": ms, "knn_ns_per_pair": ms["knn_points"] * 1e6 / (n * n),
                    "max_abs_diff": float((d_old - d_new).abs().max()),
                    "max_rel_diff_vs_cdist": float(((d_old - d_new).abs() / d_new.clamp_min(1e-12)).max())})
        del d_old, d_new, res
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "knn_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda")
    name, power = card()
    result = {"card": name, "power_limit": power, "reps": a.reps, "statistic": "median",
              "render_all_leaves_post_process": render_workload(a.reps, dev), "knn_points": knn_workload(a.reps, dev)}
    line = json.dumps(result, indent=1)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
