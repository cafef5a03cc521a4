"""bench.py contract checks that need no GPU: the reference arm (CPU restatement of the reference path)
prints ONE JSON line with the keys the driver reads, and the algorithmic-byte model of DESIGN.md section 4."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")      # what torchrun exports; the arm must still use every thread
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                        "plumbing_10k_256", "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                       env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("fwd+bwd frames/sec") and d["value"] > 0 and d["steps"] == 2
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "oracle" in cb["sample"]
    assert d["config"]["workload"] == "plumbing_10k_256" and d["config"]["image"] == [256, 256]
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    assert cb["cores"] == avail                       # OMP_NUM_THREADS=1 was overridden


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_sample_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: float32 files of the kept step's outputs and gradients, the same seeded sample of pixels and
    Gaussians on every call, everything when it fits, and never more than DUMP_BYTES."""
    import types
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    P, H, W, V = 5000, 40, 60, 3
    g = torch.Generator().manual_seed(0)
    params = {k: torch.zeros(P, *s) for k, s in (("means3D", (3,)), ("opacities", (1,)), ("shs", (16, 3)),
                                                  ("scales", (3,)), ("rotations", (4,)))}
    for t in params.values():
        t.grad = torch.randn(t.shape, generator=g)
    means2D = torch.zeros(P, 3)
    means2D.grad = torch.randn(P, 3, generator=g)

    def out(*shape):            # what the rasterizer returns: a non-leaf tensor attached to the autograd graph
        return torch.randn(*shape, generator=g).requires_grad_(True) * 1.0

    kept = [(out(3, H, W), None, out(1, H, W), out(1, H, W), torch.randint(0, 9, (P,), generator=g, dtype=torch.int32))
            for _ in range(V)]
    wl = types.SimpleNamespace(cx=types.SimpleNamespace(torch=torch, dev=torch.device("cpu")), kept=kept, params=params,
                               means2D=means2D, extra=None, P=P, H=H, W=W)

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}

    bench.dump_outputs(wl, str(tmp_path / "all"))
    full = load(tmp_path / "all")
    assert sorted(full) == ["alpha", "color", "depth", "grad_means2D", "grad_means3D", "grad_opacities", "grad_rotations",
                            "grad_scales", "grad_shs", "radii"]
    assert all(a.dtype == np.float32 for a in full.values())
    assert np.array_equal(full["color"], torch.stack([k[0] for k in kept]).flatten(2).detach().numpy())
    assert np.array_equal(full["radii"], torch.stack([k[4] for k in kept]).float().numpy())
    assert np.array_equal(full["grad_shs"], params["shs"].grad.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    for d in ("a", "b"):
        bench.dump_outputs(wl, str(tmp_path / d))
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(x.nbytes for x in a.values()) <= 200_000
    assert a["color"].shape[:2] == (V, 3) and 0 < a["color"].shape[2] < H * W
    assert a["grad_shs"].shape[1:] == (16, 3) and 0 < a["grad_shs"].shape[0] < P
    assert np.isin(a["grad_shs"].reshape(-1), full["grad_shs"].reshape(-1)).all()


def test_algorithmic_bytes_worked_example():
    """SURVEY.md section 8d's worked example: P = P_vis = 1 M, N = 8 M, 1080p, C = 3, degree 3, 45 key bits."""
    sys.path.insert(0, ROOT)
    import bench
    d = bench.algorithmic_bytes(1_000_000, 1_000_000, 8_000_000, 1080, 1920, 3, 3, 13)
    assert d["preprocess_fwd"] == 1_000_000 * (236 + 48)
    assert d["blend_fwd"] == 8_000_000 * 48 + 1920 * 1080 * (4 * 5 + 8)
    assert d["tile_sort"] == 8_000_000 * 12 * 2
    total = sum(d.values())
    assert 1.5e9 < total < 3.2e9                      # the survey's 3.0 GB uses 6 passes of a 64-bit sort


def test_bench_helpers_and_flat_layout():
    """Pure-host pieces of the bench and of the multi-GPU plumbing: the median, the issue roofline arithmetic, the
    rank-invariant gradient layout and the fixed-point bit budget of the exact centroid sums."""
    sys.path.insert(0, ROOT)
    import torch
    import bench
    from opengaussian_b200 import dist as ogd
    from opengaussian_b200.kmeans_quantize import fixed_point_bits
    assert bench.median([3.0, 1.0, 2.0]) == 2.0 and bench.median([4.0, 1.0, 2.0, 3.0]) == 2.5
    stats = {"interactions_to_last_contributor": 3_200_000, "interactions_listed": 9_000_000}
    traffic = {"blend_bwd": {"warp_insts_per_frame": 3.2e6}, "blend_fwd": {"warp_insts_per_frame": 1.6e6}}
    iss = bench.issue_roofline(stats, {"blend_bwd": 0.5, "blend_fwd": 0.25}, traffic, 2000)
    assert abs(iss["blend_bwd"]["warp_insts_per_32_interactions"] - 32.0) < 1e-9
    assert abs(iss["blend_bwd"]["issue_frac_of_peak"] - 3.2e6 / 0.5e-3 / (148 * 4 * 2000e6)) < 1e-12
    assert abs(iss["blend_fwd"]["fp32_floor_ms"] * 3 - iss["blend_bwd"]["fp32_floor_ms"]) < 1e-12
    # gradient layout: a function of the shapes only, 64-float aligned slices, span ends with the last tensor
    ps = [torch.zeros(10, 3), torch.zeros(7), torch.zeros(5, 16, 3)]
    offs, span = ogd._flat_layout(ps)
    assert offs == [0, 64, 128] and span == 128 + 240
    # fixed-point budget: |x| * 2^bits < 2^31 and N * |x| * 2^bits < 2^62
    assert fixed_point_bits(5_000_000, 0.999) == 30
    assert fixed_point_bits(5_000_000, 1.0) == 30 and fixed_point_bits(5_000_000, 2.5) == 29
    assert fixed_point_bits(2 ** 31, 1000.0) == 20
    for n, m in ((10, 1e-3), (5_000_000, 7.3), (2 ** 33, 100.0)):
        b = fixed_point_bits(n, m)
        assert m * 2.0 ** b < 2.0 ** 31 and n * m * 2.0 ** b < 2.0 ** 62
