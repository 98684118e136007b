"""Closest-point query throughput on one GPU (rt_closest_point), with traversal counters and a parity verdict.

Meshes: the config-2 icosphere (327 680 triangles), the config-4 soup (1 M) and the config-3 heightfield (4.19 M).
Point sets: (a) 10 M points jittered around the surface (sigma = 1 % of the bbox diagonal), (b) 10 M points uniform in
the 1.2x bbox, (c) a 256^3 grid over the 1.2x bbox in row-major order (an SDF bake), (d) = (b) with max_distance =
2 % of the diagonal.  Each call is timed with CUDA events after a warm-up, with L2 overwritten before every timed pass
(the blob and the points would otherwise stay in the 126 MB L2 between passes).  A separate instrumented call gives
nodes and triangles per point; bytes per point = 80 per node + 48 per triangle + 12 in + 28 out, an upper bound of
what traversal touches (most of it is served from L2, not HBM).  A 1 M-point sample of every set is compared bit for
bit with the binary32 MIRROR oracle (tests/pointquery/), whose median-split BVH on all host cores is the CPU baseline.

    python tools/closest_point_probe.py [--out profiles/closest_point_probe.json] [--points 10000000] [--grid 256]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tests", "pointquery")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import pointquery as pq  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def point_sets(v, n, grid, dev):
    lo = torch.tensor(v.min(0), device=dev, dtype=torch.float64)
    hi = torch.tensor(v.max(0), device=dev, dtype=torch.float64)
    c, h = 0.5 * (lo + hi), 0.6 * (hi - lo)
    diag = float(torch.linalg.norm(hi - lo))
    g = torch.Generator(device=dev)
    g.manual_seed(2024)
    vt = torch.from_numpy(v).to(dev)
    idx = torch.randint(0, len(v), (n,), generator=g, device=dev)
    a = (vt[idx].double() + torch.randn((n, 3), generator=g, device=dev, dtype=torch.float64) * (0.01 * diag)).float()
    b = (c + (torch.rand((n, 3), generator=g, device=dev, dtype=torch.float64) * 2 - 1) * h).float()
    axes = [torch.linspace(float(c[k] - h[k]), float(c[k] + h[k]), grid, device=dev, dtype=torch.float64) for k in range(3)]
    gr = torch.stack(torch.meshgrid(*axes, indexing="ij"), dim=-1).reshape(-1, 3).float()
    return diag, {"a_surface": (a, float("inf")), "b_uniform": (b, float("inf")), "c_grid": (gr, float("inf")),
                  "d_uniform_maxdist": (b, 0.02 * diag)}


def time_call(fn, reps, flush):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        flush.add_(1)                       # overwrite L2 between timed passes
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "closest_point_probe.json"))
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=1_000_000, help="points per set compared with the MIRROR oracle")
    ap.add_argument("--meshes", default="config2_icosphere,config4_soup,config3_heightfield")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("closest_point_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    makers = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000),
              "config3_heightfield": lambda: synth.heightfield(2048, 1024)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "host_threads": pq.num_threads(), "points": a.points,
           "grid": a.grid, "reps": a.reps, "timing": "CUDA events per call, median of reps, L2 overwritten before each",
           "rows": []}
    for mname in a.meshes.split(","):
        v, f = makers[mname]()
        rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
        acc = rmi.as_wrapper
        t0 = time.time()
        om = pq.PointMesh(v, f, use_bvh=True)
        oracle_build_s = time.time() - t0
        diag, sets = point_sets(v, a.points, a.grid, dev)
        for sname, (pts, md) in sets.items():
            n = pts.shape[0]
            ms = time_call(lambda: hops.closest_point(acc, pts, md), a.reps, flush)
            cnt = torch.zeros(4, dtype=torch.int64, device=dev)
            res = hops.closest_point(acc, pts, md, counters=cnt)
            nodes, tris, npts, found = cnt.tolist()
            med = float(np.median(ms))
            # parity on a sample: random points are i.i.d., so the first ones are a sample; the grid is strided
            step = max(1, n // a.parity) if sname == "c_grid" else 1
            sl = slice(0, a.parity * step, step)
            sample = pts[sl].cpu().numpy()
            t0 = time.time()
            ref = pq.query(om, sample, pq.MIRROR, md)
            cpu_s = time.time() - t0
            got = [x[sl].cpu().numpy() for x in res]
            same = (np.array_equal(got[2], ref["tri"]) and all(np.array_equal(g.view(np.uint32), ref[k].view(np.uint32))
                                                               for g, k in ((got[0], "closest"), (got[1], "distance"), (got[3], "uv"))))
            row = dict(mesh=mname, tris=int(len(f)), points=sname, n=n, max_distance=md, ms_median=med, ms_all=ms,
                       mpts_s=n / med / 1e3, nodes_per_pt=nodes / npts, tris_per_pt=tris / npts, found_frac=found / npts,
                       bytes_per_pt=(80 * nodes + 48 * tris) / npts + 12 + 28,
                       parity_points=len(sample), parity_mirror_bit_exact=bool(same),
                       cpu_oracle_mpts_s=len(sample) / cpu_s / 1e6, cpu_oracle_bvh_build_s=oracle_build_s)
            out["rows"].append(row)
            print(json.dumps({k: (round(x, 4) if isinstance(x, float) else x) for k, x in row.items() if k != "ms_all"}), flush=True)
            del res
        del rmi, acc, om, sets
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
