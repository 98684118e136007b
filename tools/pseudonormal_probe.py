"""Pseudo-normal signed distance on one GPU: the precompute (rt_pseudonormals) and the throughput of
signed_distance in all three sign modes, on the closest-point probe's meshes and point sets.

Meshes: the config-2 icosphere (327 680 triangles, closed), the config-4 soup (1 M, open) and the config-3
heightfield (4.19 M, open).  Point sets (tools/closest_point_probe.py): (a) points jittered around the surface, (b)
uniform in the 1.2x bbox, (c) a row-major grid over it.  Each call is timed with CUDA events after a warm-up, median of
reps, L2 overwritten before every timed pass.  sign="contains" includes its host sync and retry launch, sign="winding"
its second walk; both include the closest-point walk.  The precompute is timed with the cache dropped before every
pass.  A sample of every set is compared bit for bit with the host simulator (tests/pseudonormal/), the normals and
edge counts in full; the fraction of points on which the three modes agree in sign is reported.

    python tools/pseudonormal_probe.py [--out profiles/pseudonormal_probe.json] [--points 10000000] [--grid 256]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tools"),
          os.path.join(ROOT, "tests", "pseudonormal")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import pseudonormal as P  # noqa: E402
from closest_point_probe import card, point_sets, time_call  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pseudonormal_probe.json"))
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=100_000, help="points per set compared with the host simulator")
    ap.add_argument("--meshes", default="config2_icosphere,config4_soup,config3_heightfield")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pseudonormal_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    makers = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000),
              "config3_heightfield": lambda: synth.heightfield(2048, 1024)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "points": a.points, "grid": a.grid, "reps": a.reps,
           "timing": "CUDA events per call, median of reps, L2 overwritten before each", "meshes": [], "rows": []}
    for mname in a.meshes.split(","):
        v, f = makers[mname]()
        rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
        acc = rmi.as_wrapper

        def precompute():
            acc._inner.pseudo_normals = None
            hops.pseudo_normals(acc)

        pre_ms = time_call(precompute, a.reps, flush)
        normals, counts = hops.pseudo_normals(acc)
        blob = acc.blob.cpu().numpy()
        rows, hcounts = P.sim_normals(blob)
        normals_exact = bool(np.array_equal(normals.cpu().numpy().view(np.uint32), rows.view(np.uint32)))
        m = dict(mesh=mname, tris=int(len(f)), precompute_ms_median=float(np.median(pre_ms)), precompute_ms_all=pre_ms,
                 edge_counts=counts.tolist(), normals_bytes=int(normals.numel() * 4),
                 normals_and_counts_match_hostsim=normals_exact and tuple(counts.tolist()) == hcounts)
        out["meshes"].append(m)
        print(json.dumps({k: x for k, x in m.items() if k != "precompute_ms_all"}), flush=True)
        _, sets = point_sets(v, a.points, a.grid, dev)
        for sname, (pts, _) in sets.items():
            if sname == "d_uniform_maxdist":
                continue
            n = pts.shape[0]
            row = dict(mesh=mname, tris=int(len(f)), points=sname, n=n)
            res = {}
            for mode in ("pseudonormal", "winding", "contains"):
                ms = time_call(lambda: rmi.signed_distance(pts, sign=mode), a.reps, flush)
                med = float(np.median(ms))
                row[f"{mode}_ms_median"] = med
                row[f"{mode}_mpts_s"] = n / med / 1e3
                res[mode] = rmi.signed_distance(pts, sign=mode)
            ms = time_call(lambda: hops.closest_point(acc, pts), a.reps, flush)
            row["closest_point_ms_median"] = float(np.median(ms))
            row["closest_point_mpts_s"] = n / float(np.median(ms)) / 1e3
            pos = {k: r > 0 for k, r in res.items()}
            row["sign_agree_pn_winding"] = float((pos["pseudonormal"] == pos["winding"]).float().mean())
            row["sign_agree_pn_contains"] = float((pos["pseudonormal"] == pos["contains"]).float().mean())
            step = max(1, n // a.parity) if sname == "c_grid" else 1
            sl = slice(0, a.parity * step, step)
            sample = pts[sl].cpu().numpy()
            sim = P.sim_signed_distance(blob, sample, rows)["sd"]
            row["parity_points"] = len(sample)
            row["parity_hostsim_bit_exact"] = bool(np.array_equal(res["pseudonormal"][sl].cpu().numpy().view(np.uint32),
                                                                  sim.view(np.uint32)))
            out["rows"].append(row)
            print(json.dumps({k: (round(x, 4) if isinstance(x, float) else x) for k, x in row.items()}), flush=True)
            del res, pos
        del rmi, acc, sets, normals, counts
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
