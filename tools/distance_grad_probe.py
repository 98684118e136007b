"""Distance gradient on one GPU: the forward with and without grad tracking, the pseudo-normal forward that also
returns the closest points against the plain one, and the backward (rt_distance_grad) split into its per-point pass,
sort and reduction, next to a float32 index_add_ baseline written in eager torch.

Meshes: the config-2 icosphere (327 680 triangles), the config-4 soup (1 M) and the config-3 heightfield (4.19 M).
Point sets: (a) points jittered around the surface and (b) uniform in the 1.2x bbox (tools/closest_point_probe.py),
and (e) every point on one vertex: points 100 diagonals from the mesh centre in one direction, jittered by 1e-3 of
the diagonal, whose closest feature is one extreme vertex.  Calls are timed with CUDA events after a warm-up, median
of reps, L2 overwritten before every timed pass.  The split of the backward comes from a separate torch.profiler run
(CUDA kernel time summed per kernel family).  A sample of every set is compared bit for bit with the host simulator
(tests/distgrad/).

    python tools/distance_grad_probe.py [--out profiles/distance_grad_probe.json] [--points 10000000]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tools"),
          os.path.join(ROOT, "tests", "distgrad")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import distgrad as D  # noqa: E402
from closest_point_probe import card, point_sets, time_call  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

FAMILIES = {"points": ("k_dg_points",), "sort": ("k_histogram", "k_scan_hist", "k_onesweep_pass"),
            "reduce": ("k_dg_run_start", "k_dg_level0", "k_dg_level")}


def kernel_split(fn):
    """CUDA kernel time (ms) of one call of fn per kernel family, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in FAMILIES}
    out["other"] = 0.0
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if not us:
            continue
        fam = next((k for k, names in FAMILIES.items() if any(n in e.key for n in names)), "other")
        out[fam] += us / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "distance_grad_probe.json"))
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=200_000, help="points per set compared with the host simulator")
    ap.add_argument("--meshes", default="config2_icosphere,config4_soup,config3_heightfield")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("distance_grad_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    makers = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000),
              "config3_heightfield": lambda: synth.heightfield(2048, 1024)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "points": a.points, "reps": a.reps,
           "timing": "CUDA events per call, median of reps, L2 overwritten before each; split: torch.profiler kernel time",
           "rows": []}
    for mname in a.meshes.split(","):
        v, f = makers[mname]()
        rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
        acc, faces, nv = rmi.as_wrapper, rmi.mesh_faces, len(v)
        diag, sets = point_sets(v, a.points, 16, dev)
        g = torch.Generator(device=dev)
        g.manual_seed(7)
        centre = torch.tensor(0.5 * (v.min(0) + v.max(0)), device=dev, dtype=torch.float64)
        far = centre + torch.tensor([0.48, 0.6, 0.64], device=dev, dtype=torch.float64) * 100 * diag
        one = (far + torch.randn((a.points, 3), generator=g, device=dev, dtype=torch.float64) * 1e-3 * diag).float()
        for sname, pts in (("a_surface", sets["a_surface"][0]), ("b_uniform", sets["b_uniform"][0]), ("e_one_vertex", one)):
            n = pts.shape[0]
            row = dict(mesh=mname, tris=int(len(f)), verts=nv, points=sname, n=n)
            med = lambda fn: float(np.median(time_call(fn, a.reps, flush)))  # noqa: E731
            row["forward_ms"] = med(lambda: rmi.closest_point(pts))
            tracked = pts.clone().requires_grad_()
            row["forward_tracked_ms"] = med(lambda: rmi.closest_point(tracked))
            row["pseudonormal_ms"] = med(lambda: hops.signed_distance_pseudonormal(acc, pts))
            row["pseudonormal_closest_ms"] = med(lambda: hops.signed_distance_pseudonormal(acc, pts, return_closest=True))
            c, d, t, uv = hops.closest_point(acc, pts)
            go = torch.rand(n, generator=g, device=dev)
            row["backward_points_ms"] = med(lambda: hops.distance_grad(pts, go, d, c, t, uv, faces, nv, vertices_grad=False))
            row["backward_vertices_ms"] = med(lambda: hops.distance_grad(pts, go, d, c, t, uv, faces, nv, points_grad=False))
            row["backward_both_ms"] = med(lambda: hops.distance_grad(pts, go, d, c, t, uv, faces, nv))
            row["workspace_bytes"] = hops.distance_grad_workspace_bytes(n, nv)

            def eager():
                live = (t >= 0) & (d > 0) & torch.isfinite(d)
                q = torch.where(live[:, None], go[:, None] * (pts - c) / d[:, None], 0.0)
                w = torch.stack([uv[:, 0], uv[:, 1], 1 - uv[:, 0] - uv[:, 1]], 1)
                gv = torch.zeros((nv, 3), device=dev)
                gv.index_add_(0, faces[t.clamp_min(0).long()].long().reshape(-1), (-w[:, :, None] * q[:, None, :]).reshape(-1, 3))
                return q, gv

            row["eager_index_add_ms"] = med(eager)
            row["backward_split_ms"] = kernel_split(lambda: hops.distance_grad(pts, go, d, c, t, uv, faces, nv))
            gp, gv = hops.distance_grad(pts, go, d, c, t, uv, faces, nv)
            gp2, gv2 = hops.distance_grad(pts, go, d, c, t, uv, faces, nv)
            row["repeat_bit_exact"] = bool(torch.equal(gp.view(torch.int32), gp2.view(torch.int32))
                                           and torch.equal(gv.view(torch.int32), gv2.view(torch.int32)))
            _, ref = eager()
            row["max_abs_diff_vs_index_add"] = float((gv - ref).abs().max())
            row["distinct_vertices_hit"] = int(torch.unique(faces[t[t >= 0].long()]).numel())
            s = slice(0, a.parity)
            sp, sv = hops.distance_grad(pts[s], go[s], d[s], c[s], t[s], uv[s], faces, nv)
            hp, hv = D.sim_grad(pts[s].cpu().numpy(), go[s].cpu().numpy(), d[s].cpu().numpy(), c[s].cpu().numpy(),
                                t[s].cpu().numpy(), uv[s].cpu().numpy(), faces.cpu().numpy(), nv)
            row["parity_points"] = a.parity
            row["parity_hostsim_bit_exact"] = bool(np.array_equal(sp.cpu().numpy().view(np.uint32), hp.view(np.uint32))
                                                   and np.array_equal(sv.cpu().numpy().view(np.uint32), hv.view(np.uint32)))
            out["rows"].append(row)
            print(json.dumps({k: (round(x, 4) if isinstance(x, float) else x) for k, x in row.items()}), flush=True)
            del c, d, t, uv, go, gp, gv, gp2, gv2, ref, tracked
        del rmi, acc, sets, one
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
