"""Hit gradient on one GPU: the ray queries' forward with and without grad tracking, and the backward (rt_ray_grad)
with rays only and with vertices, split into its per-row pass, sort and reduction, next to an eager float32 torch
backward of the same formula that sums with index_add_.

Workloads: config 2 (icosphere subdivision 7, 327 680 triangles, 3840x2160 pinhole rays, closest hit) and config 4
(1 M-triangle soup, 10 M random rays, closest hit and all hits at max_hits 8).  The incoming gradient is that of a
depth loss, g_L = d, plus a random g_U for the closest hit.  Calls are timed with CUDA events after a warm-up, median
of reps, L2 overwritten before every timed pass; the split comes from a separate torch.profiler run.  The first 200 k
rows are compared bit for bit with the host simulator (tests/raygrad/).

    python tools/ray_grad_probe.py [--out profiles/ray_grad_probe.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tools"),
          os.path.join(ROOT, "tests", "raygrad")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import raygrad as R  # noqa: E402
from closest_point_probe import card, time_call  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

FAMILIES = {"rows": ("k_rg_rows",), "sort": ("k_histogram", "k_scan_hist", "k_onesweep_pass"),
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


def eager_backward(o, d, tri, ray_idx, gl, gu, verts, faces):
    """The formula of DESIGN.md §4.10 in eager float32 torch, vertex sums with index_add_ (not bit-exact).  Miss rows
    stay in as zero contributions to the vertices of triangle 0, as a masked eager backward would write them."""
    rows = ray_idx.long() if ray_idx is not None else torch.arange(tri.numel(), device=tri.device)
    live = tri >= 0
    fi = faces[tri.clamp_min(0).long()].long()
    v0, v1, v2 = verts[fi[:, 0]], verts[fi[:, 1]], verts[fi[:, 2]]
    ro, rd = o.reshape(-1, 3)[rows], d.reshape(-1, 3)[rows]
    e1, e2, s = v1 - v0, v2 - v0, ro - v0
    p = torch.cross(rd, e2, dim=1)
    det = (e1 * p).sum(1)
    r = torch.cross(s, e1, dim=1)
    b1, b2, t = (s * p).sum(1) / det, (rd * r).sum(1) / det, (e2 * r).sum(1) / det
    gb1 = (gl * e1).sum(1) + (0 if gu is None else gu[:, 1] - gu[:, 0])
    gb2 = (gl * e2).sum(1) - (0 if gu is None else gu[:, 0])
    lam = (gb1[:, None] * p + gb2[:, None] * torch.cross(e1, rd, dim=1)) / det[:, None]
    lam = torch.where(live[:, None], lam, 0.0)
    go = torch.zeros_like(o.reshape(-1, 3)).index_add_(0, rows, lam)
    gd = torch.zeros_like(o.reshape(-1, 3)).index_add_(0, rows, torch.where(live[:, None], t[:, None] * lam, 0.0))
    w = torch.where(live[:, None], torch.stack([1 - b1 - b2, b1, b2], 1), 0.0)
    gv = torch.zeros_like(verts).index_add_(0, fi.reshape(-1), (w[:, :, None] * (gl - lam)[:, None, :]).reshape(-1, 3))
    return go, gd, gv


def conditioning(o, d, tri, ray_idx, verts, faces):
    """per row |e1| |e2| |d| / |det| in binary64 (inf for a miss): how much the recomputed hit amplifies rounding"""
    rows = ray_idx.long() if ray_idx is not None else torch.arange(tri.numel(), device=tri.device)
    fi = faces[tri.clamp_min(0).long()].long()
    v = verts.double()
    e1, e2 = v[fi[:, 1]] - v[fi[:, 0]], v[fi[:, 2]] - v[fi[:, 0]]
    rd = d.reshape(-1, 3)[rows].double()
    det = (e1 * torch.cross(rd, e2, dim=1)).sum(1).abs()
    k = e1.norm(dim=1) * e2.norm(dim=1) * rd.norm(dim=1) / det
    return torch.where(tri >= 0, k, torch.inf)


def diffs(got, ref):
    """per output (grad_origins, grad_directions, grad_vertices): max |got - ref| and that over max |ref|"""
    out = []
    for x, y in zip(got, ref):
        x, y = x.reshape(-1, 3).double(), y.reshape(-1, 3).double()
        a = float((x - y).abs().max()) if x.numel() else 0.0
        m = float(y.abs().max()) if y.numel() else 0.0
        out.append({"max_abs": a, "max_abs_over_max_ref": a / m if m > 0 else 0.0})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ray_grad_probe.json"))
    ap.add_argument("--rays4", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=200_000, help="rows compared with the host simulator")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ray_grad_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "reps": a.reps,
           "timing": "CUDA events per call, median of reps, L2 overwritten before each; split: torch.profiler kernel time",
           "rows": []}
    med = lambda fn: float(np.median(time_call(fn, a.reps, flush)))  # noqa: E731
    work = []
    v, f = synth.icosphere(7)
    o, d = synth.pinhole_rays(3840, 2160, device=dev)
    work.append(("config2_icosphere", v, f, o.contiguous(), d, ("closest",)))
    v4, f4 = synth.triangle_soup(1_000_000)
    o4, d4 = synth.random_rays(a.rays4, seed=4, device=dev)
    work.append(("config4_soup", v4, f4, o4, d4, ("closest", "allhits")))
    for mname, v, f, o, d, modes in work:
        rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
        verts, faces, nv = rmi.mesh_vertices, rmi.mesh_faces, len(v)
        for mode in modes:
            row = dict(mesh=mname, tris=int(len(f)), verts=nv, mode=mode, rays=int(o.numel() // 3))
            ot, dt = o.clone().requires_grad_(), d.clone().requires_grad_()
            if mode == "closest":
                row["forward_ms"] = med(lambda: rmi.intersects_closest(o, d))
                row["forward_tracked_ms"] = med(lambda: rmi.intersects_closest(ot, dt))
                hit, _, tri, _, _ = hops.intersects_closest(rmi.as_wrapper, o, d)
                tri, ray_idx = tri.reshape(-1), None
                gl = d.reshape(-1, 3).contiguous()
                gu = torch.randn(tri.numel(), 2, device=dev)
            else:
                row["forward_ms"] = med(lambda: rmi.intersects_location(o, d))
                row["forward_tracked_ms"] = med(lambda: rmi.intersects_location(ot, dt))
                _, ray_idx, tri = hops.intersects_location(rmi.as_wrapper, o, d, rmi.max_hits)
                gl = d.reshape(-1, 3)[ray_idx.long()].contiguous()
                gu = None
            row["rows"] = int(tri.numel())
            row["hit_rows"] = int((tri >= 0).sum())

            def bwd(rays=True, vertices=True):
                return hops.ray_grad(o, d, tri, gl, gu, verts, faces, ray_idx=ray_idx, origins_grad=rays,
                                     directions_grad=rays, vertices_grad=vertices)

            row["backward_rays_ms"] = med(lambda: bwd(vertices=False))
            row["backward_vertices_ms"] = med(lambda: bwd(rays=False))
            row["backward_both_ms"] = med(bwd)
            row["workspace_bytes"] = hops.ray_grad_workspace_bytes(tri.numel(), nv)
            row["eager_index_add_ms"] = med(lambda: eager_backward(o, d, tri, ray_idx, gl, gu, verts, faces))
            row["backward_split_ms"] = kernel_split(bwd)
            g1, g2 = bwd(), bwd()
            row["repeat_bit_exact"] = all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(g1, g2))
            ref = eager_backward(o, d, tri, ray_idx, gl, gu, verts, faces)
            row["diff_vs_eager"] = diffs(g1, ref)
            # the same comparison on the well-conditioned rows only (|e1| |e2| |d| / |det| < 100, the others dropped)
            kappa = conditioning(o, d, tri, ray_idx, verts, faces)
            tri_wc = torch.where(kappa < 100, tri, -1)
            row["rows_kappa_lt_100"] = int((tri_wc >= 0).sum())
            row["max_kappa"] = float(kappa[tri >= 0].max()) if bool((tri >= 0).any()) else 0.0
            row["diff_vs_eager_kappa_lt_100"] = diffs(
                hops.ray_grad(o, d, tri_wc, gl, gu, verts, faces, ray_idx=ray_idx),
                eager_backward(o, d, tri_wc, ray_idx, gl, gu, verts, faces))
            del kappa, tri_wc
            # parity: the first rows (and their rays) against the host simulator
            s = slice(0, a.parity)
            ts = tri[s]
            if ray_idx is None:
                rs, os_, ds_ = None, o.reshape(-1, 3)[s], d.reshape(-1, 3)[s]
            else:
                n_r = int(ray_idx[s][-1]) + 1 if ts.numel() else 0
                rs, os_, ds_ = ray_idx[s], o.reshape(-1, 3)[:n_r], d.reshape(-1, 3)[:n_r]
            os_, ds_ = os_.contiguous(), ds_.contiguous()
            gp = hops.ray_grad(os_, ds_, ts, gl[s].contiguous(), None if gu is None else gu[s].contiguous(), verts, faces,
                               ray_idx=rs)
            hp = R.sim_grad(os_.cpu().numpy(), ds_.cpu().numpy(), ts.cpu().numpy(), gl[s].cpu().numpy(),
                            None if gu is None else gu[s].cpu().numpy(), v, f, None if rs is None else rs.cpu().numpy())
            row["parity_rows"] = int(ts.numel())
            row["parity_hostsim_bit_exact"] = all(np.array_equal(x.cpu().numpy().view(np.uint32), y.view(np.uint32))
                                                  for x, y in zip(gp, hp))
            out["rows"].append(row)
            print(json.dumps({k: (round(x, 4) if isinstance(x, float) else x) for k, x in row.items()}), flush=True)
            del g1, g2, ref, gp, tri, gl, gu, ray_idx, ot, dt
            torch.cuda.empty_cache()
        del rmi, verts, faces
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
