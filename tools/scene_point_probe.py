"""Point queries on instanced scenes on one GPU (RayMeshScene.closest_point / signed_distance, rt_scene_point.cu):
the scene against one RayMeshIntersector over the same geometry flattened with the kernels' binary32 world vertices
(affine_row, DESIGN.md §4.12), on the same points, with the bit-exact agreement of closest_point reported; the
preparation time of the side array and of the members' pseudo-normals; and one scene call against M separate
single-mesh calls plus an eager merge of their closest points.

Scenes: those of BASELINE §11, "icos20k_x1000" (1 000 instances of a 20 480-triangle icosphere on a 10^3 grid, random
rotations and non-uniform scales 0.6-1.2, about half of them mirrored, 20.5 M triangles flattened) and "config2_x64"
(64 instances of the 327 680-triangle config-2 icosphere on a 4^3 grid, 21.0 M flattened), plus "icos20k_x1000_rigid",
the first with unit scales (rotations and mirrors only), where the instance walk's singular-value bound is tight.
Points: 4 M uniform in the grid box and 4 M near the surface (on random flattened triangles plus N(0, (1e-3
spacing)^2) offsets).  Calls are timed with CUDA events after a warm-up (the agreement call), median of reps (fewer
for the slow scene calls), L2 overwritten before every timed pass.  The card's name and power limit are read in the
same run.  The flattened mesh keeps each instance's face order, so a mirrored instance is inside-out there: the sign
agreement compares the scene's sign with the flattened sign flipped on the points whose closest instance is mirrored.

    python tools/scene_point_probe.py [--out profiles/scene_point_probe.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tools"),
          os.path.join(ROOT, "tests", "scene")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import scenepoint as sp  # noqa: E402  (tests/scene: the binary32 affine_row flattening)
from closest_point_probe import card, time_call  # noqa: E402
from scene_probe import grid_transforms  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402
from triro.ray.scene import RayMeshScene  # noqa: E402


def points(kind: str, half: float, fv: torch.Tensor, ff: torch.Tensor, spacing: float, n: int, dev):
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    if kind == "uniform":
        return (torch.rand((n, 3), generator=g, device=dev) * 2 - 1) * half
    t = torch.randint(0, ff.shape[0], (n,), generator=g, device=dev)
    w = -torch.log(torch.rand((n, 3), generator=g, device=dev))
    w = w / w.sum(1, keepdim=True)
    tri = fv[ff[t].long()]
    p = (w[:, :, None] * tri).sum(1)
    return p + torch.randn((n, 3), generator=g, device=dev) * (1e-3 * spacing)


def timed(fn, reps, flush):
    """time_call without its own warm-up call"""
    ms = []
    for _ in range(reps):
        flush.add_(1)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def bits_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return bool(torch.equal(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scene_point_probe.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scene-reps", type=int, default=1)
    ap.add_argument("--points", type=int, default=4_000_000)
    ap.add_argument("--only", default="", help="comma-separated scene names and/or 'separate' (default: everything)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scene_point_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "reps": a.reps, "scene_reps": a.scene_reps, "points": a.points,
           "timing": "CUDA events per call, median of reps (scene calls: scene_reps after the agreement calls), L2 "
                     "overwritten before each", "scenes": [], "prepare": [],
           "separate_calls": []}
    med = lambda ms: float(np.median(ms))  # noqa: E731
    only = set(x for x in a.only.split(",") if x)
    for name, sub, k, spacing, smin, smax in (("icos20k_x1000", 5, 10, 3.0, 0.6, 1.2),
                                              ("icos20k_x1000_rigid", 5, 10, 3.0, 1.0, 1.0),
                                              ("config2_x64", 7, 4, 3.0, 0.6, 1.2)):
        if only and name not in only:
            continue
        v, f = synth.icosphere(sub)
        t = grid_transforms(k, spacing, seed=1, smin=smin, smax=smax)
        mirrored = torch.from_numpy(np.linalg.det(t[:, :, :3].double().numpy()) < 0).to(dev)
        mesh = RayMeshIntersector(vertices=torch.from_numpy(v).to(dev), faces=torch.from_numpy(f).to(dev))
        scene = RayMeshScene([mesh], torch.zeros(t.shape[0], dtype=torch.int64), t)
        fvn, ffn, _, _ = sp.flatten_affine([(v, f)], np.zeros(t.shape[0], np.int64), t.numpy())
        fv, ff = torch.from_numpy(fvn).to(dev), torch.from_numpy(ffn).to(dev)
        flat = RayMeshIntersector(vertices=fv, faces=ff)
        # preparation: the side array, then the member's pseudo-normals (dropped from its cache first)
        scene._point_state(True)
        prep = {"scene": name, "instances": t.shape[0]}
        for what in ("side", "normals"):
            ms = []
            for _ in range(a.reps + 1):
                scene._point_side = None
                scene._normals = None
                if what == "normals":
                    scene._point_state(False)
                    mesh.as_wrapper._inner.pseudo_normals = None
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                scene._point_state(what == "normals")
                torch.cuda.synchronize()
                ms.append((time.perf_counter() - t0) * 1e3)
            prep[what + "_ms"] = med(ms[1:])
        out["prepare"].append(prep)
        print(json.dumps(prep), flush=True)
        half = 0.5 * k * spacing
        for kind in ("uniform", "near_surface"):
            p = points(kind, half, fv, ff, spacing, a.points, dev)
            sc_, sd_, si, st, su = scene.closest_point(p, return_uv=True)
            fc, fd, ft, fu = flat.closest_point(p, return_uv=True)
            face = torch.where(si >= 0, si.long() * f.shape[0] + st.long(), -1).int()
            exact = bits_equal(sc_, fc) and bits_equal(sd_, fd) and bits_equal(face, ft) and bits_equal(su, fu)
            ssd = scene.signed_distance(p)
            fsd = flat.signed_distance(p, sign="pseudonormal")
            flip = mirrored[si.long().clamp(min=0)] & (si >= 0)
            row = {"scene": name, "instances": t.shape[0], "mirrored": int(mirrored.sum()), "mesh_tris": int(f.shape[0]),
                   "flat_tris": int(ff.shape[0]), "points": kind, "n_points": a.points,
                   "closest_point_bit_exact_vs_flat": exact,
                   "signed_distance_sign_agreement_vs_flat": float(((ssd > 0) == ((fsd > 0) ^ flip)).float().mean()),
                   "signed_distance_abs_bit_exact_vs_flat": bits_equal(ssd.abs(), fsd.abs()),
                   "inside_fraction": float((ssd > 0).float().mean())}
            calls = {"closest_point": (lambda: scene.closest_point(p), lambda: flat.closest_point(p)),
                     "signed_distance": (lambda: scene.signed_distance(p),
                                         lambda: flat.signed_distance(p, sign="pseudonormal"))}
            for q, (fs, ffl) in calls.items():
                ms_s = timed(fs, a.scene_reps, flush)     # warmed up by the agreement calls above
                ms_f = time_call(ffl, a.reps, flush)
                row[q] = {"scene_ms": med(ms_s), "flat_ms": med(ms_f), "scene_mpoints_s": a.points / med(ms_s) / 1e3,
                          "flat_mpoints_s": a.points / med(ms_f) / 1e3}
            out["scenes"].append(row)
            print(json.dumps(row), flush=True)
        del flat, scene, fv, ff
        torch.cuda.empty_cache()
    # one scene call vs M single-mesh calls + an eager merge (argmin of the distances), 1 M uniform points
    v, f = synth.icosphere(3)
    mesh = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    for m in ((10, 50) if not only or "separate" in only else ()):
        t = grid_transforms(4, 3.0, seed=3)[:m]
        scene = RayMeshScene([mesh], torch.zeros(m, dtype=torch.int64), t)
        sep = []
        for i in range(m):
            fvn, ffn, _, _ = sp.flatten_affine([(v, f)], np.zeros(1, np.int64), t[i:i + 1].numpy())
            sep.append(RayMeshIntersector(vertices=torch.from_numpy(fvn).to(dev), faces=torch.from_numpy(ffn).to(dev)))
        p = (torch.rand((1_000_000, 3), device=dev) * 2 - 1) * 6.0

        def merged():
            res = [r.closest_point(p) for r in sep]
            d = torch.stack([r[1] for r in res])
            best = d.argmin(0)
            return d.gather(0, best[None])[0], best.int()

        ms_s = time_call(lambda: scene.closest_point(p), a.reps, flush)
        ms_m = time_call(merged, a.reps, flush)
        _, sd_, si, _ = scene.closest_point(p)
        md_, mi = merged()
        row = {"meshes": m, "mesh_tris": int(f.shape[0]), "points": "1 M uniform", "scene_ms": med(ms_s),
               "separate_calls_plus_merge_ms": med(ms_m), "distance_bit_exact": bits_equal(sd_, md_),
               "agree_inst": float((si == mi).float().mean())}
        out["separate_calls"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
