"""Gradients of instanced-scene queries on one GPU (rt_distgrad.cu through RayMeshScene's autograd, DESIGN.md
§4.13): backward against forward time, and one pose-optimisation step against what a user does without the feature.

- Ray rows: the scenes of BASELINE §11, "icos20k_x1000" (1 000 instances of a 20 480-triangle icosphere, random
  rotations and non-uniform scales 0.6-1.2) and "config2_x64" (64 instances of the 327 680-triangle icosphere), with
  1920 x 1080 camera rays.  Forward = intersects_closest (grad mode off); backward of sum(loc * g) with the rays only,
  rays + transforms, rays + transforms + member vertices requiring grad.
- Point rows: "icos20k_x1000_rigid" (unit scales) with 1 M near-surface points; forward = closest_point; backward of
  sum(distance * g) with the points only, + transforms, + member vertices.
- One optimisation step on icos20k_x1000 with the camera rays and a loss on loc, transforms requiring grad:
  scene.update + forward + backward, against flattening in torch (A v + b over every instance) + RayMeshIntersector
  build + forward + backward with the vertex gradient + torch's chain to the transforms.

Backward passes are timed with CUDA events around torch.autograd.backward after a fresh forward; steps with a host
clock around work that ends in a synchronise.  Median of reps after one warm-up, L2 overwritten before each timed
pass.  The card's name and power limit are read in the same run.

    python tools/scene_grad_probe.py [--out profiles/scene_grad_probe.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from closest_point_probe import card, time_call  # noqa: E402
from scene_point_probe import points  # noqa: E402
from scene_probe import grid_transforms, rays  # noqa: E402
from triro import synth  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402
from triro.ray.scene import RayMeshScene  # noqa: E402


def backward_ms(forward, reps, flush):
    """median ms of torch.autograd.backward of forward()'s loss, a fresh forward before each timed pass"""
    ms = []
    for k in range(reps + 1):
        loss = forward()
        torch.cuda.synchronize()
        flush.add_(1)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); loss.backward(); e1.record()
        torch.cuda.synchronize()
        if k:
            ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def step_ms(step, reps, flush):
    ms = []
    for k in range(reps + 1):
        flush.add_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step()
        torch.cuda.synchronize()
        if k:
            ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scene_grad_probe.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--points", type=int, default=1_000_000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scene_grad_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "reps": a.reps, "rays": [], "points": [], "step": []}
    cases = {"icos20k_x1000": (5, 10, 0.6, 1.2), "config2_x64": (7, 4, 0.6, 1.2), "icos20k_x1000_rigid": (5, 10, 1.0, 1.0)}
    for name, (sub, k, smin, smax) in cases.items():
        v, f = synth.icosphere(sub)
        t = grid_transforms(k, 3.0, seed=1, smin=smin, smax=smax).to(dev)
        verts = torch.from_numpy(v).to(dev)
        mesh = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f).to(dev))
        scene = RayMeshScene([mesh], torch.zeros(t.shape[0], dtype=torch.int64), t)
        half = 0.5 * k * 3.0
        g = torch.Generator(device=dev)
        g.manual_seed(3)
        if not name.endswith("rigid"):
            o, d = rays("camera", half, dev)
            o, d = o.reshape(-1, 3).contiguous(), d.reshape(-1, 3).contiguous()
            gl = torch.randn(o.shape, generator=g, device=dev)
            with torch.no_grad():
                fwd = float(np.median(time_call(lambda: scene.intersects_closest(o, d), a.reps, flush)))
                hit = scene.intersects_closest(o, d)[0]
            row = {"scene": name, "instances": t.shape[0], "mesh_tris": int(f.shape[0]), "rays": o.shape[0],
                   "hit_fraction": float(hit.float().mean()), "forward_ms": fwd}
            for what in ("rays", "rays+transforms", "rays+transforms+vertices"):
                tt = t.clone().requires_grad_("transforms" in what)
                scene.update(tt)
                mesh.mesh_vertices.requires_grad_("vertices" in what)
                oo, dd = o.clone().requires_grad_(), d.clone().requires_grad_()
                row[what + "_backward_ms"] = backward_ms(
                    lambda: (scene.intersects_closest(oo, dd)[4] * gl).sum(), a.reps, flush)
                mesh.mesh_vertices.requires_grad_(False)
            out["rays"].append(row)
            print(json.dumps(row), flush=True)
            scene.update(t)
        if name.endswith("rigid"):
            fv = torch.einsum("nij,vj->nvi", t[:, :, :3], verts) + t[:, None, :, 3]
            ff = (torch.from_numpy(f).to(dev)[None].long() + torch.arange(t.shape[0], device=dev)[:, None, None]
                  * verts.shape[0]).reshape(-1, 3)
            p = points("near_surface", half, fv.reshape(-1, 3), ff, 3.0, a.points, dev)
            gp = torch.randn(p.shape[0], generator=g, device=dev)
            with torch.no_grad():
                fwd = float(np.median(time_call(lambda: scene.closest_point(p), max(1, a.reps // 2), flush)))
            row = {"scene": name, "instances": t.shape[0], "mesh_tris": int(f.shape[0]), "points": p.shape[0],
                   "forward_ms": fwd}
            for what in ("points", "points+transforms", "points+transforms+vertices"):
                tt = t.clone().requires_grad_("transforms" in what)
                scene.update(tt)
                mesh.mesh_vertices.requires_grad_("vertices" in what)
                pp = p.clone().requires_grad_()
                row[what + "_backward_ms"] = backward_ms(lambda: (scene.closest_point(pp)[1] * gp).sum(),
                                                         max(1, a.reps // 2), flush)
                mesh.mesh_vertices.requires_grad_(False)
            out["points"].append(row)
            print(json.dumps(row), flush=True)
        if name == "icos20k_x1000":
            tt = t.clone().requires_grad_()
            faces = (torch.from_numpy(f).to(dev)[None].long() + torch.arange(t.shape[0], device=dev)[:, None, None]
                     * verts.shape[0]).reshape(-1, 3).int()

            def scene_step():
                scene.update(tt)
                (scene.intersects_closest(o, d)[4] * gl).sum().backward()

            def flat_step():
                w = (torch.einsum("nij,vj->nvi", tt[:, :, :3], verts) + tt[:, None, :, 3]).reshape(-1, 3)
                flat = RayMeshIntersector(vertices=w, faces=faces)
                (flat.intersects_closest(o, d)[3] * gl).sum().backward()

            row = {"scene": name, "rays": o.shape[0], "flat_tris": int(faces.shape[0]),
                   "scene_step_ms": step_ms(scene_step, a.reps, flush), "flatten_step_ms": step_ms(flat_step, a.reps, flush)}
            out["step"].append(row)
            print(json.dumps(row), flush=True)
        del scene, mesh
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
