"""Instanced scenes on one GPU (RayMeshScene, rt_scene.cu): the scene against one RayMeshIntersector over the same
geometry flattened into one mesh, on the same rays; the time of update() (prepare + top-level build); and one scene
call against M separate single-mesh calls plus an eager merge of their closest hits.

Scenes: "icos20k_x1000" (1 000 instances of a 20 480-triangle icosphere on a 10^3 grid, random rotations and
non-uniform scales, 20.5 M triangles flattened) and "config2_x64" (64 instances of the 327 680-triangle config-2
icosphere on a 4^3 grid, 21.0 M flattened).  Rays: 1920x1080 pinhole rays from one origin outside the grid, and 4 M
random rays with origins inside the grid box.  Calls are timed with CUDA events after a warm-up, median of reps, L2
overwritten before every timed pass.  The card's name and power limit are read in the same run.

    python tools/scene_probe.py [--out profiles/scene_probe.json]
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
from triro import synth  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402
from triro.ray.scene import RayMeshScene  # noqa: E402


def grid_transforms(k: int, spacing: float, seed: int, smin=0.6, smax=1.2) -> torch.Tensor:
    """float32 [k^3,3,4]: random rotations times non-uniform scales, centred on a k^3 grid of the given spacing"""
    rng = np.random.default_rng(seed)
    n = k ** 3
    t = np.zeros((n, 3, 4), np.float64)
    g = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), -1).reshape(-1, 3) * spacing
    for i in range(n):
        q, r = np.linalg.qr(rng.normal(size=(3, 3)))
        q = q * np.sign(np.diag(r))
        t[i, :, :3] = q * rng.uniform(smin, smax, size=3)
        t[i, :, 3] = g[i] - 0.5 * (k - 1) * spacing
    return torch.from_numpy(t.astype(np.float32))


def flatten(v: torch.Tensor, f: torch.Tensor, t: torch.Tensor):
    """every instance's vertices transformed in float64 on the GPU, concatenated"""
    td = t.to(v.device, torch.float64)
    w = torch.einsum("nij,vj->nvi", td[:, :, :3], v.double()) + td[:, None, :, 3]
    faces = (f[None].long() + torch.arange(t.shape[0], device=v.device)[:, None, None] * v.shape[0]).reshape(-1, 3)
    return w.reshape(-1, 3).float(), faces.int()


def rays(kind: str, half: float, dev):
    if kind == "camera":
        o, d = synth.pinhole_rays(1920, 1080, device=dev, origin=(0.3 * half, 0.2 * half, 3.0 * half))
        return o, d
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    o = (torch.rand((4_000_000, 3), generator=g, device=dev) * 2 - 1) * half
    d = torch.randn((4_000_000, 3), generator=g, device=dev)
    return o, d / d.norm(dim=1, keepdim=True)


def merge_closest(calls, o, d):
    """closest of M dense closest-hit results by t = |loc - o| / |d| (eager torch): (hit, inst, tri, loc)"""
    t = torch.stack([torch.where(h, ((l - o).norm(dim=-1) / d.norm(dim=-1)), torch.inf) for h, _, _, l, _ in calls])
    best = t.argmin(0)
    hit = torch.stack([c[0] for c in calls]).gather(0, best[None])[0]
    tri = torch.stack([c[2] for c in calls]).gather(0, best[None])[0]
    loc = torch.stack([c[3] for c in calls]).gather(0, best[None, ..., None].expand(1, *calls[0][3].shape))[0]
    return hit, torch.where(hit, best.int(), -1), tri, loc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scene_probe.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scene_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "reps": a.reps,
           "timing": "CUDA events per call, median of reps, L2 overwritten before each", "scenes": [], "update": [],
           "separate_calls": []}
    med = lambda ms: float(np.median(ms))  # noqa: E731
    for name, sub, k, spacing in (("icos20k_x1000", 5, 10, 3.0), ("config2_x64", 7, 4, 3.0)):
        v, f = synth.icosphere(sub)
        vt, ft = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
        t = grid_transforms(k, spacing, seed=1)
        mesh = RayMeshIntersector(vertices=vt, faces=ft)
        scene = RayMeshScene([mesh], torch.zeros(t.shape[0], dtype=torch.int64), t)
        fv, ff = flatten(vt, ft, t)
        flat = RayMeshIntersector(vertices=fv, faces=ff)
        half = 0.5 * k * spacing
        for kind in ("camera", "random"):
            o, d = rays(kind, half, dev)
            n = o.reshape(-1, 3).shape[0]
            sh, _, si, st, sl, _ = scene.intersects_closest(o, d)
            fh, _, ftri, fl, _ = flat.intersects_closest(o, d)
            same_hit = float((sh == fh).float().mean())
            both = sh & fh
            same_tri = float(((si.long() * f.shape[0] + st.long()) == ftri.long())[both].float().mean())
            row = {"scene": name, "instances": t.shape[0], "mesh_tris": int(f.shape[0]), "flat_tris": int(ff.shape[0]),
                   "rays": kind, "n_rays": n, "hit_fraction": float(sh.float().mean()),
                   "agree_hit": same_hit, "agree_tri_where_both_hit": same_tri,
                   "max_loc_diff_where_both_hit": float((sl - fl).abs().max(dim=-1)[0][both].max()) if both.any() else 0.0}
            for mode in ("closest", "count"):
                fs = getattr(scene, "intersects_" + mode)
                ff_ = getattr(flat, "intersects_" + mode)
                ms_s = time_call(lambda: fs(o, d), a.reps, flush)
                ms_f = time_call(lambda: ff_(o, d), a.reps, flush)
                row[mode] = {"scene_ms": med(ms_s), "flat_ms": med(ms_f), "scene_mrays_s": n / med(ms_s) / 1e3,
                             "flat_mrays_s": n / med(ms_f) / 1e3}
            out["scenes"].append(row)
            print(json.dumps(row), flush=True)
        del flat, scene
        torch.cuda.empty_cache()
    # update(): prepare + top-level build (+ the header read the build makes), host clock around a synchronised call
    v, f = synth.icosphere(3)
    mesh = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    for n in (1_000, 10_000, 100_000):
        k = round(n ** (1 / 3))
        t = grid_transforms(k, 3.0, seed=2)
        t = torch.cat([t, t[: n - t.shape[0]]]) if t.shape[0] < n else t[:n]
        scene = RayMeshScene([mesh], torch.zeros(n, dtype=torch.int64), t)
        ms = []
        for _ in range(a.reps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            scene.update()
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
        row = {"instances": n, "update_ms": med(ms[1:]), "runs_ms": ms[1:]}
        out["update"].append(row)
        print(json.dumps(row), flush=True)
    # one scene call vs M single-mesh calls + merge (640x360 camera rays)
    o, d = synth.pinhole_rays(640, 360, device=dev, origin=(0.0, 0.0, 20.0))
    o = o.contiguous()
    for m in (10, 50):
        t = grid_transforms(4, 3.0, seed=3)[:m]
        scene = RayMeshScene([mesh], torch.zeros(m, dtype=torch.int64), t)
        sep = []
        for i in range(m):
            fv, ff = flatten(torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev), t[i:i + 1])
            sep.append(RayMeshIntersector(vertices=fv, faces=ff))
        ms_s = time_call(lambda: scene.intersects_closest(o, d), a.reps, flush)
        ms_m = time_call(lambda: merge_closest([r.intersects_closest(o, d) for r in sep], o, d), a.reps, flush)
        ms_c = time_call(lambda: [r.intersects_closest(o, d) for r in sep], a.reps, flush)
        sh, _, si, _, _, _ = scene.intersects_closest(o, d)
        mh, mi, _, _ = merge_closest([r.intersects_closest(o, d) for r in sep], o, d)
        row = {"meshes": m, "mesh_tris": int(f.shape[0]), "rays": "640x360 camera", "scene_ms": med(ms_s),
               "separate_calls_ms": med(ms_c), "separate_calls_plus_merge_ms": med(ms_m),
               "agree_hit": float((sh == mh).float().mean()), "agree_inst_where_both_hit": float((si == mi)[sh & mh].float().mean())}
        out["separate_calls"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
