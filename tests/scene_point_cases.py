"""Query points and sign-test scenes shared by the scene point-query tests (test infrastructure)."""
from __future__ import annotations

import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pseudonormal"))
import pseudonormal as pn  # noqa: E402
from triro import synth  # noqa: E402


def scene_box(flat_vertices) -> tuple[np.ndarray, np.ndarray]:
    v = np.asarray(flat_vertices, np.float64)
    return v.min(0), v.max(0)


def uniform_points(lo, hi, n: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)


def surface_points(flat_v, flat_f, n: int, seed: int = 1, offset: float = 1e-3) -> np.ndarray:
    """points on world triangles (random barycentrics), on their vertices and edge midpoints, plus small offsets"""
    rng = np.random.default_rng(seed)
    v = np.asarray(flat_v, np.float64)
    f = np.asarray(flat_f)
    t = f[rng.integers(0, len(f), size=n)]
    w = rng.dirichlet([1.0, 1.0, 1.0], size=n)
    kind = rng.integers(0, 3, size=n)                  # 0 face, 1 vertex, 2 edge midpoint
    w[kind == 1] = np.eye(3)[rng.integers(0, 3, size=int((kind == 1).sum()))]
    w[kind == 2] = np.array([0.5, 0.5, 0.0])
    p = np.einsum("nk,nkd->nd", w, v[t])
    scale = float(np.abs(v).max()) if len(v) else 1.0
    off = rng.normal(size=(n, 3)) * offset * scale * (rng.uniform(size=(n, 1)) < 0.5)
    return (p + off).astype(np.float32)


def special_points(lo, hi) -> np.ndarray:
    """far points (10^3 times the scene size), NaN and +-inf"""
    c = (np.asarray(lo) + np.asarray(hi)) / 2
    size = float(np.max(np.asarray(hi) - np.asarray(lo)))
    far = c + 1e3 * size * np.array([[1, 0, 0], [0, -1, 0], [0.3, 0.5, -0.8], [-1, -1, -1]])
    bad = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [np.nan, np.nan, np.nan]])
    return np.concatenate([far, bad]).astype(np.float32)


def rotation(rng) -> np.ndarray:
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q


def sign_scene(seed: int = 0):
    """(meshes, inst_mesh, transforms [I,3,4]): closed meshes (torus, star prism, notched cube, icosphere) as disjoint
    instances under rotations, uniform scales from 1e-3 to 1e3 and mirrors.  The instances of scale s lie along their
    own direction from the origin at 5 s to 20 s, so that every instance is resolved by binary32 and none overlap."""
    ms = [pn.torus(), pn.star_prism(), pn.notched_cube(), synth.icosphere(3)]
    rng = np.random.default_rng(seed)
    scales = [1e-3, 1e-2, 0.1, 1.0, 7.0, 1e2, 1e3, 0.5]
    dirs = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [1, 1, 1], [-1, -1, 1]], float)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    inst_mesh, ts = [], []
    k = 0
    for g, s in enumerate(scales):
        for m in range(len(ms)):
            a = rotation(rng) * s
            if k % 3 == 1:
                a[:, int(rng.integers(3))] *= -1.0          # mirrored
            v = np.asarray(ms[m][0], np.float64)
            centre = (v.min(0) + v.max(0)) / 2
            b = dirs[g] * s * 5.0 * (m + 1) - a @ centre
            t = np.zeros((3, 4))
            t[:, :3], t[:, 3] = a, b
            inst_mesh.append(m); ts.append(t)
            k += 1
    return ms, np.asarray(inst_mesh, np.int32), np.asarray(ts, np.float32)


def outward_faces(faces, face_inst, transforms) -> np.ndarray:
    """flattened faces with the corners of mirrored instances reversed, so that every instance faces outward in
    world space (the orientation the binary64 winding-number truth needs)"""
    mirrored = np.linalg.det(np.asarray(transforms, np.float64)[:, :, :3]) < 0
    f = np.array(faces)
    flip = mirrored[face_inst]
    f[flip] = f[flip][:, ::-1]
    return f


def sign_points(meshes, inst_mesh, transforms, per_instance: int = 40, seed: int = 3):
    """points in and around each instance's world box (1.3 times its size), with the index of that instance"""
    rng = np.random.default_rng(seed)
    pts, owner = [], []
    for i, m in enumerate(inst_mesh):
        v = np.asarray(meshes[int(m)][0], np.float64) @ transforms[i, :, :3].astype(np.float64).T + transforms[i, :, 3]
        lo, hi = v.min(0), v.max(0)
        c, h = (lo + hi) / 2, (hi - lo) / 2 * 1.3
        pts.append(c + rng.uniform(-1, 1, size=(per_instance, 3)) * h)
        owner.append(np.full(per_instance, i))
    return np.concatenate(pts).astype(np.float32), np.concatenate(owner)
