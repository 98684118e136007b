"""Instanced scenes shared by the scene tests (test infrastructure): meshes, transforms and rays."""
from __future__ import annotations

import numpy as np

from triro import synth


def meshes():
    """(vertices, faces) of the scene meshes: an icosphere, a soup, a heightfield and an empty mesh."""
    return [synth.icosphere(2), synth.triangle_soup(400, sigma=0.05, seed=3), synth.heightfield(16, 12, 0.2),
            (np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))]


def random_transforms(n: int, seed: int = 0, spread: float = 6.0, mirror_fraction: float = 0.3) -> np.ndarray:
    """float32 [n,3,4]: random rotations times non-uniform scales in [0.3, 2], a share of them mirrored, translations
    in [-spread, spread]^3"""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 3, 4), np.float32)
    for i in range(n):
        q, r = np.linalg.qr(rng.normal(size=(3, 3)))
        q = q * np.sign(np.diag(r))
        if np.linalg.det(q) < 0:
            q[:, 0] = -q[:, 0]
        s = rng.uniform(0.3, 2.0, size=3)
        if rng.uniform() < mirror_fraction:
            s[rng.integers(3)] *= -1.0
        out[i, :, :3] = q * s
        out[i, :, 3] = rng.uniform(-spread, spread, size=3)
    return out


def scene(n_inst: int = 300, seed: int = 0, coincident: int = 8):
    """(meshes, inst_mesh [I], transforms [I,3,4]): instances of every mesh (mostly the first three), the last
    `coincident` instances exact copies of earlier ones, and one instance of the empty mesh."""
    rng = np.random.default_rng(seed + 100)
    ms = meshes()
    inst_mesh = rng.integers(0, 3, size=n_inst).astype(np.int32)
    t = random_transforms(n_inst, seed)
    for k in range(coincident):
        j = n_inst - 1 - k
        src = int(rng.integers(0, n_inst - coincident))
        inst_mesh[j] = inst_mesh[src]
        t[j] = t[src]
    inst_mesh[n_inst // 2] = 3
    return ms, inst_mesh, t


def rays(n: int, seed: int = 1, radius: float = 10.0):
    """random rays: origins in [-radius, radius]^3, directions normalised N(0, I)"""
    rng = np.random.default_rng(seed)
    o = rng.uniform(-radius, radius, size=(n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    return o, (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def camera_rays(w: int = 64, h: int = 48, origin=(0.0, -2.0, 14.0)):
    """pinhole rays of one shared origin looking down -z: origins [h*w,3] (all equal), directions [h*w,3]"""
    o, d = synth.pinhole_rays(w, h, origin=origin)
    return np.ascontiguousarray(o.reshape(-1, 3).numpy()), np.ascontiguousarray(d.reshape(-1, 3).numpy())


def box_rays(blobs, inst_mesh, transforms, per_instance: int = 12, seed: int = 2, reach: float = 3.0):
    """Rays aimed at the corners, edges and faces of the instances' (unpadded) world boxes, from origins within
    `reach` times the box size around them: where the world box test and the object-space walk meet."""
    rng = np.random.default_rng(seed)
    os_, ds = [], []
    for i, m in enumerate(inst_mesh):
        hdr = np.asarray(blobs[int(m)][:256]).view(np.float32)
        lo, hi = hdr[12:15].astype(np.float64), hdr[15:18].astype(np.float64)
        if not (lo <= hi).all() or int(np.asarray(blobs[int(m)][8:12]).view(np.uint32)[0]) == 0:
            continue
        a = transforms[i, :, :3].astype(np.float64)
        b = transforms[i, :, 3].astype(np.float64)
        corners = np.array([[(hi if (c >> k) & 1 else lo)[k] for k in range(3)] for c in range(8)]) @ a.T + b
        wlo, whi = corners.min(0), corners.max(0)
        size = float((whi - wlo).max())
        for k in range(per_instance):
            u = rng.uniform(size=3)
            kind = k % 3          # 0 corner, 1 edge, 2 face: fix 3, 2 or 1 coordinates to the box planes
            fixed = rng.permutation(3)[: 3 - kind]
            for ax in fixed:
                u[ax] = float(rng.integers(2))
            target = wlo + u * (whi - wlo)
            o = target + rng.uniform(-reach, reach, size=3) * size
            d = target - o
            d = d / np.linalg.norm(d)
            os_.append(o); ds.append(d)
    return np.asarray(os_, np.float32).reshape(-1, 3), np.asarray(ds, np.float32).reshape(-1, 3)
