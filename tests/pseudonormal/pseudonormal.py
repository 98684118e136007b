"""Pseudo-normal test infrastructure: the ctypes front end of pnsim.cpp (host simulator of rt_pseudonormal.cu and of
the signed-distance kernel) and a binary64 truth built from the brute-force oracles of tests/pointquery (distance to
the surface) and tests/winding (inside = winding number > 1/2).  TEST INFRASTRUCTURE ONLY: tests, tools and
__graft_entry__ import it, the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
for _d in ("pointquery", "winding"):
    _p_ = os.path.join(_HERE, "..", _d)
    if _p_ not in sys.path:
        sys.path.insert(0, _p_)
import pointquery as _pq  # noqa: E402
import winding as _W  # noqa: E402

_SIM = None


def _stale(so, deps):
    return not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps)


def build(force: bool = False) -> str:
    """Compile libpnsim.so (g++) next to this file."""
    so = os.path.join(_HERE, "libpnsim.so")
    deps = [os.path.join(_HERE, "pnsim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                 ("rt_core.cuh", "rt_traverse.cuh", "rt_point.cuh", "rt_winding.cuh",
                                                  "rt_pseudonormal.cuh")]
    if force or _stale(so, deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", deps[0], "-o", so])
    return so


def _lib():
    global _SIM
    if _SIM is None:
        ls = C.CDLL(build())
        ls.pn_normals.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        ls.pn_signed_distance.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        ls.pn_region.restype = C.c_uint32
        ls.pn_region.argtypes = [C.c_void_p, C.c_void_p]
        _SIM = ls
    return _SIM


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pts(points) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 3))


def n_tris(blob: np.ndarray) -> int:
    return int(np.frombuffer(np.ascontiguousarray(blob)[8:12].tobytes(), np.uint32)[0])


def sim_normals(blob: np.ndarray) -> tuple[np.ndarray, tuple[int, int, int]]:
    """(float32 [n_tris, 24] rows: vertex a, b, c, edge ab, ac, bc as float4; (boundary, non-manifold, inconsistent))"""
    blob = np.ascontiguousarray(blob)
    rows = np.zeros((n_tris(blob), 24), np.float32)
    counts = np.zeros(3, np.uint64)
    rc = _lib().pn_normals(_p(blob), _p(rows), _p(counts))
    if rc != 0:
        raise RuntimeError(f"pn_normals failed: {rc}")
    return rows, tuple(int(c) for c in counts)


def sim_signed_distance(blob: np.ndarray, points, normals: np.ndarray | None = None) -> dict:
    """signed distances (float32) and counters {nodes, tris, points, found} of the signed-distance kernel"""
    blob = np.ascontiguousarray(blob)
    if normals is None:
        normals = sim_normals(blob)[0]
    normals = np.ascontiguousarray(normals, dtype=np.float32)
    p = _pts(points)
    sd = np.zeros(len(p), np.float32)
    stats = np.zeros(4, np.uint64)
    rc = _lib().pn_signed_distance(_p(blob), _p(normals), len(p), _p(p), _p(sd), _p(stats))
    if rc != 0:
        raise RuntimeError(f"pn_signed_distance failed: {rc}")
    return dict(sd=sd, stats=dict(nodes=int(stats[0]), tris=int(stats[1]), points=int(stats[2]), found=int(stats[3])))


REGIONS = ("face", "a", "b", "c", "ab", "ac", "bc")


def sim_region(point, tri_vertices) -> str:
    """point_tri's Voronoi region of the closest point on one triangle"""
    r = _lib().pn_region(_p(np.ascontiguousarray(point, dtype=np.float32)),
                         _p(np.ascontiguousarray(tri_vertices, dtype=np.float32).reshape(9)))
    return REGIONS[r]


# ------------------------------------------------------------------ binary64 truth
def truth(vertices, faces, points) -> tuple[np.ndarray, np.ndarray]:
    """(distance to the surface in binary64, inside by the binary64 winding number > 1/2) of every point"""
    p = _pts(points)
    d = _pq.query(_pq.PointMesh(vertices, faces), p, _pq.TRUTH)["distance"]
    return d, _W.truth(vertices, faces, p) > 0.5


# ------------------------------------------------------------------ test meshes
def torus(n_major: int = 48, n_minor: int = 24, R: float = 1.0, r: float = 0.35):
    """closed torus around z, outward orientation"""
    u = 2 * np.pi * np.arange(n_major) / n_major
    w = 2 * np.pi * np.arange(n_minor) / n_minor
    uu, ww = np.meshgrid(u, w, indexing="ij")
    v = np.stack([(R + r * np.cos(ww)) * np.cos(uu), (R + r * np.cos(ww)) * np.sin(uu), r * np.sin(ww)], -1)
    idx = np.arange(n_major * n_minor).reshape(n_major, n_minor)
    a, b = idx, np.roll(idx, -1, 0)
    c, d = np.roll(idx, -1, 1), np.roll(b, -1, 1)
    f = np.concatenate([np.stack([a, b, d], -1).reshape(-1, 3), np.stack([a, d, c], -1).reshape(-1, 3)])
    return v.reshape(-1, 3).astype(np.float32), f.astype(np.int32)


def star_prism(points: int = 5, r_out: float = 1.0, r_in: float = 0.38, height: float = 0.5):
    """a star polygon extruded along z: acute convex edges at the tips (where a face normal alone gives the wrong
    sign), reflex (concave) edges at the inner corners and saddle vertices where those meet the caps"""
    k = 2 * points
    ang = np.pi / 2 + 2 * np.pi * np.arange(k) / k
    rad = np.where(np.arange(k) % 2 == 0, r_out, r_in)
    ring = np.stack([rad * np.cos(ang), rad * np.sin(ang)], -1)                 # CCW seen from +z
    bot = np.concatenate([ring, np.zeros((k, 1))], 1)
    top = np.concatenate([ring, np.full((k, 1), height)], 1)
    v = np.concatenate([bot, top, [[0, 0, 0], [0, 0, height]]]).astype(np.float32)
    cb, ct = 2 * k, 2 * k + 1
    f = []
    for i in range(k):
        j = (i + 1) % k
        f += [[i, j, k + j], [i, k + j, k + i], [ct, k + i, k + j], [cb, j, i]]
    return v, np.asarray(f, np.int32)


def voxels(cells):
    """closed outward surface of a union of unit cubes (integer cell corners), two triangles per exposed unit face;
    vertices welded"""
    cells = {tuple(int(x) for x in c) for c in cells}
    quads = []
    for c in sorted(cells):
        for axis in range(3):
            for s in (-1, 1):
                nb = list(c); nb[axis] += s
                if tuple(nb) in cells:
                    continue
                a1, a2 = (axis + 1) % 3, (axis + 2) % 3          # (a1, a2, axis) is right-handed
                base = np.array(c, np.float64); base[axis] += 1 if s > 0 else 0
                e1, e2 = np.eye(3)[a1], np.eye(3)[a2]
                q = [base, base + e1, base + e1 + e2, base + e2]
                quads.append(q if s > 0 else q[::-1])
    pts = np.array(quads).reshape(-1, 3)
    v, inv = np.unique(pts, axis=0, return_inverse=True)
    q = inv.reshape(-1, 4)
    f = np.concatenate([q[:, [0, 1, 2]], q[:, [0, 2, 3]]])
    return v.astype(np.float32), f.astype(np.int32)


def notched_cube():
    """2 x 2 x 2 cells without one corner cell: three reflex edges meeting in a concave vertex at (1, 1, 1)"""
    return voxels([(x, y, z) for x in range(2) for y in range(2) for z in range(2) if (x, y, z) != (1, 1, 1)])


def soup(v, f):
    """the same triangles with every corner its own vertex (an STL-style soup)"""
    return np.ascontiguousarray(np.asarray(v, np.float32)[np.asarray(f)].reshape(-1, 3)), \
        np.arange(3 * len(f), dtype=np.int32).reshape(-1, 3)
