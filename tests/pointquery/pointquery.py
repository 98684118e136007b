"""Closest-point test infrastructure: ctypes front ends of point_oracle.c (CPU oracle, MIRROR / TRUTH) and
pointsim.cpp (host simulator of rt_point.cuh).  TEST INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it,
the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
_ORACLE = None
_SIM = None
TRUTH, MIRROR = oracle.TRUTH, oracle.MIRROR


def _stale(so, deps):
    return not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps)


def build(force: bool = False) -> tuple[str, str]:
    """Compile libpointoracle.so (gcc + OpenMP) and libpointsim.so (g++) next to this file."""
    so_o = os.path.join(_HERE, "libpointoracle.so")
    deps_o = [os.path.join(_HERE, f) for f in ("point_oracle.c", "point_tri.inc")]
    if force or _stale(so_o, deps_o):
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.check_call([cc, "-O2", "-fopenmp", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-o", so_o,
                               deps_o[0], "-lm"])
    so_s = os.path.join(_HERE, "libpointsim.so")
    deps_s = [os.path.join(_HERE, "pointsim.cpp")] + [os.path.join(_CSRC, f) for f in ("rt_core.cuh", "rt_traverse.cuh", "rt_point.cuh")]
    if force or _stale(so_s, deps_s):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", deps_s[0], "-o", so_s])
    return so_o, so_s


def _libs():
    global _ORACLE, _SIM
    if _ORACLE is None:
        so_o, so_s = build()
        lo = C.CDLL(so_o)
        lo.point_bvh_build.restype = C.c_void_p
        lo.point_bvh_build.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
        lo.point_bvh_free.argtypes = [C.c_void_p]
        lo.point_query.restype = C.c_int
        lo.point_query.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int64, C.c_void_p,
                                   C.c_double] + [C.c_void_p] * 5
        lo.point_all_d2.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
        lo.point_num_threads.restype = C.c_int
        ls = C.CDLL(so_s)
        ls.hs_closest_point.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_float] + [C.c_void_p] * 6
        ls.hs_slot_bounds_check.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        ls.hs_point_tri.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _ORACLE, _SIM = lo, ls
    return _ORACLE, _SIM


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pts(points) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 3))


def num_threads() -> int:
    return int(_libs()[0].point_num_threads())


class PointMesh:
    """Mesh + optional median-split BVH2 of the point oracle (same answers as brute force)."""

    def __init__(self, vertices, faces, use_bvh: bool | None = None):
        self.vertices = np.ascontiguousarray(np.asarray(vertices, dtype=np.float32).reshape(-1, 3))
        self.faces = np.ascontiguousarray(np.asarray(faces, dtype=np.int32).reshape(-1, 3))
        if use_bvh is None:
            use_bvh = len(self.faces) > 64
        self._bvh = _libs()[0].point_bvh_build(_p(self.vertices), len(self.vertices), _p(self.faces), len(self.faces)) if use_bvh else None

    def __del__(self):
        if getattr(self, "_bvh", None):
            _libs()[0].point_bvh_free(self._bvh)
            self._bvh = None


def query(mesh: PointMesh, points, mode: int = MIRROR, max_distance: float = float("inf"), brute: bool = False) -> dict:
    """Closest point of every point of a flat [n,3] batch: closest, distance, tri, uv, d2 (float32 in MIRROR mode,
    float64 in TRUTH mode; tri int32, -1 = none)."""
    p = _pts(points)
    n = len(p)
    closest = np.zeros((n, 3)); distance = np.zeros(n); tri = np.zeros(n, np.int32); uv = np.zeros((n, 2)); d2 = np.zeros(n)
    rc = _libs()[0].point_query(_p(mesh.vertices), len(mesh.vertices), _p(mesh.faces), len(mesh.faces),
                                None if brute else mesh._bvh, int(mode), n, _p(p), float(max_distance), _p(closest),
                                _p(distance), _p(tri), _p(uv), _p(d2))
    if rc != 0:
        raise RuntimeError(f"point_query failed: {rc}")
    out = dict(closest=closest, distance=distance, tri=tri, uv=uv, d2=d2)
    if mode == MIRROR:
        for k in ("closest", "distance", "uv", "d2"):
            out[k] = out[k].astype(np.float32)
    return out


def all_d2(mesh: PointMesh, points, mode: int = TRUTH) -> np.ndarray:
    """[n, n_faces] squared distance of every (point, triangle) pair."""
    p = _pts(points)
    out = np.zeros((len(p), len(mesh.faces)))
    _libs()[0].point_all_d2(_p(mesh.vertices), len(mesh.vertices), _p(mesh.faces), len(mesh.faces), int(mode), len(p), _p(p), _p(out))
    return out


class PointOracleIntersector(oracle.OracleIntersector):
    """oracle.OracleIntersector plus the closest-point queries (trimesh.proximity)."""

    def __init__(self, vertices, faces, mode: int = MIRROR, use_bvh: bool | None = None):
        super().__init__(vertices, faces, mode, use_bvh)
        self.pmesh = PointMesh(vertices, faces, use_bvh)

    def closest_point(self, points, max_distance: float = float("inf")):
        """(closest [*b,3], distance [*b], tri [*b], uv [*b,2])"""
        b = np.asarray(points).shape[:-1]
        r = query(self.pmesh, points, self.mode, max_distance)
        return r["closest"].reshape(*b, 3), r["distance"].reshape(b), r["tri"].reshape(b), r["uv"].reshape(*b, 2)

    def signed_distance(self, points):
        """distance, positive where the oracle's contains_points says inside (exact 0 stays +0)"""
        p = np.asarray(points, dtype=np.float32).reshape(-1, 3)
        _, d, _, _ = self.closest_point(p)
        inside = self.contains_points(p)
        return np.where(inside | (d == 0), d, -d)


# ------------------------------------------------------------------ host simulator
def sim_closest_point(blob: np.ndarray, points, max_distance: float = float("inf")) -> dict:
    p = _pts(points)
    n = len(p)
    closest = np.zeros((n, 3), np.float32); distance = np.zeros(n, np.float32); tri = np.zeros(n, np.int32)
    uv = np.zeros((n, 2), np.float32); stats = np.zeros(4, np.uint64); ms = np.zeros(1, np.int32)
    rc = _libs()[1].hs_closest_point(_p(np.ascontiguousarray(blob)), n, _p(p), C.c_float(max_distance), _p(closest),
                                     _p(distance), _p(tri), _p(uv), _p(stats), _p(ms))
    if rc != 0:
        raise RuntimeError(f"hs_closest_point failed: {rc}")
    return dict(closest=closest, distance=distance, tri=tri, uv=uv,
                stats=dict(nodes=int(stats[0]), tris=int(stats[1]), points=int(stats[2]), found=int(stats[3])),
                max_stack=int(ms[0]))


def slot_bounds_check(blob: np.ndarray, points) -> tuple[int, int, float]:
    """(violations, slot/subtree pairs checked, worst bound / d2 ratio) of slot_lower_bounds over every node."""
    p = _pts(points)
    out = np.zeros(2, np.uint64); worst = np.zeros(1, np.float64)
    rc = _libs()[1].hs_slot_bounds_check(_p(np.ascontiguousarray(blob)), len(p), _p(p), _p(out), _p(worst))
    if rc != 0:
        raise RuntimeError(f"hs_slot_bounds_check failed: {rc}")
    return int(out[0]), int(out[1]), float(worst[0])


def sim_point_tri(point, tri_vertices) -> np.ndarray:
    """rt_point.cuh point_tri on the host: [cx, cy, cz, d2, w0, w1] (float32)."""
    out = np.zeros(6, np.float32)
    _libs()[1].hs_point_tri(_p(np.ascontiguousarray(point, dtype=np.float32)),
                            _p(np.ascontiguousarray(tri_vertices, dtype=np.float32).reshape(9)), _p(out))
    return out
