"""Point queries on instanced scenes, test infrastructure: ctypes front end of scenepointsim.cpp (host simulator of the
point queries of rt_scene.cuh) over a scene prepared by scene.SimScene, and the scene flattened with the kernels'
binary32 world vertices.  TEST INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it, the product never does.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

import scene as _scene

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
_SIM = None
MODES = {"tree": 0, "instances": 1, "brute": 2}


def build(force: bool = False) -> str:
    """Compile libscenepointsim.so (g++) next to this file."""
    import subprocess

    so = os.path.join(_HERE, "libscenepointsim.so")
    deps = [os.path.join(_HERE, "scenepointsim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                         ("rt_core.cuh", "rt_traverse.cuh", "rt_point.cuh",
                                                          "rt_winding.cuh", "rt_pseudonormal.cuh", "rt_scene.cuh")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", deps[0], "-o", so])
    return so


def lib():
    global _SIM
    if _SIM is None:
        s = C.CDLL(build())
        s.ss_point_prepare.argtypes = [C.c_void_p, C.c_void_p]
        s.ss_point_query.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_float] + \
            [C.c_void_p] * 7
        s.ss_bound_check.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _SIM = s
    return _SIM


_p = _scene._p


def point_side(s: _scene.SimScene) -> np.ndarray:
    """the side array of the point queries as float32 [I, 4] (sigma, alpha, beta, 0)"""
    side = np.zeros((max(len(s.inst_mesh), 1), 4), np.float32)
    lib().ss_point_prepare(_p(s.table), _p(side))
    return side[:len(s.inst_mesh)]


def closest_point(s: _scene.SimScene, points, max_distance: float = float("inf"), mode: str = "tree",
                  normals=None) -> dict:
    """closest, distance, inst, tri, uv of rt_scene_closest_point; with `normals` (float32 rows per mesh, as
    pseudonormal.sim_normals) the signed distance `sd` of rt_scene_signed_distance instead of `distance`.
    mode "tree" walks the top-level tree, "instances" every instance in order, "brute" every triangle."""
    p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    n = len(p)
    side = point_side(s)
    out = dict(closest=np.zeros((n, 3), np.float32), distance=np.zeros(n, np.float32), inst=np.zeros(n, np.int32),
               tri=np.zeros(n, np.int32), uv=np.zeros((n, 2), np.float32), sd=np.zeros(n, np.float32))
    addrs = None
    if normals is not None:
        keep = [np.ascontiguousarray(r, dtype=np.float32).reshape(-1) for r in normals]
        keep = [k if k.size else np.zeros(4, np.float32) for k in keep]
        addrs = np.array([k.ctypes.data for k in keep] or [0], dtype=np.uint64)
    rc = lib().ss_point_query(_p(s.table), _p(s.tlas), _p(side), MODES[mode], n, _p(p), C.c_float(max_distance),
                              _p(addrs), *[_p(out[k]) for k in ("closest", "distance", "inst", "tri", "uv", "sd")])
    if rc != 0:
        raise RuntimeError(f"ss_point_query failed: {rc}")
    del out["distance" if normals is not None else "sd"]
    return out


def bound_check(s: _scene.SimScene, points) -> tuple[int, int, float]:
    """(violations, pairs checked, worst bound / d2) of the instance walk's world bound and the instance box bound,
    over every instance, node slot and world triangle below it"""
    p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    side = point_side(s)
    out = np.zeros(2, np.uint64)
    worst = np.zeros(1, np.float64)
    lib().ss_bound_check(_p(s.table), _p(side), len(p), _p(p), _p(out), _p(worst))
    return int(out[0]), int(out[1]), float(worst[0])


def flatten_affine(meshes, inst_mesh, transforms):
    """The scene as one mesh with the kernels' own binary32 world vertices: affine_row of each transform row with
    the offset 0 taken as -0 (DESIGN.md §4.12), faces offset in instance order; returns (vertices, faces,
    face_inst, face_row)."""
    t = _scene.transforms34(transforms)
    vs, fs, fi, fr = [], [], [], []
    base = 0
    for i, m in enumerate(np.asarray(inst_mesh).reshape(-1)):
        v, f = meshes[int(m)]
        v = np.asarray(v, dtype=np.float32).reshape(-1, 3)
        w = np.zeros_like(v)
        for k in range(3):
            row = t[i, k].copy()
            if row[3] == 0.0:
                row[3] = np.float32(-0.0)
            w[:, k] = _scene.affine_row(row, v)
        vs.append(w); fs.append(np.asarray(f, dtype=np.int32).reshape(-1, 3) + base)
        fi.append(np.full(len(f), i, np.int32)); fr.append(np.arange(len(f), dtype=np.int32))
        base += len(v)
    if not vs:
        return np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32)
    return np.concatenate(vs), np.concatenate(fs), np.concatenate(fi), np.concatenate(fr)
