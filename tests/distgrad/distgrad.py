"""Distance-gradient test infrastructure: the ctypes front end of dgsim.cpp (host simulator of rt_distgrad.cu) and
a binary64 numpy reference of the same formula.  TEST INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it,
the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
_SIM = None
GROUP = 32          # rt_distgrad.cuh kDgGroup


def _stale(so, deps):
    return not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps)


def build(force: bool = False) -> str:
    """Compile libdgsim.so (g++) next to this file."""
    so = os.path.join(_HERE, "libdgsim.so")
    deps = [os.path.join(_HERE, "dgsim.cpp")] + [os.path.join(_CSRC, f) for f in ("rt_core.cuh", "rt_distgrad.cuh")]
    if force or _stale(so, deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", deps[0], "-o", so])
    return so


def _lib():
    global _SIM
    if _SIM is None:
        ls = C.CDLL(build())
        ls.dg_grad.argtypes = [C.c_int64] + [C.c_void_p] * 7 + [C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        _SIM = ls
    return _SIM


def _f32(a, shape):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(shape))


def sim_grad(points, g, value, closest, tri, uv, faces, n_verts: int, window: int = 0):
    """(grad_points float32 [n,3], grad_vertices float32 [n_verts,3]) of rt_distance_grad for a dense batch, run as
    windows of `window` points (0: one window)"""
    p = _f32(points, (-1, 3))
    n = len(p)
    faces = np.ascontiguousarray(np.asarray(faces, np.int32).reshape(-1, 3))
    args = [_f32(g, (n,)), _f32(value, (n,)), _f32(closest, (n, 3)),
            np.ascontiguousarray(np.asarray(tri, np.int32).reshape(n)), _f32(uv, (n, 2)), faces]
    gp = np.zeros((n, 3), np.float32)
    gv = np.zeros((int(n_verts), 3), np.float32)
    rc = _lib().dg_grad(n, p.ctypes.data_as(C.c_void_p), *[a.ctypes.data_as(C.c_void_p) for a in args], len(faces),
                        int(n_verts), int(window), gp.ctypes.data_as(C.c_void_p), gv.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise RuntimeError(f"dg_grad failed: {rc}")
    return gp, gv


def reference(points, g, value, closest, tri, uv, faces, n_verts: int):
    """binary64 grad_points and grad_vertices (np.add.at) of the same formula and the same zero rules"""
    p = np.asarray(points, np.float64).reshape(-1, 3)
    value = np.asarray(value, np.float64).reshape(-1)
    tri = np.asarray(tri).reshape(-1)
    a = np.abs(value)
    live = (a > 0) & np.isfinite(a) & (tri >= 0) & (tri < len(faces))
    s = np.where(np.signbit(value), -1.0, 1.0)
    q = np.zeros_like(p)
    q[live] = (np.asarray(g, np.float64).reshape(-1)[live] * s[live] / a[live])[:, None] * \
        (p[live] - np.asarray(closest, np.float64).reshape(-1, 3)[live])
    uv = np.asarray(uv, np.float64).reshape(-1, 2)
    w = np.stack([uv[:, 0], uv[:, 1], 1.0 - uv[:, 0] - uv[:, 1]], 1)
    gv = np.zeros((int(n_verts), 3))
    f = np.asarray(faces).reshape(-1, 3)
    for k in range(3):
        np.add.at(gv, f[tri[live], k], -w[live, k:k + 1] * q[live])
    return q, gv


def tree_sum(c: np.ndarray) -> np.ndarray:
    """float32 sum of one vertex's contributions [L, 3] in the documented order: groups of GROUP left to right, then
    the same over the group sums, until one value remains"""
    c = np.asarray(c, np.float32)
    while len(c) > 1:
        out = []
        for i in range(0, len(c), GROUP):
            s = c[i].copy()
            for x in c[i + 1:i + GROUP]:
                s = (s + x).astype(np.float32)
            out.append(s)
        c = np.asarray(out, np.float32)
    return c[0]
