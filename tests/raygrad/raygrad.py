"""Hit-gradient test infrastructure: the ctypes front end of rgsim.cpp (host simulator of rt_ray_grad), a binary64
numpy restatement of the same formula, and a binary64 ray/triangle intersection for finite differences.  TEST
INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it, the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(_HERE, "..", "distgrad"))
import distgrad  # noqa: E402

_SIM = None


def build(force: bool = False) -> str:
    """Compile librgsim.so (g++) next to this file."""
    return distgrad.compile_sim(os.path.join(_HERE, "rgsim.cpp"), ("rt_core.cuh", "rt_distgrad.cuh", "rt_raygrad.cuh"),
                                force)


def _lib():
    global _SIM
    if _SIM is None:
        ls = C.CDLL(build())
        vp, i64 = C.c_void_p, C.c_int64
        ls.rg_grad.argtypes = [i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, vp, i64, i64, vp, vp, vp]
        ls.rg_row_values.argtypes = [i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, vp, i64, vp, vp, vp, vp, vp]
        _SIM = ls
    return _SIM


def _f32(a, shape):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(shape))


def _i32(a, shape):
    return np.ascontiguousarray(np.asarray(a, np.int32).reshape(shape))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def sim_grad(o, d, tri, grad_loc, grad_uv, vertices, faces, row_ray=None, window: int = 0):
    """(grad_origins [n,3], grad_directions [n,3], grad_vertices [n_verts,3]) float32 of rt_ray_grad for dense
    origins / directions [n,3] and hit rows (tri, grad_loc or None, grad_uv or None, row_ray or None), the vertex
    sums run as windows of `window` rows (0: one window)"""
    o = _f32(o, (-1, 3))
    n = len(o)
    d = _f32(d, (n, 3))
    tri = _i32(tri, (-1,))
    h = len(tri)
    gl = None if grad_loc is None else _f32(grad_loc, (h, 3))
    gu = None if grad_uv is None else _f32(grad_uv, (h, 2))
    rr = None if row_ray is None else _i32(row_ray, (h,))
    v = _f32(vertices, (-1, 3))
    f = _i32(faces, (-1, 3))
    go = np.zeros((n, 3), np.float32)
    gd = np.zeros((n, 3), np.float32)
    gv = np.zeros((len(v), 3), np.float32)
    rc = _lib().rg_grad(n, _p(o), _p(d), h, _p(rr), _p(tri), _p(gl), _p(gu), _p(v), len(v), _p(f), len(f), int(window),
                        _p(go), _p(gd), _p(gv))
    if rc != 0:
        raise RuntimeError(f"rg_grad failed: {rc}")
    return go, gd, gv


def sim_rows(o, d, tri, grad_loc, grad_uv, vertices, faces, row_ray=None):
    """per row of the simulator: (lambda [h,3], t lambda [h,3], q [h,3], w [h,2], live bool [h])"""
    o = _f32(o, (-1, 3))
    d = _f32(d, (len(o), 3))
    tri = _i32(tri, (-1,))
    h = len(tri)
    gl = None if grad_loc is None else _f32(grad_loc, (h, 3))
    gu = None if grad_uv is None else _f32(grad_uv, (h, 2))
    rr = None if row_ray is None else _i32(row_ray, (h,))
    v = _f32(vertices, (-1, 3))
    f = _i32(faces, (-1, 3))
    lam, tlam, q = (np.zeros((h, 3), np.float32) for _ in range(3))
    w = np.zeros((h, 2), np.float32)
    live = np.zeros(h, np.uint8)
    _lib().rg_row_values(len(o), _p(o), _p(d), h, _p(rr), _p(tri), _p(gl), _p(gu), _p(v), len(v), _p(f), len(f),
                         _p(lam), _p(tlam), _p(q), _p(w), _p(live))
    return lam, tlam, q, w, live.astype(bool)


def _rows(o, d, tri, vertices, faces, row_ray):
    o = np.asarray(o, np.float64).reshape(-1, 3)
    d = np.asarray(d, np.float64).reshape(-1, 3)
    tri = np.asarray(tri, np.int64).reshape(-1)
    ray = np.arange(len(tri)) if row_ray is None else np.asarray(row_ray, np.int64).reshape(-1)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    v = np.asarray(vertices, np.float64).reshape(-1, 3)
    ok = (tri >= 0) & (tri < len(f)) & (ray >= 0) & (ray < len(o))
    fi = f[np.where(ok, tri, 0)] if len(f) else np.zeros((len(tri), 3), np.int64)
    ok &= ((fi >= 0) & (fi < len(v))).all(1)
    fi = np.where(ok[:, None], fi, 0)
    rs = np.where(ok, ray, 0)
    return o[rs], d[rs], v[fi[:, 0]], v[fi[:, 1]], v[fi[:, 2]], fi, ray, ok


def hit64(o, d, v0, v1, v2):
    """binary64 Moeller-Trumbore of DESIGN.md §4.10 for given triangles: (t, b1, b2, det, p, e1, e2)"""
    e1, e2, s = v1 - v0, v2 - v0, o - v0
    p = np.cross(d, e2)
    det = (e1 * p).sum(1)
    with np.errstate(all="ignore"):
        r = np.cross(s, e1)
        return (e2 * r).sum(1) / det, (s * p).sum(1) / det, (d * r).sum(1) / det, det, p, e1, e2


def locate64(o, d, tri, vertices, faces):
    """binary64 (loc [h,3], uv [h,2]) of ray i against triangle tri[i] (no inside test: for finite differences)"""
    o, d, v0, v1, v2, _, _, _ = _rows(o, d, tri, vertices, faces, None)
    t, b1, b2, _, _, _, _ = hit64(o, d, v0, v1, v2)
    w0 = 1.0 - b1 - b2
    return w0[:, None] * v0 + b1[:, None] * v1 + b2[:, None] * v2, np.stack([w0, b1], 1)


def reference(o, d, tri, grad_loc, grad_uv, vertices, faces, row_ray=None):
    """binary64 grad_origins, grad_directions and grad_vertices (np.add.at) of the same formula and zero rules"""
    n = len(np.asarray(o).reshape(-1, 3))
    ro, rd, v0, v1, v2, fi, ray, ok = _rows(o, d, tri, vertices, faces, row_ray)
    h = len(ok)
    gl = np.zeros((h, 3)) if grad_loc is None else np.asarray(grad_loc, np.float64).reshape(h, 3)
    gu = np.zeros((h, 2)) if grad_uv is None else np.asarray(grad_uv, np.float64).reshape(h, 2)
    t, b1, b2, det, p, e1, e2 = hit64(ro, rd, v0, v1, v2)
    with np.errstate(all="ignore"):
        gb1 = (gl * e1).sum(1) - gu[:, 0] + gu[:, 1]
        gb2 = (gl * e2).sum(1) - gu[:, 0]
        lam = (gb1[:, None] * p + gb2[:, None] * np.cross(e1, rd)) / det[:, None]
        w = np.stack([1.0 - b1 - b2, b1, b2], 1)
        q = lam - gl
        tl = t[:, None] * lam
    ok &= (det != 0) & np.isfinite(lam).all(1) & np.isfinite(tl).all(1) & np.isfinite(q).all(1) & np.isfinite(w).all(1)
    go, gd = np.zeros((n, 3)), np.zeros((n, 3))
    np.add.at(go, ray[ok], lam[ok])
    np.add.at(gd, ray[ok], tl[ok])
    gv = np.zeros((len(np.asarray(vertices).reshape(-1, 3)), 3))
    for k in range(3):
        np.add.at(gv, fi[ok, k], -w[ok, k:k + 1] * q[ok])
    return go, gd, gv
