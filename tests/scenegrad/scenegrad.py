"""Instanced-scene gradient test infrastructure: the ctypes front end of sgsim.cpp (host simulator of
rt_scene_grad.cu) on a table prepared by tests/scene, and a numpy restatement of the contract of DESIGN.md §4.13
(binary32 per-row arithmetic written out in numpy, and distgrad's fixed tree order).  TEST INFRASTRUCTURE ONLY:
tests, tools and __graft_entry__ import it, the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
sys.path.insert(0, os.path.join(_HERE, "..", "scene"))
import scene  # noqa: E402

_SIM = None
TRANSFORMS, VERTICES = 1, 2


def build(force: bool = False) -> str:
    """Compile libsgsim.so (g++) next to this file."""
    so = os.path.join(_HERE, "libsgsim.so")
    deps = [os.path.join(_HERE, "sgsim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                 ("rt_core.cuh", "rt_distgrad.cuh", "rt_raygrad.cuh", "rt_scene.cuh",
                                                  "rt_scenegrad.cuh")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", "-I", os.path.join(_HERE, "..", "..", "include"), deps[0],
                               "-o", so])
    return so


def _lib():
    global _SIM
    if _SIM is None:
        s = C.CDLL(build())
        vp, i64, ci = C.c_void_p, C.c_int64, C.c_int
        s.sg_ray_grad.argtypes = [vp, i64, vp, i64, i64, i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, ci, vp, vp, vp, vp]
        s.sg_point_grad.argtypes = [vp, i64, vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, i64, ci, vp, vp, vp]
        s.sg_hit_rows.argtypes = [vp, i64, vp, i64, i64, i64, vp, vp, i64, vp, vp, vp, vp, vp] + [vp] * 7
        _SIM = s
    return _SIM


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a, shape):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(shape))


def _i32(a, shape):
    return np.ascontiguousarray(np.asarray(a, np.int32).reshape(shape))


class SimGradScene:
    """A host scene (scene.SimScene) plus its member table: members [(vertices, faces)] in mesh order."""

    def __init__(self, meshes, inst_mesh, transforms):
        self.meshes = [(_f32(v, (-1, 3)), _i32(f, (-1, 3))) for v, f in meshes]
        self.sim = scene.SimScene([scene.hostsim.build_blob(v, f) for v, f in self.meshes], inst_mesh, transforms)
        self.n_inst = len(self.sim.inst_mesh)
        self.base = np.concatenate([[0], np.cumsum([len(v) for v, _ in self.meshes])]).astype(np.int64)
        self.n_verts = int(self.base[-1])
        rows = np.zeros((max(len(self.meshes), 1), 5), np.int64)
        for k, (v, f) in enumerate(self.meshes):
            rows[k] = [v.ctypes.data, f.ctypes.data, len(v), len(f), self.base[k]]
        self.members = rows
        self.transforms = self.sim.transforms

    def _scene(self):
        return (_p(self.sim.table), self.n_inst, _p(self.members), len(self.meshes), self.n_verts)

    def ray_grad(self, o, d, inst, tri, grad_loc, grad_uv, row_ray=None, window: int = 0, outputs: int = 3):
        """(grad_origins, grad_directions, grad_transforms [I,3,4], grad_vertices [n_verts,3]) float32"""
        o = _f32(o, (-1, 3)); n = len(o); d = _f32(d, (n, 3))
        tri = _i32(tri, (-1,)); h = len(tri); inst = _i32(inst, (h,))
        gl = None if grad_loc is None else _f32(grad_loc, (h, 3))
        gu = None if grad_uv is None else _f32(grad_uv, (h, 2))
        rr = None if row_ray is None else _i32(row_ray, (h,))
        go, gd = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        gt, gv = np.zeros((self.n_inst, 3, 4), np.float32), np.zeros((self.n_verts, 3), np.float32)
        _lib().sg_ray_grad(*self._scene(), n, _p(o), _p(d), h, _p(rr), _p(inst), _p(tri), _p(gl), _p(gu), int(window),
                           int(outputs), _p(go), _p(gd), _p(gt), _p(gv))
        return go, gd, gt, gv

    def point_grad(self, p, grad_out, value, closest, inst, tri, uv, window: int = 0, outputs: int = 3):
        """(grad_points, grad_transforms [I,3,4], grad_vertices [n_verts,3]) float32"""
        p = _f32(p, (-1, 3)); n = len(p)
        args = [_f32(grad_out, (n,)), _f32(value, (n,)), _f32(closest, (n, 3)), _i32(inst, (n,)), _i32(tri, (n,)),
                _f32(uv, (n, 2))]
        gp = np.zeros((n, 3), np.float32)
        gt, gv = np.zeros((self.n_inst, 3, 4), np.float32), np.zeros((self.n_verts, 3), np.float32)
        _lib().sg_point_grad(*self._scene(), n, _p(p), *[_p(a) for a in args], int(window), int(outputs), _p(gp),
                             _p(gt), _p(gv))
        return gp, gt, gv

    def hit_rows(self, o, d, inst, tri, grad_loc, grad_uv, row_ray=None):
        """per row: dict(lam, tlam, q, qo, x [h,3], w [h,2], live bool [h])"""
        o = _f32(o, (-1, 3)); n = len(o); d = _f32(d, (n, 3))
        tri = _i32(tri, (-1,)); h = len(tri); inst = _i32(inst, (h,))
        gl = None if grad_loc is None else _f32(grad_loc, (h, 3))
        gu = None if grad_uv is None else _f32(grad_uv, (h, 2))
        rr = None if row_ray is None else _i32(row_ray, (h,))
        out = {k: np.zeros((h, 3), np.float32) for k in ("lam", "tlam", "q", "qo", "x")}
        out["w"] = np.zeros((h, 2), np.float32)
        live = np.zeros(h, np.uint8)
        _lib().sg_hit_rows(*self._scene(), n, _p(o), _p(d), h, _p(rr), _p(inst), _p(tri), _p(gl), _p(gu),
                           *[_p(out[k]) for k in ("lam", "tlam", "q", "qo", "x", "w")], _p(live))
        out["live"] = live.astype(bool)
        return out


# ------------------------------------------------------------------ numpy restatement of the contract (§4.13)
def _affine_row(m0, m1, m2, c, x, y, z):
    """affine_row in binary32: ffma steps (exact product + one rounding, via float64), zero coefficients skipped"""
    acc = np.float32(c)
    for m, v in ((m2, z), (m1, y), (m0, x)):
        if m != 0:
            acc = np.float32(np.float64(m) * np.float64(v) + np.float64(acc))
    return acc


def tree_sum(contribs: np.ndarray) -> np.ndarray:
    """distgrad's fixed order for one key's list [n,3] float32: groups of 32 left to right, level after level"""
    s = np.asarray(contribs, np.float32)
    while len(s) > 32:
        s = np.stack([_left_sum(s[i:i + 32]) for i in range(0, len(s), 32)])
    return _left_sum(s)


def _left_sum(g):
    acc = g[0].copy()
    for r in g[1:]:
        acc = (acc + r).astype(np.float32)
    return acc


def restate_point(gs: SimGradScene, p, grad_out, value, closest, inst, tri, uv, window: int = 0):
    """grad_points, grad_transforms and grad_vertices of point rows written out from the contract with numpy binary32
    operations, the per-key lists in ascending (row, corner) order summed by tree_sum per window."""
    p = _f32(p, (-1, 3)); n = len(p)
    recs = gs.sim.records()
    fwd_all = recs[:, :12]
    mesh_of = recs[:, 24].view(np.int32)
    gp = np.zeros((n, 3), np.float32)
    lists: dict = {}
    window = n if window <= 0 else window
    acc = np.zeros((gs.n_verts + 4 * gs.n_inst, 3), np.float32)
    for base in range(0, n, window):
        lists = {}
        for i in range(base, min(n, base + window)):
            row = _point_row(gs, fwd_all, mesh_of, p[i], grad_out[i], value[i], closest[i], int(inst[i]), int(tri[i]),
                             uv[i])
            if row is None:
                continue
            q, qo, x, w, vkeys, ins = row
            gp[i] = q
            for k in range(3):
                lists.setdefault(vkeys[k], []).append((-w[k] * qo).astype(np.float32))
            for j in range(4):
                c = (-x[j] * q).astype(np.float32) if j < 3 else -q
                lists.setdefault(gs.n_verts + 4 * ins + j, []).append(c)
        for key, cs in lists.items():
            acc[key] = (acc[key] + tree_sum(np.stack(cs))).astype(np.float32)
    gt = acc[gs.n_verts:].reshape(gs.n_inst, 4, 3).transpose(0, 2, 1).copy()
    return gp, gt, acc[:gs.n_verts].copy()


def _point_row(gs, fwd_all, mesh_of, p, g, value, c, inst, tri, uv):
    f32 = np.float32
    if not (0 <= inst < gs.n_inst):
        return None
    m = int(mesh_of[inst])
    v_m, f_m = gs.meshes[m]
    if not (0 <= tri < len(f_m)):
        return None
    idx = f_m[tri]
    if ((idx < 0) | (idx >= len(v_m))).any():
        return None
    a = abs(f32(value))
    if not (a > 0 and np.isfinite(a)):
        return None
    gsn = -f32(g) if f32(value) < 0 else f32(g)
    q = np.array([f32(gsn * f32(f32(p[k] - c[k]) / a)) for k in range(3)], np.float32)
    w0, w1 = f32(uv[0]), f32(uv[1])
    w2 = f32(f32(f32(1) - w0) - w1)
    v = v_m[idx]
    x = np.array([f32(f32(f32(w0 * v[0, k]) + f32(w1 * v[1, k])) + f32(w2 * v[2, k])) for k in range(3)], np.float32)
    fw = fwd_all[inst]
    qo = np.array([_affine_row(fw[k], fw[4 + k], fw[8 + k], f32(-0.0), q[0], q[1], q[2]) for k in range(3)], np.float32)
    w = np.array([w0, w1, w2], np.float32)
    if not (np.isfinite(q).all() and np.isfinite(qo).all() and np.isfinite(x).all() and np.isfinite(w).all()):
        return None
    return q, qo, x, w, [int(gs.base[m] + idx[k]) for k in range(3)], inst
