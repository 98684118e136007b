"""Instanced-scene test infrastructure: ctypes front end of scenesim.cpp (host simulator of rt_scene.cuh) and the
flattened-scene reference.  TEST INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it, the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
sys.path.insert(0, os.path.join(_HERE, "..", "hostsim"))
import hostsim  # noqa: E402

_SIM = None
MODES = {"closest": 0, "any": 1, "count": 2}


def build(force: bool = False) -> str:
    """Compile libscenesim.so (g++) next to this file."""
    so = os.path.join(_HERE, "libscenesim.so")
    deps = [os.path.join(_HERE, "scenesim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                    ("rt_core.cuh", "rt_traverse.cuh", "rt_scene.cuh")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", deps[0], "-o", so])
    return so


def lib():
    global _SIM
    if _SIM is None:
        s = C.CDLL(build())
        s.ss_table_bytes.restype = C.c_size_t
        s.ss_table_bytes.argtypes = [C.c_int64, C.c_int64]
        s.ss_prepare.argtypes = [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        s.ss_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_float] + [C.c_void_p] * 7
        s.ss_affine_row.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _SIM = s
    return _SIM


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def transforms34(transforms) -> np.ndarray:
    """float32 [I,3,4] from [I,3,4] or [I,4,4]"""
    t = np.asarray(transforms, dtype=np.float32)
    return np.ascontiguousarray(t.reshape(-1, t.shape[-2], 4)[:, :3, :])


class SimScene:
    """A prepared scene on the host: the table (holding the host addresses of `blobs`, kept alive here), the top-level
    geometry and its hostsim blob."""

    def __init__(self, blobs, inst_mesh, transforms):
        self.blobs = [np.ascontiguousarray(b, dtype=np.uint8) for b in blobs]
        self.inst_mesh = np.ascontiguousarray(inst_mesh, dtype=np.int32).reshape(-1)
        self.transforms = transforms34(transforms)
        n = len(self.inst_mesh)
        addrs = np.array([b.ctypes.data for b in self.blobs], dtype=np.uint64)
        self.table = np.zeros(lib().ss_table_bytes(len(self.blobs), n), np.uint8)
        self.tlas_v = np.zeros((2 * n, 3), np.float32)
        self.tlas_f = np.zeros((n, 3), np.int32)
        rc = lib().ss_prepare(len(self.blobs), _p(addrs), n, _p(self.inst_mesh), _p(self.transforms), _p(self.table),
                              _p(self.tlas_v), _p(self.tlas_f))
        if rc != 0:
            raise ValueError("ss_prepare: bad mesh index or transform")
        self.tlas = hostsim.build_blob(self.tlas_v, self.tlas_f)

    def records(self) -> np.ndarray:
        """the instance records as float32 [I, 32] (fwd 12, inv 12, mesh, flags, lo 3, hi 3 as raw words)"""
        off = int(self.table[16:24].view(np.uint64)[0])
        n = len(self.inst_mesh)
        return self.table[off:off + 128 * n].view(np.float32).reshape(n, 32)

    def trace(self, mode: str, origins, directions, tmax: float = 1.0e7, brute: bool = False) -> dict:
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(directions, dtype=np.float32).reshape(-1, 3)
        n = len(o)
        hit = np.zeros(n, np.uint8); front = np.zeros(n, np.uint8); inst = np.zeros(n, np.int32); tri = np.zeros(n, np.int32)
        loc = np.zeros((n, 3), np.float32); uv = np.zeros((n, 2), np.float32); count = np.zeros(n, np.int32)
        rc = lib().ss_trace(_p(self.table), None if brute else _p(self.tlas), MODES[mode], n, _p(o), _p(d), C.c_float(tmax),
                            _p(hit), _p(front), _p(inst), _p(tri), _p(loc), _p(uv), _p(count))
        if rc != 0:
            raise RuntimeError(f"ss_trace failed: {rc}")
        if mode == "closest":
            return dict(hit=hit, front=front, inst=inst, tri=tri, loc=loc, uv=uv)
        if mode == "any":
            return dict(hit=hit)
        return dict(count=count)


def affine_row(m4, xyz) -> np.ndarray:
    p = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
    out = np.zeros(len(p), np.float32)
    lib().ss_affine_row(len(p), _p(np.ascontiguousarray(m4, dtype=np.float32).reshape(4)), _p(p), _p(out))
    return out


def flatten(meshes, inst_mesh, transforms):
    """The scene as one mesh: each instance's vertices transformed in float64 (the binary32 transform's values) and
    rounded to float32, faces offset; returns (vertices, faces, face_inst, face_row)."""
    t = transforms34(transforms).astype(np.float64)
    vs, fs, fi, fr = [], [], [], []
    base = 0
    for i, m in enumerate(np.asarray(inst_mesh).reshape(-1)):
        v, f = meshes[int(m)]
        v = np.asarray(v, dtype=np.float32).astype(np.float64)
        w = v @ t[i, :, :3].T + t[i, :, 3]
        vs.append(w.astype(np.float32)); fs.append(np.asarray(f, dtype=np.int32) + base)
        fi.append(np.full(len(f), i, np.int32)); fr.append(np.arange(len(f), dtype=np.int32))
        base += len(v)
    if not vs:
        return np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32)
    return np.concatenate(vs), np.concatenate(fs), np.concatenate(fi), np.concatenate(fr)
