"""ctypes front end of tests/hostsim/hostsim.cpp — TEST INFRASTRUCTURE ONLY.

Steps the product's __host__ __device__ builder/traversal functions on the CPU so that their
logic is covered by the CPU-only test tier, and validates blobs produced on the GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libhostsim.so")
    src = os.path.join(_HERE, "hostsim.cpp")
    csrc = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("rt_core.cuh", "rt_traverse.cuh", "rt_build_core.cuh")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC",
                               "-Wno-unknown-pragmas", src, "-o", so])
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.hs_blob_bytes.restype = C.c_size_t
        _LIB.hs_blob_bytes.argtypes = [C.c_int64]
        _LIB.hs_build.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t]
        _LIB.hs_build_sah.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t]
        _LIB.hs_trace.argtypes = [C.c_void_p, C.c_int, C.c_int64] + [C.c_void_p] * 10
        _LIB.hs_check_blob.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        _LIB.hs_canonical.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        _LIB.hs_frame_check.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _LIB.hs_blob_prims.argtypes = [C.c_void_p, C.c_void_p]
        _LIB.hs_refit.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t]
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def build_blob(vertices, faces) -> np.ndarray:
    v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
    f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    blob = np.zeros(lib().hs_blob_bytes(len(f)), dtype=np.uint8)
    rc = lib().hs_build(_p(v), len(v), _p(f), len(f), _p(blob), blob.nbytes)
    if rc != 0:
        raise RuntimeError(f"hs_build failed: {rc}")
    return blob


def build_blob_sah(vertices, faces) -> np.ndarray:
    """Experiment hook: BVH8 blob collapsed from a binned-SAH binary tree (see hs_build_sah)."""
    v = np.ascontiguousarray(vertices, dtype=np.float32); f = np.ascontiguousarray(faces, dtype=np.int32)
    nb = lib().hs_blob_bytes(len(f))
    blob = np.zeros(nb, dtype=np.uint8)
    rc = lib().hs_build_sah(_p(v), len(v), _p(f), len(f), _p(blob), nb)
    if rc != 0:
        raise RuntimeError(f"hs_build_sah failed: {rc}")
    return blob


def refit_blob(blob: np.ndarray, vertices, faces) -> np.ndarray:
    v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
    f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    out = np.ascontiguousarray(blob).copy()
    rc = lib().hs_refit(_p(v), len(v), _p(f), len(f), _p(out), out.nbytes)
    if rc != 0:
        raise RuntimeError(f"hs_refit failed: {rc}")
    return out


def check_blob(blob: np.ndarray, vertices=None, faces=None):
    """Returns (code, info) — code 0 means valid: structure, conservative slot boxes, parent links, header and layout,
    zero padding.  With vertices and faces also every record against its face and bad_index_faces (codes: hs_check_blob)."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    info = np.zeros(4, dtype=np.uint64)
    v = f = None
    if faces is not None:
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
        f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    rc = lib().hs_check_blob(_p(blob), blob.nbytes, _p(v), 0 if v is None else len(v), _p(f), 0 if f is None else len(f),
                             _p(info))
    return rc, dict(nodes=int(info[0]), tris=int(info[1]), depth=int(info[2]), children=int(info[3]))


def canonical(blob: np.ndarray) -> np.ndarray:
    """hs_canonical: the blob with nodes numbered breadth-first and records in the order the nodes reference them."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    out = np.empty_like(blob)
    rc = lib().hs_canonical(_p(blob), blob.nbytes, _p(out))
    if rc != 0:
        raise RuntimeError(f"hs_canonical failed: {rc}")
    return out


def blob_prims(blob: np.ndarray, n_tris: int) -> np.ndarray:
    out = np.zeros(n_tris, dtype=np.int32)
    lib().hs_blob_prims(_p(np.ascontiguousarray(blob)), _p(out))
    return out


def tile_map(height: int, width: int, w_log2: int = 3) -> np.ndarray:
    """rt_core.cuh tile_map for every work index of a height x width image (the device's work order of image batches)."""
    out = np.zeros(height * width, np.uint32)
    lib().hs_tile_map(C.c_uint32(height * width), C.c_uint32(width >> w_log2), C.c_uint32(width), C.c_uint32(w_log2), _p(out))
    return out


def frame_check(blob: np.ndarray, origins, directions):
    """(rays rejected by the root-frame test, rejected rays the root node test would still enter [must be 0],
    rays the root node test rejects) - rt_core.cuh frame_missed vs node_test on the root, the code the device runs."""
    o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(directions, dtype=np.float32).reshape(-1, 3)
    out = np.zeros(3, np.uint64)
    rc = lib().hs_frame_check(_p(blob), len(o), _p(o), _p(d), _p(out))
    if rc != 0:
        raise RuntimeError(f"hs_frame_check failed: {rc}")
    return int(out[0]), int(out[1]), int(out[2])


def trace(blob: np.ndarray, mode: str, origins, directions):
    o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(directions, dtype=np.float32).reshape(-1, 3)
    n = len(o)
    m = {"closest": 0, "any": 1, "count": 2}[mode]
    hit = np.zeros(n, np.uint8); front = np.zeros(n, np.uint8); tri = np.zeros(n, np.int32)
    loc = np.zeros((n, 3), np.float32); uv = np.zeros((n, 2), np.float32); count = np.zeros(n, np.int32)
    stats = np.zeros(4, np.uint64); ms = np.zeros(1, np.int32)
    rc = lib().hs_trace(_p(blob), m, n, _p(o), _p(d), _p(hit), _p(front), _p(tri), _p(loc), _p(uv), _p(count),
                        _p(stats), _p(ms))
    if rc != 0:
        raise RuntimeError(f"hs_trace failed: {rc}")
    return dict(hit=hit, front=front, tri=tri, loc=loc, uv=uv, count=count,
                stats=dict(nodes=int(stats[0]), tris=int(stats[1]), rays=int(stats[2]), hits=int(stats[3])),
                max_stack=int(ms[0]))
