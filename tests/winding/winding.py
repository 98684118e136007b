"""Winding-number test infrastructure: ctypes front ends of winding_oracle.c (binary64 brute-force truth) and
windsim.cpp (host simulator of rt_winding.cuh).  TEST INFRASTRUCTURE ONLY: tests, tools and __graft_entry__ import it,
the product never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "trimesh-ray-optix_b200", "csrc")
_ORACLE = None
_SIM = None


def _stale(so, deps):
    return not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps)


def build(force: bool = False) -> tuple[str, str]:
    """Compile libwindoracle.so (gcc + OpenMP) and libwindsim.so (g++) next to this file."""
    so_o = os.path.join(_HERE, "libwindoracle.so")
    src_o = os.path.join(_HERE, "winding_oracle.c")
    if force or _stale(so_o, [src_o]):
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.check_call([cc, "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-o", so_o, src_o, "-lm"])
    so_s = os.path.join(_HERE, "libwindsim.so")
    deps_s = [os.path.join(_HERE, "windsim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                     ("rt_core.cuh", "rt_traverse.cuh", "rt_point.cuh", "rt_winding.cuh")]
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
        lo.wo_winding.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        lo.wo_solid_angle.restype = C.c_double
        lo.wo_solid_angle.argtypes = [C.c_void_p, C.c_void_p]
        ls = C.CDLL(so_s)
        ls.ws_moments.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        ls.ws_n_nodes.restype = C.c_uint32
        ls.ws_n_nodes.argtypes = [C.c_void_p]
        ls.ws_winding.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                                  C.c_void_p]
        ls.ws_moment_check.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        ls.ws_far_field.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        ls.ws_atan2.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        ls.ws_solid_angle.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _ORACLE, _SIM = lo, ls
    return _ORACLE, _SIM


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pts(points) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 3))


def truth(vertices, faces, points) -> np.ndarray:
    """float64 [n]: brute-force winding number in binary64"""
    v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
    f = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    p = _pts(points)
    out = np.zeros(len(p))
    _libs()[0].wo_winding(_p(v), len(v), _p(f), len(f), len(p), _p(p), _p(out))
    return out


def truth_solid_angle(point, tri_vertices) -> float:
    return float(_libs()[0].wo_solid_angle(_p(np.ascontiguousarray(point, dtype=np.float64)),
                                           _p(np.ascontiguousarray(tri_vertices, dtype=np.float64).reshape(9))))


# ------------------------------------------------------------------ host simulator
def n_nodes(blob: np.ndarray) -> int:
    return int(_libs()[1].ws_n_nodes(_p(np.ascontiguousarray(blob))))


def sim_moments(blob: np.ndarray) -> np.ndarray:
    """float32 [n_nodes, 16]: the moment records (px, py, pz, rho, nx, ny, nz, M row-major)"""
    blob = np.ascontiguousarray(blob)
    nn = n_nodes(blob)
    m = np.zeros((nn, 16), np.float32)
    w = np.zeros(nn, np.float32)
    rc = _libs()[1].ws_moments(_p(blob), _p(m), _p(w))
    if rc != 0:
        raise RuntimeError(f"ws_moments failed: {rc}")
    return m


def sim_winding(blob: np.ndarray, points, beta: float = 2.0, moments: np.ndarray | None = None) -> dict:
    """winding numbers (float32), counters and deepest stack of rt_winding.cuh's traversal, with the host moments or
    the given ones"""
    blob = np.ascontiguousarray(blob)
    if moments is None:
        moments = sim_moments(blob)
    moments = np.ascontiguousarray(moments, dtype=np.float32)
    p = _pts(points)
    w = np.zeros(len(p), np.float32)
    stats = np.zeros(4, np.uint64)
    ms = np.zeros(1, np.int32)
    rc = _libs()[1].ws_winding(_p(blob), _p(moments), len(p), _p(p), C.c_float(beta), _p(w), _p(stats), _p(ms))
    if rc != 0:
        raise RuntimeError(f"ws_winding failed: {rc}")
    return dict(w=w, stats=dict(nodes=int(stats[0]), tris=int(stats[1]), points=int(stats[2]), far=int(stats[3])),
                max_stack=int(ms[0]))


def moment_check(blob: np.ndarray, moments: np.ndarray | None = None) -> dict:
    """Every moment record against its node's own triangles in binary64 (ws_moment_check): rho violations and the
    (node, vertex) pairs checked, nodes checked, and the worst relative deviations of rho, p~, N and M."""
    blob = np.ascontiguousarray(blob)
    if moments is None:
        moments = sim_moments(blob)
    out = np.zeros(3, np.uint64)
    worst = np.zeros(4, np.float64)
    rc = _libs()[1].ws_moment_check(_p(blob), _p(np.ascontiguousarray(moments, dtype=np.float32)), _p(out), _p(worst))
    if rc != 0:
        raise RuntimeError(f"ws_moment_check failed: {rc}")
    return dict(rho_violations=int(out[0]), vertices=int(out[1]), nodes=int(out[2]), rho_ratio=float(worst[0]),
                p_err=float(worst[1]), n_err=float(worst[2]), m_err=float(worst[3]))


def sim_far_field(record, points) -> np.ndarray:
    """rt_winding.cuh far_field() of one moment record [16] from every point: 4 pi times the node's approximate w"""
    p = _pts(points)
    out = np.zeros(len(p), np.float32)
    _libs()[1].ws_far_field(_p(np.ascontiguousarray(record, dtype=np.float32).reshape(16)), len(p), _p(p), _p(out))
    return out


def sim_atan2(y, x) -> np.ndarray:
    y = np.ascontiguousarray(y, dtype=np.float32).ravel()
    x = np.ascontiguousarray(x, dtype=np.float32).ravel()
    out = np.zeros(len(y), np.float32)
    _libs()[1].ws_atan2(len(y), _p(y), _p(x), _p(out))
    return out


def sim_solid_angle(points, tri_vertices) -> np.ndarray:
    p = _pts(points)
    out = np.zeros(len(p), np.float32)
    _libs()[1].ws_solid_angle(len(p), _p(p), _p(np.ascontiguousarray(tri_vertices, dtype=np.float32).reshape(9)), _p(out))
    return out
