"""Meshes of an exact triangle count in every distribution the BVH builder must handle, shared by the CPU tests of the
host builder (test_hostsim_blob_checks.py) and the GPU-against-host builder tests (test_gpu_builder_reference.py).

Every generator is deterministic: mesh(dist, n) -> (float32 vertices [m, 3], int32 faces [n, 3])."""
from __future__ import annotations

import numpy as np

from triro import synth

ONE_TRI = np.array([[0.5, -0.5, 0.25], [0.0, 0.5, 0.25], [-0.5, -0.5, 0.25]], np.float32)


def _soup(n, seed=3, sigma=0.01):
    return synth.triangle_soup(n, sigma=sigma, seed=seed)


def _grid(n, amplitude=0.1):
    """heightfield cut to n triangles (whole rows first)"""
    nx = max(1, int(np.ceil(np.sqrt(n / 2.0))))
    ny = max(1, int(np.ceil(n / (2.0 * nx))))
    v, f = synth.heightfield(nx, ny, amplitude=amplitude)
    return v, np.ascontiguousarray(f[:n])


def _ico(n):
    s = 0
    while 20 * 4 ** s < n:
        s += 1
    v, f = synth.icosphere(s)
    return v, np.ascontiguousarray(f[:n])


def _identical(n):
    """every triangle the same three vertices: all Morton keys equal, equal-key runs cross every tile"""
    return ONE_TRI.copy(), np.zeros((n, 3), np.int32) + np.array([0, 1, 2], np.int32)


def _cluster_far(n):
    """n - 1 triangles in a 1e-3 cube and one 1e3 away: almost every key in one Morton cell"""
    v, f = _soup(n, seed=5, sigma=1e-5)
    v = (v * np.float32(5e-4)).astype(np.float32)
    v[-3:] = ONE_TRI + np.float32(1e3)
    return v, f


def _line(n):
    """small triangles strung along the x axis"""
    c = np.zeros((n, 1, 3), np.float64)
    c[:, 0, 0] = np.linspace(-1.0, 1.0, n) if n > 1 else 0.0
    v = (c + ONE_TRI[None].astype(np.float64) * (0.5 / max(n, 1))).reshape(-1, 3).astype(np.float32)
    return v, np.arange(3 * n, dtype=np.int32).reshape(n, 3)


def _plane(n):
    return _grid(n, amplitude=0.0)


def _scaled(n, scale, offset=0.0):
    v, f = _soup(n, seed=7, sigma=0.02)
    return (v.astype(np.float64) * scale + offset).astype(np.float32), f


def _nan_some(n):
    v, f = _soup(n, seed=9, sigma=0.02)
    rng = np.random.default_rng(9)
    v[rng.random(len(v)) < 0.05, rng.integers(0, 3)] = np.nan
    return v, f


def _nan_all(n):
    v, f = _soup(n, seed=9, sigma=0.02)
    v[:] = np.nan
    return v, f


def _degenerate(n):
    """zero-area triangles (a repeated vertex, three collinear vertices) mixed with duplicated faces"""
    v, f = _soup(n, seed=11, sigma=0.02)
    f = f.copy()
    f[0::4, 2] = f[0::4, 1]                                   # repeated vertex
    v3 = v.reshape(-1, 3, 3)
    v3[1::4, 2] = 2.0 * v3[1::4, 1] - v3[1::4, 0]             # collinear
    f[2::4] = f[(np.arange(n)[2::4] // 2)]                    # duplicates of earlier faces
    return v3.reshape(-1, 3).astype(np.float32), f


def _bad_index(n):
    """some faces name vertices outside [0, n_verts): built through rt_bvh_build directly (the Python layer refuses)"""
    v, f = _soup(n, seed=13, sigma=0.02)
    f = f.copy()
    f[0::5, 0] = -1
    f[1::7, 2] = len(v)
    f[3::11, 1] = 2 ** 31 - 1
    return v, f


DISTRIBUTIONS = {
    "soup": _soup,
    "heightfield": _grid,
    "icosphere": _ico,
    "identical": _identical,
    "cluster_far": _cluster_far,
    "line": _line,
    "plane": _plane,
    "scale_1e-30": lambda n: _scaled(n, 1e-30),
    "scale_1e30": lambda n: _scaled(n, 1e30),
    "offset_3e7": lambda n: _scaled(n, 1.0, 3e7),
    "nan_some": _nan_some,
    "nan_all": _nan_all,
    "degenerate": _degenerate,
    "bad_index": _bad_index,
}


def mesh(dist: str, n: int):
    if dist == "hf_4097x4096":                                # 33 562 624 triangles: 21 bits per axis, 8 sort passes
        assert n == 2 * 4097 * 4096
        return synth.heightfield(4097, 4096)
    v, f = DISTRIBUTIONS[dist](n)
    assert f.shape == (n, 3) and f.dtype == np.int32 and v.dtype == np.float32
    return np.ascontiguousarray(v), np.ascontiguousarray(f)
