"""Hit gradient, CPU tier: the host simulator of rt_ray_grad (its own RT_HD code, std::stable_sort in place of the
onesweep sort) against known answers, identities of the formula, a binary64 numpy restatement on every mesh family
and scale, central finite differences of a binary64 ray/triangle intersection, the zero rules, and the documented
summation orders (per ray in row order, per vertex the tree of DESIGN.md §4.9 in row windows).

The hit rows fed to the simulator come from the oracle's binary32 mirror, which the trace kernels reproduce bit for
bit."""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "raygrad"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "distgrad"))
import distgrad as D  # noqa: E402
import raygrad as R  # noqa: E402
from oracle import oracle  # noqa: E402
from test_closest_point_logic import MESHES, bits_equal, sample_points  # noqa: E402
from triro import synth  # noqa: E402

TRI_V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
TRI_F = np.array([[0, 1, 2]], np.int32)


def random_rays(v, n, rng):
    """rays from points around the mesh towards points near its vertices (about half of them hit)"""
    o = sample_points(v, n, rng)[:n].astype(np.float64)
    good = v[np.isfinite(v).all(axis=1)].astype(np.float64)
    diag = float(np.linalg.norm(good.max(0) - good.min(0)))
    tgt = good[rng.integers(0, len(good), len(o))] + rng.normal(0, 0.05 * diag, (len(o), 3))
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o.astype(np.float32), d.astype(np.float32)


def closest_rows(v, f, o, d):
    """(tri [n], hit [n]) of the mirror's closest hit"""
    r = oracle.query(oracle.OracleMesh(v, f), o, d, oracle.MIRROR, want=("hit", "tri"))
    return r["tri"].astype(np.int32), r["hit"].astype(bool)


def test_known_answers():
    o = np.array([[0.2, 0.3, 1.0]], np.float32)
    d = np.array([[0.0, 0.0, -1.0]], np.float32)
    go, gd, gv = R.sim_grad(o, d, [0], [[0, 0, 1]], None, TRI_V, TRI_F)
    assert (go == 0).all() and (gd == 0).all()
    np.testing.assert_allclose(gv, [[0, 0, 0.5], [0, 0, 0.2], [0, 0, 0.3]], atol=1e-7)
    go, gd, gv = R.sim_grad(o, d, [0], [[1, 0, 0]], None, TRI_V, TRI_F)
    assert go.tolist() == [[1, 0, 0]] and gd.tolist() == [[1, 0, 0]] and (gv == 0).all()
    # uv = (w0, b1): d(w0)/d(o_x) = -1, d(b1)/d(o_x) = +1, d(b2)/d(o_y) = +1
    go, gd, gv = R.sim_grad(o, d, [0], None, [[1, 0]], TRI_V, TRI_F)
    assert go.tolist() == [[-1, -1, 0]] and gd.tolist() == [[-1, -1, 0]]
    go, _, _ = R.sim_grad(o, d, [0], None, [[0, 1]], TRI_V, TRI_F)
    assert go.tolist() == [[1, 0, 0]]


@pytest.fixture(scope="module")
def ico_hits():
    v, f = synth.icosphere(3)
    rng = np.random.default_rng(1)
    o, d = random_rays(v, 4000, rng)
    tri, hit = closest_rows(v, f, o, d)
    assert hit.sum() > 1000
    return v, f, o[hit], d[hit], tri[hit], rng


def test_identities_on_random_hits(ico_hits):
    v, f, o, d, tri, rng = ico_hits
    n = len(o)
    gl = rng.normal(size=(n, 3)).astype(np.float32)
    gu = rng.normal(size=(n, 2)).astype(np.float32)
    assert R.sim_rows(o, d, tri, gl, gu, v, f)[4].all()
    # a common translation of the rays and the mesh moves loc by the same amount and leaves uv alone:
    # sum grad_o + sum grad_v = sum g_L
    go, gd, gv = R.sim_grad(o, d, tri, gl, gu, v, f)
    np.testing.assert_allclose(go.sum(0, dtype=np.float64) + gv.sum(0, dtype=np.float64), gl.sum(0, dtype=np.float64),
                               rtol=1e-4, atol=1e-3)
    # lambda is orthogonal to d, so is grad_d
    dots = np.abs((gd.astype(np.float64) * d).sum(1))
    assert (dots <= 1e-5 * (np.linalg.norm(gd, axis=1) + 1)).all()
    # scaling d by 2 halves t and grad_d and leaves the hit, grad_o and grad_v unchanged (powers of 2 are exact)
    go2, gd2, gv2 = R.sim_grad(o, 2 * d, tri, gl, gu, v, f)
    bits_equal(go2, go, "grad_o with 2d")
    bits_equal(gd2, gd / 2, "grad_d with 2d")
    bits_equal(gv2, gv, "grad_v with 2d")


def conditioning(o, d, tri, v, f):
    """per row |e1| |e2| |d| / |det| (binary64): how much the recomputed hit amplifies rounding"""
    ro, rd, v0, v1, v2, _, _, _ = R._rows(o, d, tri, v, f, None)
    e1, e2 = v1 - v0, v2 - v0
    det = (e1 * np.cross(rd, e2)).sum(1)
    with np.errstate(all="ignore"):
        return np.linalg.norm(e1, axis=1) * np.linalg.norm(e2, axis=1) * np.linalg.norm(rd, axis=1) / np.abs(det)


@pytest.mark.parametrize("name", list(MESHES))
def test_hostsim_matches_binary64_reference(name):
    v, f = MESHES[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    o, d = random_rays(v, 3000, rng)
    tri, hit = closest_rows(v, f, o, d)
    kappa = conditioning(o, d, tri, v, f)
    keep = hit & (kappa < 100)              # grazing hits amplify float32 rounding without bound: compared elsewhere
    assert keep.sum() > 100, keep.sum()
    tri = np.where(keep, tri, -1).astype(np.int32)
    n = len(o)
    gl = rng.normal(size=(n, 3)).astype(np.float32)
    gu = rng.normal(size=(n, 2)).astype(np.float32)
    go, gd, gv = R.sim_grad(o, d, tri, gl, gu, v, f)
    ro, rd, rv = R.reference(o, d, tri, gl, gu, v, f)
    assert np.isfinite(go).all() and np.isfinite(gd).all() and np.isfinite(gv).all()
    # bound of each row's terms, times kappa and a few dozen roundings
    _, rdd, v0, v1, v2, fi, _, ok = R._rows(o, d, tri, v, f, None)
    e1, e2 = v1 - v0, v2 - v0
    t, b1, b2, det, p, _, _ = R.hit64(R._rows(o, d, tri, v, f, None)[0], rdd, v0, v1, v2)
    with np.errstate(all="ignore"):
        mag = (np.abs(gl).sum(1) * (np.linalg.norm(e1, axis=1) + np.linalg.norm(e2, axis=1)) + 2 * np.abs(gu).sum(1)) \
            * (np.linalg.norm(p, axis=1) + np.linalg.norm(np.cross(e1, rdd), axis=1)) / np.abs(det)
    mag = np.where(keep, mag, 0)
    tol = 1e-5 * np.where(keep, kappa, 0) * mag
    assert (np.abs(go - ro).max(1) <= tol + 1e-30).all()
    assert (np.abs(gd - rd).max(1) <= tol * (1 + np.abs(np.where(keep, t, 0))) + 1e-30).all()
    vm = np.zeros(len(v))
    for k in range(3):
        np.add.at(vm, fi[keep, k], (tol + 1e-6 * (mag + np.abs(gl).sum(1)))[keep] * 2)
    assert (np.abs(gv - rv).max(1) <= vm).all()


def test_finite_differences_of_the_binary64_intersection():
    v, f = synth.icosphere(1)
    rng = np.random.default_rng(11)
    n = 600
    # rays from outside towards interior points of random faces: barycentrics >= 0.1, far from every edge
    tri = rng.integers(0, len(f), n).astype(np.int32)
    bc = rng.dirichlet([4, 4, 4], n)
    bc = bc[(bc > 0.1).all(1)]
    tri = tri[:len(bc)]
    tgt = (bc[:, :, None] * v[f[tri]].astype(np.float64)).sum(1)
    o = (tgt * rng.uniform(2, 3, (len(bc), 1)) + rng.normal(0, 0.2, (len(bc), 3))).astype(np.float32)
    d = (tgt - o) * rng.uniform(0.5, 2, (len(bc), 1))
    d = d.astype(np.float32)
    got, hit = closest_rows(v, f, o, d)
    keep = hit & (got == tri)
    o, d, tri = o[keep], d[keep], tri[keep]
    assert len(o) > 300
    gl = rng.normal(size=(len(o), 3)).astype(np.float32)
    gu = rng.normal(size=(len(o), 2)).astype(np.float32)
    go, gd, gv = R.sim_grad(o, d, tri, gl, gu, v, f)

    def loss(oo, dd, vv):
        loc, uv = R.locate64(oo, dd, tri, vv, f)
        return (gl * loc).sum(1) + (gu * uv).sum(1)

    h = 1e-4
    o64, d64, v64 = o.astype(np.float64), d.astype(np.float64), v.astype(np.float64)
    for a in range(3):
        e = np.zeros(3); e[a] = h
        fd_o = (loss(o64 + e, d64, v64) - loss(o64 - e, d64, v64)) / (2 * h)
        fd_d = (loss(o64, d64 + e, v64) - loss(o64, d64 - e, v64)) / (2 * h)
        assert (np.abs(go[:, a] - fd_o) <= 2e-4 * (1 + np.abs(fd_o))).all(), a
        assert (np.abs(gd[:, a] - fd_d) <= 2e-4 * (1 + np.abs(fd_d))).all(), a
    for j in range(len(v)):
        for a in range(3):
            hi, lo = v64.copy(), v64.copy()
            hi[j, a] += h; lo[j, a] -= h
            fd = (loss(o64, d64, hi).sum() - loss(o64, d64, lo).sum()) / (2 * h)
            assert abs(gv[j, a] - fd) <= 1e-3 * max(1.0, abs(fd)), (j, a, gv[j, a], fd)


def test_degenerate_rows_give_exact_zeros():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [np.nan, 0, 0], [2, 0, 0]], np.float32)
    f = np.array([[0, 1, 2], [0, 1, 3], [0, 1, 7], [0, 1, 4]], np.int32)
    o = np.array([[0.2, 0.3, 1.0]] * 6 + [[-1, 0.3, 0]], np.float32)
    d = np.array([[0, 0, -1.0]] * 6 + [[1, 0, 0]], np.float32)
    # tri -1, NaN vertex, vertex index out of range, tri out of range, zero-area triangle (det 0), ray in the plane
    tri = np.array([-1, 1, 2, 4, 3, 0, 0], np.int32)
    tri_in_plane = tri.copy()
    gl = np.ones((7, 3), np.float32)
    gu = np.ones((7, 2), np.float32)
    go, gd, gv = R.sim_grad(o, d, tri, gl, gu, v, f)
    live = np.zeros(7, bool); live[5] = True
    for g in (go, gd):
        assert (g[~live] == 0).all() and not np.signbit(g[~live]).any()
    # only row 5 reaches the vertices
    _, _, gv5 = R.sim_grad(o[5:6], d[5:6], tri_in_plane[5:6], gl[5:6], gu[5:6], v, f)
    bits_equal(gv, gv5, "grad_v of the degenerate batch")
    assert not np.signbit(gv[3:]).any() and (gv[3:] == 0).all()
    # a row_ray outside the batch, and a non-finite incoming gradient, contribute nothing either
    go, gd, gv = R.sim_grad(o[:1], d[:1], [0, 0], [[1, 2, 3], [4, 5, 6]], None, v, f, row_ray=[-1, 1])
    assert (go == 0).all() and (gd == 0).all() and (gv == 0).all()
    go, gd, gv = R.sim_grad(o[:1], d[:1], [0], [[np.inf, 0, 0]], None, v, f)
    assert (go == 0).all() and (gd == 0).all() and (gv == 0).all()
    ro, rd, rv = R.reference(o, d, tri, gl, gu, v, f)
    assert (ro[~live] == 0).all() and (rv[3:] == 0).all()


def test_per_ray_sums_run_in_row_order():
    v, f = synth.icosphere(2)
    rng = np.random.default_rng(4)
    n_rays = 50
    o, d = random_rays(v, n_rays * 4, rng)
    o, d = o[:n_rays], d[:n_rays]
    # 0 to 64 rows per ray, non-decreasing ray index, on random triangles (the formula does not re-test the hit)
    counts = rng.integers(0, 65, n_rays)
    counts[3] = 0
    row_ray = np.repeat(np.arange(n_rays), counts).astype(np.int32)
    h = len(row_ray)
    tri = rng.integers(0, len(f), h).astype(np.int32)
    gl = rng.normal(size=(h, 3)).astype(np.float32)
    go, gd, gv = R.sim_grad(o, d, tri, gl, None, v, f, row_ray=row_ray)
    lam, tlam, _, _, _ = R.sim_rows(o, d, tri, gl, None, v, f, row_ray=row_ray)
    want_o = np.zeros((n_rays, 3), np.float32)
    want_d = np.zeros((n_rays, 3), np.float32)
    for j in range(h):
        want_o[row_ray[j]] = (want_o[row_ray[j]] + lam[j]).astype(np.float32)
        want_d[row_ray[j]] = (want_d[row_ray[j]] + tlam[j]).astype(np.float32)
    bits_equal(go, want_o, "grad_o")
    bits_equal(gd, want_d, "grad_d")
    assert (go[counts == 0] == 0).all()


@pytest.mark.parametrize("window", [0, 1000, 777, 1])
def test_vertex_sums_are_the_documented_tree(window):
    v, f = synth.icosphere(2)
    rng = np.random.default_rng(window + 1)
    n = 3000 if window != 1 else 300
    o, d = random_rays(v, n, rng)
    tri, hit = closest_rows(v, f, o, d)
    # many rows on a few triangles: runs of thousands of pairs, three levels of the tree
    tri = np.where(rng.random(len(o)) < 0.5, rng.integers(0, 4, len(o)), tri).astype(np.int32)
    gl = rng.normal(size=(len(o), 3)).astype(np.float32)
    gu = rng.normal(size=(len(o), 2)).astype(np.float32)
    _, _, gv = R.sim_grad(o, d, tri, gl, gu, v, f, window=window)
    _, _, q, w, live = R.sim_rows(o, d, tri, gl, gu, v, f)
    bits_equal(gv, D.documented_order(q, w, live, tri, f, len(v), window), f"window {window}")


def test_workspace_sizes_and_argument_checks():
    import ctypes as C

    from triro.backend import ops as hops

    lib = hops.get_module()
    per_row = (hops.ray_grad_workspace_bytes(8_000_000, 1000) - hops.ray_grad_workspace_bytes(4_000_000, 1000)) / 4e6
    assert 100 < per_row < 110                     # DESIGN §4.10: about 105 B per row
    assert hops.ray_grad_workspace_bytes(1000, 10_000) - hops.ray_grad_workspace_bytes(1000, 0) == 40_192   # 4 B per vertex
    assert hops.ray_grad_workspace_bytes(10**10, 5) == hops.ray_grad_workspace_bytes((1 << 30) // 3, 5)
    # the exact layouts (DESIGN §4.9, §4.10, §4.13): (n_rows, n_verts) -> (distance, ray) bytes
    for (n, nv), (dist, ray) in {(1, 0): (19456, 19712), (1000, 10000): (148736, 156928), (7777, 642): (773376, 835840),
                                 (10_000_000, 163842): (975670784, 1055670784),
                                 (10**10, 5): (34896617984, 37759929600)}.items():
        assert hops.distance_grad_workspace_bytes(n, nv) == dist, (n, nv)
        assert hops.ray_grad_workspace_bytes(n, nv) == ray, (n, nv)
    for args, want in {(1, 1, 3, 1): 19968, (1, 1, 3, 2): 19968, (1, 1, 3, 3): 19968,
                       (2_073_600, 1000, 10242, 1): 327865344, (2_073_600, 1000, 10242, 3): 505160192,
                       (1_000_000, 64, 163842, 2): 132140032, (10**10, 7, 9, 3): 37350885632}.items():
        assert hops.scene_grad_workspace_bytes(*args) == want, args
    wb = C.c_size_t()
    assert lib.rt_ray_grad_sizes(-1, 3, C.byref(wb)) != 0
    assert lib.rt_ray_grad_sizes(3, 1 << 32, C.byref(wb)) != 0
    rd = hops.RayDesc()
    rd.nray = 4
    for i, s in enumerate((1, 1, 4, 3)):
        rd.shape[i] = s
    # without row_ray there must be one row per ray; a null descriptor and a bad window are rejected
    assert lib.rt_ray_grad(C.byref(rd), None, 3, None, None, None, None, None, 3, None, 1, None, None, None, None, 0,
                           None) == -1
    assert lib.rt_ray_grad(None, None, 4, None, None, None, None, None, 3, None, 1, None, None, None, None, 0, None) == -1
    opts = hops.trace_opts(None, 2, 3)
    assert lib.rt_ray_grad(C.byref(rd), C.byref(opts), 3, None, None, None, None, None, 3, None, 1, None, None, None,
                           None, 0, None) == -1
    # no rows (every ray missed): accepted with any row_ray, NULL included, as an empty ray_idx tensor passes it
    assert lib.rt_ray_grad(C.byref(rd), None, 0, None, None, None, None, None, 3, None, 1, None, None, None, None, 0,
                           None) == 0
    # nothing to do: no rows, or no output, succeeds without touching memory
    assert lib.rt_ray_grad(C.byref(rd), None, 4, None, None, None, None, None, 3, None, 1, None, None, None, None, 0,
                           None) == 0
