"""Closest-point query, CPU tier: oracle known answers, MIRROR vs TRUTH, the host simulator of rt_point.cuh (the
kernel's own RT_HD code) against the brute-force MIRROR oracle bit for bit, and the lower bounds of the BVH8 slots."""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import hostsim  # noqa: E402
import pointquery as pq  # noqa: E402
from triro import synth  # noqa: E402

TRI = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)


def bits_equal(a, b, what):
    a = np.ascontiguousarray(a, dtype=np.float32); b = np.ascontiguousarray(b, dtype=np.float32)
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ (first at {np.argwhere(bad)[0]})"


def one(points, v=TRI, f=((0, 1, 2),), mode=pq.MIRROR, max_distance=float("inf")):
    o = pq.PointOracleIntersector(v, np.asarray(f, np.int32), mode=mode, use_bvh=False)
    return o.closest_point(np.asarray(points, np.float32), max_distance)


@pytest.mark.parametrize("mode", [pq.MIRROR, pq.TRUTH])
def test_known_answers_voronoi_regions(mode):
    pts = [[0.25, 0.25, 2.0],     # face
           [0.5, -1.0, 0.0],      # edge v0-v1
           [-1.0, 0.5, 0.0],      # edge v0-v2
           [1.0, 1.0, 0.5],       # edge v1-v2
           [-1.0, -1.0, 0.0],     # vertex v0
           [2.0, -0.5, 0.0],      # vertex v1
           [-0.5, 2.0, 0.0],      # vertex v2
           [0.2, 0.3, 0.0]]       # on the triangle
    c, d, t, uv = one(pts, mode=mode)
    want_c = [[0.25, 0.25, 0], [0.5, 0, 0], [0, 0.5, 0], [0.5, 0.5, 0], [0, 0, 0], [1, 0, 0], [0, 1, 0], [0.2, 0.3, 0]]
    want_d = [2.0, 1.0, 1.0, np.sqrt(0.5 + 0.25), np.sqrt(2.0), np.sqrt(1.25), np.sqrt(1.25), 0.0]
    want_uv = [[0.5, 0.25], [0.5, 0.5], [0.5, 0.0], [0.0, 0.5], [1, 0], [0, 1], [0, 0], [0.5, 0.2]]
    assert t.tolist() == [0] * 8
    np.testing.assert_allclose(c, want_c, atol=1e-7)
    np.testing.assert_allclose(d, want_d, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(uv, want_uv, atol=1e-6)
    assert d[7] == 0.0


def test_zero_area_and_collinear_triangles():
    v = np.array([[0, 0, 0], [0, 0, 0], [1, 0, 0],       # two equal vertices: a segment
                  [2, 2, 2], [2, 2, 2], [2, 2, 2],       # one point
                  [0, 3, 0], [1, 3, 0], [2, 3, 0]], np.float32)   # collinear
    for mode in (pq.MIRROR, pq.TRUTH):
        c, d, t, uv = one([[0.5, 1.0, 0.0]], v, [[0, 1, 2]], mode)
        np.testing.assert_allclose(c[0], [0.5, 0, 0], atol=1e-7); assert d[0] == 1.0
        c, d, t, uv = one([[2.0, 2.0, 3.0]], v, [[3, 4, 5]], mode)
        np.testing.assert_allclose(c[0], [2, 2, 2]); assert d[0] == 1.0
        c, d, t, uv = one([[1.5, 4.0, 0.0], [5.0, 3.0, 0.0]], v, [[6, 7, 8]], mode)
        np.testing.assert_allclose(c, [[1.5, 3, 0], [2, 3, 0]], atol=1e-7)
        np.testing.assert_allclose(d, [1.0, 3.0])
        assert np.isfinite(uv).all()
    # the product's own point_tri agrees with the mirror on these
    for p, tri in (([0.5, 1.0, 0.0], v[0:3]), ([2.0, 2.0, 3.0], v[3:6]), ([1.5, 4.0, 0.0], v[6:9])):
        r = pq.sim_point_tri(p, tri)
        m = pq.query(pq.PointMesh(tri, [[0, 1, 2]], use_bvh=False), [p], pq.MIRROR)
        bits_equal(r[:3], m["closest"][0], "closest"); bits_equal(r[3:4], m["d2"], "d2"); bits_equal(r[4:], m["uv"][0], "uv")


def test_nan_triangle_is_never_selected():
    v = np.array([[np.nan, 0, 0], [0, 1, 0], [1, 0, 0], [0, 0, 5], [1, 0, 5], [0, 1, 5]], np.float32)
    f = [[0, 1, 2], [3, 4, 5]]
    for mode in (pq.MIRROR, pq.TRUTH):
        c, d, t, uv = one([[0.1, 0.1, 0.0], [0.1, 0.1, 10.0]], v, f, mode)
        assert t.tolist() == [1, 1]
        np.testing.assert_allclose(d, [5.0, 5.0])
    blob = hostsim.build_blob(v, f)
    s = pq.sim_closest_point(blob, [[0.1, 0.1, 0.0], [0.1, 0.1, 10.0]])
    assert s["tri"].tolist() == [1, 1]


def test_max_distance_boundary():
    p = [[0.25, 0.25, 2.0]]
    for mode in (pq.MIRROR, pq.TRUTH):
        _, d, t, _ = one(p, mode=mode, max_distance=2.0)
        assert t.tolist() == [0] and d[0] == 2.0
        c, d, t, uv = one(p, mode=mode, max_distance=np.nextafter(np.float32(2.0), np.float32(0)))
        assert t.tolist() == [-1] and d[0] == np.inf and not c.any() and not uv.any()
    blob = hostsim.build_blob(TRI, [[0, 1, 2]])
    assert pq.sim_closest_point(blob, p, 2.0)["tri"].tolist() == [0]
    below = float(np.nextafter(np.float32(2.0), np.float32(0)))
    s = pq.sim_closest_point(blob, p, below)
    assert s["tri"].tolist() == [-1] and s["distance"][0] == np.inf


def test_non_finite_points_and_empty_mesh():
    blob = hostsim.build_blob(TRI, [[0, 1, 2]])
    p = [[np.nan, 0, 0], [np.inf, 0, 0], [0, 0, 1]]
    s = pq.sim_closest_point(blob, p)
    assert s["tri"].tolist() == [-1, -1, 0]
    r = pq.query(pq.PointMesh(TRI, [[0, 1, 2]], use_bvh=False), p, pq.MIRROR)
    assert r["tri"].tolist() == [-1, -1, 0]
    empty = hostsim.build_blob(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    s = pq.sim_closest_point(empty, [[0, 0, 0]])
    assert s["tri"].tolist() == [-1] and s["distance"][0] == np.inf


def box_distance(p, h):
    q = np.abs(p.astype(np.float64)) - h
    outside = np.linalg.norm(np.maximum(q, 0.0), axis=1)
    inside = np.minimum(np.max(q, axis=1), 0.0)
    return outside + inside   # signed: negative inside


def test_cube_closed_form_and_signed_distance():
    v, f = synth.cube(0.5)
    rng = np.random.default_rng(3)
    p = rng.uniform(-1.5, 1.5, (400, 3)).astype(np.float32)
    o = pq.PointOracleIntersector(v, f, mode=pq.MIRROR)
    _, d, _, _ = o.closest_point(p)
    sd_box = box_distance(p, 0.5)
    np.testing.assert_allclose(d, np.abs(sd_box), rtol=1e-6, atol=1e-7)
    sd = o.signed_distance(p)
    clear = np.abs(sd_box) > 1e-4
    np.testing.assert_allclose(sd[clear], -sd_box[clear], rtol=1e-6, atol=1e-7)   # trimesh: positive inside


def test_mirror_matches_truth():
    rng = np.random.default_rng(11)
    for v, f in (synth.icosphere(3), synth.triangle_soup(2000), synth.heightfield(16, 16)):
        m = pq.PointMesh(v, f, use_bvh=False)
        p = rng.uniform(v.min(0) - 0.3, v.max(0) + 0.3, (300, 3)).astype(np.float32)
        mir = pq.query(m, p, pq.MIRROR)
        tru = pq.query(m, p, pq.TRUTH)
        np.testing.assert_allclose(mir["distance"], tru["distance"], rtol=1e-6, atol=1e-7)
        # the mirror's choice is (within tolerance) a binary64 minimiser
        all_t = pq.all_d2(m, p, pq.TRUTH)
        chosen = all_t[np.arange(len(p)), mir["tri"]]
        assert np.all(chosen <= tru["d2"] * (1 + 4e-6) + 1e-12)


def meshes():
    out = {
        "ico3": synth.icosphere(3),
        "ico5": synth.icosphere(5),
        "soup20k": synth.triangle_soup(20000, seed=5),
        "hf64": synth.heightfield(64, 64),
    }
    # degenerate mix: zero-area, collinear, NaN, duplicated and ordinary triangles
    v, f = synth.icosphere(2)
    extra_v = np.array([[0, 0, 0], [0, 0, 0], [0.5, 0, 0], [0.1, 0.1, 0.1], [0.2, 0.2, 0.2], [0.3, 0.3, 0.3],
                        [np.nan, 0, 0], [0, 0.5, 0], [0, 0, 0.5]], np.float32)
    ev = np.concatenate([v, extra_v])
    n = len(v)
    ef = np.concatenate([f, f[:40], np.arange(n, n + 9, dtype=np.int32).reshape(3, 3)])
    out["degenerate"] = (ev, ef.astype(np.int32))
    ico, icf = synth.icosphere(4)
    for s, off in ((1e6, 0.0), (1e-6, 0.0), (1e4, 3e7)):
        out[f"ico4_s{s:g}_o{off:g}"] = ((ico.astype(np.float64) * s + off).astype(np.float32), icf)
    return out


MESHES = meshes()


def sample_points(v, n, rng):
    good = v[np.isfinite(v).all(axis=1)]
    lo, hi = good.min(0).astype(np.float64), good.max(0).astype(np.float64)
    diag = float(np.linalg.norm(hi - lo))
    c = 0.5 * (lo + hi)
    uni = rng.uniform(c - 0.6 * (hi - lo), c + 0.6 * (hi - lo), (n, 3))
    near = good[rng.integers(0, len(good), n)].astype(np.float64) + rng.normal(0.0, 0.01 * diag, (n, 3))
    verts = good[rng.integers(0, len(good), n // 4)]          # exactly at vertices: ties between incident triangles
    return np.concatenate([uni.astype(np.float32), near.astype(np.float32), verts])


@pytest.mark.parametrize("name", list(MESHES))
def test_hostsim_matches_mirror_bit_for_bit(name):
    v, f = MESHES[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    p = sample_points(v, 1500, rng)
    blob = hostsim.build_blob(v, f)
    s = pq.sim_closest_point(blob, p)
    m = pq.PointMesh(v, f)
    brute = pq.query(m, p, pq.MIRROR, brute=True)
    assert np.array_equal(s["tri"], brute["tri"]), f"{int((s['tri'] != brute['tri']).sum())} triangle ids differ"
    for k in ("closest", "distance", "uv"):
        bits_equal(s[k], brute[k], k)
    assert (s["tri"] >= 0).all()
    assert s["max_stack"] <= 60
    bvh = pq.query(m, p, pq.MIRROR)                 # the oracle's own BVH gives the brute-force answer
    assert np.array_equal(bvh["tri"], brute["tri"])
    bits_equal(bvh["distance"], brute["distance"], "oracle bvh distance")
    # with a max_distance that cuts through the batch
    md = float(np.median(brute["distance"]))
    s2 = pq.sim_closest_point(blob, p, md)
    b2 = pq.query(m, p, pq.MIRROR, max_distance=md)
    assert np.array_equal(s2["tri"], b2["tri"])
    bits_equal(s2["distance"], b2["distance"], "distance within max_distance")
    assert ((b2["tri"] >= 0) == (brute["d2"] <= np.float32(md) * np.float32(md))).all()


@pytest.mark.parametrize("name", list(MESHES))
def test_slot_lower_bounds_never_exceed_d2(name):
    v, f = MESHES[name]
    rng = np.random.default_rng(7)
    p = sample_points(v, 160, rng)
    blob = hostsim.build_blob(v, f)
    violations, checked, worst = pq.slot_bounds_check(blob, p)
    assert checked > 0
    assert violations == 0, f"{violations} of {checked} slot bounds exceed a triangle's d2 (worst ratio {worst})"
    assert worst <= 1.0
