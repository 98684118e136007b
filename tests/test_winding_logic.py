"""Generalized winding number, CPU tier: known answers, the own atan2 against binary64, the host simulator of
rt_winding.cuh (the kernel's own RT_HD code) against the binary64 brute-force oracle in exact mode and with beta = 2,
every moment record (radius bound, centroid, N, M) checked exhaustively in binary64, and the order of convergence of
the two-term far field.

Tolerances (DESIGN.md §4.7) were measured with this simulator, which runs the kernel's arithmetic; they are asserted
only for points farther than DELTA times the bounding-box diagonal from the surface.  The solid angle jumps by 4 pi
across a triangle, so nearer points measure the closeness of the point to the surface more than the arithmetic."""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "winding"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import builder_cases  # noqa: E402
import deep_overlap_cases as doc  # noqa: E402
import hostsim  # noqa: E402
import pointquery as pq  # noqa: E402
import winding as W  # noqa: E402
from test_closest_point_logic import MESHES, sample_points  # noqa: E402
from triro import synth  # noqa: E402

INF = float("inf")
DELTA = 0.01
# |w - truth| at beta = inf and at beta = 2, per mesh: about 1.5x what the simulator gives on these samples, so that a
# change to the far-field term or to the moments shows.  The icospheres' beta = 2 error is the truncation of the
# two-term expansion for points inside a sphere looking at caps (DESIGN.md §4.7); dup600, shells32 and stack300 sum
# hundreds of large terms of both signs or sit close to many surfaces.
TOL = {"ico3": (4e-6, 0.08), "ico5": (1.5e-5, 0.08), "soup20k": (1e-7, 2e-4), "hf64": (5e-6, 0.035),
       "degenerate": (2e-6, 0.09), "ico4_s1e+06_o0": (8e-6, 0.08), "ico4_s1e-06_o0": (8e-6, 0.08),
       "ico4_s10000_o3e+07": (8e-6, 0.08), "shells32": (2.5e-4, 0.4), "dup600": (1.6e-3, 1.6e-3),
       "book96": (2e-6, 3.5e-3), "stack300": (5e-5, 0.15), "cube_open": (1e-6, 1e-6), "heightfield_open": (3e-6, 0.035),
       "ico3_reversed": (4e-6, 0.08), "builder_nan_some": (2e-7, 2e-3), "builder_degenerate": (3e-7, 2e-3)}
TOL_FAST_ICO = 0.08
TRI = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)


def winding_meshes():
    out = dict(MESHES)
    for name in ("shells32", "dup600", "book96", "stack300"):
        out[name] = doc.scene(name)
    v, f = synth.cube(0.5)
    out["cube_open"] = (v, np.ascontiguousarray(f[2:]))          # the bottom face removed
    out["heightfield_open"] = synth.heightfield(48, 32)
    v, f = synth.icosphere(3)
    out["ico3_reversed"] = (v, np.ascontiguousarray(f[:, ::-1]))
    for dist in ("nan_some", "degenerate"):
        out["builder_" + dist] = builder_cases.mesh(dist, 3000)
    return out


WMESHES = winding_meshes()


def surface_distance(v, f, p):
    return pq.query(pq.PointMesh(v, f), p, pq.TRUTH)["distance"]


def diagonal(v):
    good = v[np.isfinite(v).all(axis=1)].astype(np.float64)
    return float(np.linalg.norm(good.max(0) - good.min(0)))


# ------------------------------------------------------------------ known answers
def test_equilateral_triangle_axis_closed_form():
    R = 1.0
    th = np.array([0.0, 2 * np.pi / 3, 4 * np.pi / 3])
    tri = np.stack([R * np.cos(th), R * np.sin(th), np.zeros(3)], 1).astype(np.float32)   # CCW seen from +z
    R2 = float((tri[0, :2].astype(np.float64) ** 2).sum())
    hs = np.array([1e-3, 0.1, 0.5, 1.0, 3.0, 30.0, 1e3])
    for sgn in (1.0, -1.0):
        q = np.stack([np.zeros_like(hs), np.zeros_like(hs), sgn * hs], 1).astype(np.float32)
        h = q[:, 2].astype(np.float64)
        L = np.sqrt(R2 + h * h)
        area2 = 3.0 * np.sqrt(3.0) / 2.0 * R2                   # twice the triangle's area
        det = -h * area2                                        # [a b c] with a = v0 - q etc.
        den = L ** 3 + 3.0 * (h * h - R2 / 2.0) * L
        want = 2.0 * np.arctan2(det, den)
        got = W.sim_solid_angle(q, tri).astype(np.float64)
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-7)
        for i in range(len(q)):
            assert abs(W.truth_solid_angle(q[i], tri) - want[i]) <= 1e-7 * max(1.0, abs(want[i]))   # float32 vertices
    # above the outward side of a CCW triangle the solid angle is negative, approaching -2 pi
    assert W.sim_solid_angle([[0, 0, 1e-4]], tri)[0] < -6.28


def test_closed_cube_from_centre_is_one():
    v, f = synth.cube(0.5)
    blob = hostsim.build_blob(v, f)
    p = np.array([[0, 0, 0], [0.1, -0.2, 0.3], [2, 0, 0]], np.float32)
    for beta in (INF, 2.0):
        w = W.sim_winding(blob, p, beta)["w"]
        np.testing.assert_allclose(w, [1, 1, 0], atol=1e-6)
    np.testing.assert_allclose(W.truth(v, f, p), [1, 1, 0], atol=1e-12)


def test_in_plane_on_triangle_and_at_vertex_give_zero():
    pts = np.array([[2, 3, 0], [-1, 0.5, 0], [0.2, 0.3, 0], [0.5, 0, 0], [0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    assert (W.sim_solid_angle(pts, TRI) == 0.0).all()
    assert (W.truth(TRI, [[0, 1, 2]], pts) == 0.0).all()
    blob = hostsim.build_blob(TRI, [[0, 1, 2]])
    w = W.sim_winding(blob, pts, INF)["w"]
    assert (w == 0.0).all() and not np.signbit(w).any()
    # zero-area triangles: a repeated vertex and three collinear vertices
    for tri in (np.array([[0, 0, 0], [0, 0, 0], [1, 0, 0]], np.float32), np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2]], np.float32)):
        q = np.array([[0.3, 0.7, 0.2], [5, -1, 2]], np.float32)
        assert (W.sim_solid_angle(q, tri) == 0.0).all() and (W.truth(tri, [[0, 1, 2]], q) == 0.0).all()


def test_non_finite_vertices_points_and_empty_mesh():
    v = np.array([[np.nan, 0, 0], [0, 1, 0], [1, 0, 0], [0, 0, 5], [1, 0, 5], [0, 1, 5], [np.inf, 0, 1]], np.float32)
    f = np.array([[0, 1, 2], [3, 4, 5], [6, 1, 2]], np.int32)
    p = np.array([[0.2, 0.2, 0.0], [0.2, 0.2, 6.0], [0.3, 0.1, 2.0]], np.float32)
    blob = hostsim.build_blob(v, f)
    alone = hostsim.build_blob(v[3:6], [[0, 1, 2]])
    for beta in (INF, 2.0):
        assert np.array_equal(W.sim_winding(blob, p, beta)["w"], W.sim_winding(alone, p, beta)["w"])
    np.testing.assert_array_equal(W.truth(v, f, p), W.truth(v[3:6], [[0, 1, 2]], p))
    q = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.1, 0.1, 1.0]], np.float32)
    w = W.sim_winding(alone, q, 2.0)["w"]
    assert np.isnan(w[:3]).all() and np.isfinite(w[3])
    assert np.isnan(W.truth(v[3:6], [[0, 1, 2]], q)[:3]).all()
    empty = hostsim.build_blob(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    for beta in (INF, 2.0):
        w = W.sim_winding(empty, [[0, 0, 0], [1, 2, 3]], beta)["w"]
        assert (w == 0.0).all() and not np.signbit(w).any()
    assert (W.truth(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), [[0, 0, 0]]) == 0.0).all()


# ------------------------------------------------------------------ atan2
def atan2_sweep():
    rng = np.random.default_rng(0)
    n = 200_000
    ang = rng.uniform(-np.pi, np.pi, n)
    mag = 2.0 ** rng.uniform(-30, 30, n)
    ratio = 2.0 ** rng.uniform(-40, 40, n)
    s1, s2 = np.where(rng.random(n) < 0.5, -1.0, 1.0), np.where(rng.random(n) < 0.5, -1.0, 1.0)
    y = np.concatenate([mag * np.sin(ang), s1 * mag * ratio, s2 * mag])
    x = np.concatenate([mag * np.cos(ang), s2 * mag, s1 * mag * ratio])
    edge = np.array([[0, 1], [0, -1], [1, 0], [-1, 0], [1, 1], [-1, -1], [1, -1], [-1, 1], [1e-30, -1], [-1e-30, -1],
                     [3, 1e-38], [1e38, 1e-38], [0.41421356, 1], [0.41421357, 1]], np.float64)
    y = np.concatenate([y, edge[:, 0]]).astype(np.float32)
    x = np.concatenate([x, edge[:, 1]]).astype(np.float32)
    return y, x


def test_atan2_against_binary64():
    y, x = atan2_sweep()
    got = W.sim_atan2(y, x).astype(np.float64)
    want = np.arctan2(y.astype(np.float64), x.astype(np.float64))
    err = np.abs(got - want)
    assert err.max() <= 3e-7, f"absolute error {err.max():.3g}"
    assert (err <= 2.5e-7 * np.abs(want)).all(), f"relative error {(err / np.maximum(np.abs(want), 1e-300)).max():.3g}"
    # every quadrant and both octants of each were swept
    q = (y >= 0).astype(int) * 2 + (x >= 0) + 4 * (np.abs(y) > np.abs(x))
    assert len(np.unique(q)) == 8
    zeros = np.array([0.0, -0.0, 0.0, -0.0], np.float32)
    assert (W.sim_atan2(zeros, zeros[::-1]) == 0.0).all()
    # the sign follows y's sign bit, as atan2's does: +-0 against a negative x is +-pi
    got = W.sim_atan2(np.array([0.0, -0.0], np.float32), np.array([-1.0, -1.0], np.float32))
    assert got[0] == np.float32(np.pi) and got[1] == -np.float32(np.pi)


# ------------------------------------------------------------------ simulator against the truth oracle
def check_mesh(name, v, f, n):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    p = sample_points(v, n, rng)
    blob = hostsim.build_blob(v, f)
    truth = W.truth(v, f, p)
    clear = surface_distance(v, f, p) > DELTA * diagonal(v)
    assert clear.sum() >= n // 4
    tol_exact, tol_fast = TOL[name]
    exact = W.sim_winding(blob, p, INF)
    fast = W.sim_winding(blob, p, 2.0)
    e_exact = np.abs(exact["w"] - truth)[clear]
    e_fast = np.abs(fast["w"] - truth)[clear]
    assert e_exact.max() <= tol_exact, f"{name}: exact |dw| {e_exact.max():.3g}"
    assert e_fast.max() <= tol_fast, f"{name}: beta 2 |dw| {e_fast.max():.3g}"
    assert exact["stats"]["far"] == 0 and exact["stats"]["tris"] == len(p) * len(f)   # exact mode sums every triangle
    assert fast["stats"]["points"] == len(p) and exact["max_stack"] <= 60
    return p, truth, exact, fast


@pytest.mark.parametrize("name", list(WMESHES))
def test_hostsim_matches_truth(name):
    v, f = WMESHES[name]
    check_mesh(name, v, f, 1200)


def test_shells_count_the_enclosing_shells():
    v, f = doc.scene("shells32")
    rng = np.random.default_rng(1)
    d = rng.normal(size=(3000, 3))
    p = (d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(0.0, 1.3, (3000, 1))).astype(np.float32)
    rho = np.linalg.norm(p.astype(np.float64), axis=1)
    radii = doc.shell_radii(32)
    inr = radii * doc.shell_inradius_factor()
    enclosing = (rho[:, None] < inr[None, :] * (1 - 1e-3)).sum(1)
    _, clear = doc.shell_parity(p, 32)
    blob = hostsim.build_blob(v, f)
    exact = W.sim_winding(blob, p, INF)["w"]
    fast = W.sim_winding(blob, p, 2.0)["w"]
    assert clear.sum() > 1000 and len(np.unique(enclosing[clear])) > 20
    np.testing.assert_allclose(exact[clear], enclosing[clear], atol=1e-3)
    assert np.array_equal(np.rint(fast[clear]), enclosing[clear])


def test_duplicates_add_up():
    v, f = doc.scene("dup600")
    rng = np.random.default_rng(2)
    p = np.stack([rng.uniform(-1, 1, 500), rng.uniform(-1, 1, 500), rng.uniform(-1, 1.5, 500)], 1).astype(np.float32)
    p = p[np.abs(p[:, 2] - 0.25) > 0.05]
    single = W.truth(doc.ONE_TRI, [[0, 1, 2]], p)
    np.testing.assert_allclose(W.truth(v, f, p), 600 * single, rtol=1e-9, atol=1e-9)
    blob = hostsim.build_blob(v, f)
    np.testing.assert_allclose(W.sim_winding(blob, p, INF)["w"], 600 * single, rtol=2e-5, atol=1e-4)


def test_reversed_orientation_negates():
    v, f = synth.icosphere(3)
    r = np.ascontiguousarray(f[:, ::-1])
    rng = np.random.default_rng(3)
    p = sample_points(v, 800, rng)
    np.testing.assert_allclose(W.truth(v, r, p), -W.truth(v, f, p), atol=1e-12)
    b, br = hostsim.build_blob(v, f), hostsim.build_blob(v, r)
    for beta in (INF, 2.0):
        np.testing.assert_allclose(W.sim_winding(br, p, beta)["w"], -W.sim_winding(b, p, beta)["w"], atol=1e-5)


def test_open_meshes_give_fractions():
    v, f = WMESHES["cube_open"]
    p = np.array([[0, 0, 0], [0, 0, -0.45], [0, 0, 0.45]], np.float32)
    w = W.sim_winding(hostsim.build_blob(v, f), p, 2.0)["w"]
    t = W.truth(v, f, p)
    np.testing.assert_allclose(w, t, atol=1e-6)
    assert abs(t[0] - 5.0 / 6.0) < 1e-9                     # from the centre every face subtends 4 pi / 6
    assert 0.5 < t[1] < t[0] < t[2] < 1.0                    # less near the missing bottom (-z) face


@pytest.mark.parametrize("name", list(WMESHES))
def test_moments_match_binary64(name):
    """every record against its node's own triangles in binary64: rho bounds every finite vertex, p~ is the
    area-weighted centroid, N the summed area vector and M the first moment about the stored p~ (relative to scales
    with the binary32 rounding floors, ws_moment_check)"""
    v, f = WMESHES[name]
    blob = hostsim.build_blob(v, f)
    r = W.moment_check(blob)
    assert r["nodes"] == W.n_nodes(blob) and r["vertices"] >= np.isfinite(v[f]).all(axis=2).sum()
    assert r["rho_violations"] == 0 and r["rho_ratio"] <= 1.0, r
    assert r["p_err"] <= 1e-2 and r["n_err"] <= 0.05 and r["m_err"] <= 0.05, r


def test_far_field_converges_at_second_order():
    """the two-term far field of a cluster (the root record of a 400-triangle soup) against the exact solid-angle sum:
    doubling the distance cuts the dipole's error 8x and the two-term error 16x, so the first-moment term, its sign,
    its trace part and the child shifts of M must all be right"""
    v, f = synth.triangle_soup(400, seed=3)
    blob = hostsim.build_blob(v, f)
    rec = W.sim_moments(blob)[0]
    p, rho, n = rec[:3].astype(np.float64), float(rec[3]), rec[4:7].astype(np.float64)
    u = np.random.default_rng(0).normal(size=(16, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    e1, e2 = [], []
    for k in (3.0, 6.0, 12.0, 24.0):
        q = (p[None] + k * rho * u).astype(np.float32)
        exact = 4 * np.pi * W.truth(v, f, q)
        r = p[None] - q.astype(np.float64)
        dipole = (r @ n) / np.linalg.norm(r, axis=1) ** 3
        e1.append(np.abs(dipole - exact))
        e2.append(np.abs(W.sim_far_field(rec, q).astype(np.float64) - exact))
    s1 = np.median(np.log2(np.array(e1[:-1]) / np.array(e1[1:])), axis=1)
    s2 = np.median(np.log2(np.array(e2[:-1]) / np.array(e2[1:])), axis=1)
    assert ((s1 > 2.6) & (s1 < 3.4)).all(), s1
    assert (s2 > 3.7).all(), s2
    ratio = [np.median(b) / np.median(a) for a, b in zip(e1, e2)]   # two-term over dipole error, falls like rho / |r|
    assert ratio[0] < 1.0 and ratio[-1] < 0.25, ratio


def test_moments_after_refit():
    """the moment pass reads nothing but the blob: two passes over copies give the same bits, and the moments of a
    re-fitted blob match the re-fitted triangles and give the truth's winding numbers"""
    v, f = synth.icosphere(4)
    blob = hostsim.build_blob(v, f)
    m1, m2 = W.sim_moments(blob), W.sim_moments(blob.copy())
    assert np.array_equal(m1.view(np.uint32), m2.view(np.uint32))
    v2 = (v * np.float32(1.3) + np.float32(0.1)).astype(np.float32)
    re = hostsim.refit_blob(blob, v2, f)
    m3 = W.sim_moments(re)
    assert not np.array_equal(m1, m3)
    r = W.moment_check(re, m3)
    assert r["rho_violations"] == 0 and r["n_err"] <= 0.05 and r["m_err"] <= 0.05, r
    p = sample_points(v2, 400, np.random.default_rng(4))
    truth = W.truth(v2, f, p)
    clear = surface_distance(v2, f, p) > DELTA * diagonal(v2)
    assert np.abs(W.sim_winding(re, p, 2.0, m3)["w"] - truth)[clear].max() <= TOL_FAST_ICO
