"""Distance gradient, CPU tier: the host simulator of rt_distgrad.cu (its own RT_HD code, std::stable_sort in place
of the onesweep sort) against known answers in every Voronoi region of a triangle and a cube, degenerate inputs, a
binary64 numpy reference of the formula on every mesh family and scale, central finite differences of the binary64
point oracle, and the documented summation order (groups of 32, level after level, per vertex and per window).

The forward outputs fed to the simulator come from the point oracle's binary32 mirror, which the closest-point
kernel reproduces bit for bit."""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "distgrad"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import distgrad as D  # noqa: E402
import pointquery as pq  # noqa: E402
from test_closest_point_logic import MESHES, bits_equal, sample_points  # noqa: E402
from triro import synth  # noqa: E402


def forward(v, f, p, max_distance=float("inf")):
    r = pq.query(pq.PointMesh(v, f), p, pq.MIRROR, max_distance)
    return r["closest"], r["distance"], r["tri"], r["uv"]


def grads(v, f, p, g=None, sign=None, window=0, max_distance=float("inf")):
    c, d, t, uv = forward(v, f, p, max_distance)
    value = d if sign is None else np.where(sign, d, -d).astype(np.float32)
    g = np.ones(len(p), np.float32) if g is None else g
    gp, gv = D.sim_grad(p, g, value, c, t, uv, f, len(v), window)
    return gp, gv, (g, value, c, t, uv)


TRI_V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
TRI_F = np.array([[0, 1, 2]], np.int32)


@pytest.mark.parametrize("negative", [False, True])
def test_triangle_known_answers_in_every_region(negative):
    # face, vertex a, b, c, edge ab, ac, bc; each above the plane by 0.5
    p = np.array([[0.2, 0.3, 0.5], [-1, -1, 0.5], [2, -0.5, 0.5], [-0.5, 2, 0.5], [0.5, -1, 0.5], [-1, 0.5, 0.5],
                  [1, 1, 0.5]], np.float32)
    s = -1.0 if negative else 1.0
    gp, gv, (_, value, c, t, uv) = grads(TRI_V, TRI_F, p, sign=np.full(len(p), not negative))
    assert (np.signbit(value) == negative).all() and (t == 0).all()
    np.testing.assert_allclose(gp[0], [0, 0, s], atol=1e-7)
    for i in range(len(p)):
        gpi, gvi = D.sim_grad(p[i:i + 1], [1.0], value[i:i + 1], c[i:i + 1], t[i:i + 1], uv[i:i + 1], TRI_F, 3)
        u = (p[i] - c[i]).astype(np.float64)
        u /= np.linalg.norm(u)
        np.testing.assert_allclose(gpi[0], s * u, atol=2e-7)
        w = np.array([uv[i, 0], uv[i, 1], 1 - uv[i, 0] - uv[i, 1]])
        np.testing.assert_allclose(gvi, -w[:, None] * s * u[None], atol=2e-7)
        if 1 <= i <= 3:                       # a vertex region: the whole weight on that vertex
            k = i - 1
            assert (gvi[np.arange(3) != k] == 0).all()
            np.testing.assert_allclose(gvi[k], -s * u, atol=2e-7)
    # face region: the vertex gradients are -w_i n (n the unit normal towards p), summing to -grad_p
    np.testing.assert_allclose(gv.sum(0), -gp.sum(0), atol=1e-6)


def test_cube_faces_and_corners():
    v, f = synth.cube(0.5)
    face_pts = np.array([[0.9, 0.1, -0.2], [-0.1, -0.8, 0.3], [0.2, 0.1, 0.7], [0.1, 0.2, 0.3]], np.float32)
    gp, _, (_, value, c, t, uv) = grads(v, f, face_pts)
    # the face-region closest point is a rounded barycentric combination: tangential error of a few ulp
    np.testing.assert_allclose(gp[:3], [[1, 0, 0], [0, -1, 0], [0, 0, 1]], atol=5e-7)
    assert abs(np.abs(gp[3]).max() - 1) < 5e-7                      # inside: the nearest face's normal
    for corner in range(8):
        p = (v[corner].astype(np.float64) * 3).astype(np.float32)[None]
        gp, gv, (_, value, c, t, uv) = grads(v, f, p)
        u = p[0].astype(np.float64) - v[corner]
        u /= np.linalg.norm(u)
        np.testing.assert_allclose(gp[0], u, atol=2e-7)
        assert (gv[np.arange(8) != corner] == 0).all()
        np.testing.assert_allclose(gv[corner], -u, atol=2e-7)


def test_degenerate_inputs_give_zero_never_nan():
    v, f = synth.icosphere(2)
    on_vertex = v[:3]
    far = np.array([[5.0, 0, 0]], np.float32)
    bad = np.array([[np.nan, 0, 0], [np.inf, 0, 0]], np.float32)
    p = np.concatenate([on_vertex, far, bad]).astype(np.float32)
    c, d, t, uv = forward(v, f, p, max_distance=2.0)
    assert (d[:3] == 0).all() and (t[3:] == -1).all() and np.isinf(d[3:]).all()
    g = np.full(len(p), 3.0, np.float32)
    gp, gv = D.sim_grad(p, g, d, c, t, uv, f, len(v))
    assert (gp == 0).all() and not np.signbit(gp).any() and (gv == 0).all() and not np.signbit(gv).any()
    # -0 and -inf signed values, and a triangle index out of range, contribute nothing either
    gp, gv = D.sim_grad(p[:2], [1, 1], [-0.0, -np.inf], c[:2], [0, len(f)], uv[:2], f, len(v))
    assert (gp == 0).all() and (gv == 0).all()
    # zero-area triangles and faces that repeat a vertex index: finite, and equal to the binary64 reference
    dv = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [0, 1, 0], [0, 1, 0]], np.float32)
    df = np.array([[0, 1, 2], [0, 0, 3], [3, 4, 1], [1, 1, 1]], np.int32)
    q = np.random.default_rng(3).uniform(-1, 3, (500, 3)).astype(np.float32)
    gp, gv, inputs = grads(dv, df, q)
    assert np.isfinite(gp).all() and np.isfinite(gv).all()
    rq, rv = D.reference(q, *inputs, df, len(dv))
    np.testing.assert_allclose(gp, rq, atol=1e-6)
    np.testing.assert_allclose(gv, rv, atol=1e-4)


@pytest.mark.parametrize("name", list(MESHES))
def test_hostsim_matches_binary64_reference(name):
    v, f = MESHES[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    p = sample_points(v, 3000, rng)
    g = rng.normal(size=len(p)).astype(np.float32)
    gp, gv, inputs = grads(v, f, p, g=g, sign=rng.random(len(p)) < 0.5)
    rq, rv = D.reference(p, *inputs, f, len(v))
    assert np.isfinite(gp).all() and np.isfinite(gv).all()
    # q is three correctly rounded operations on exact float32 inputs; a vertex sum is at most ~log32(L) + 32 roundings
    # of partial sums bounded by the sum of the magnitudes
    assert (np.abs(gp - rq) <= 4e-7 * np.abs(g)[:, None]).all()
    mag = np.zeros(len(v))
    _, c, t, uv = inputs[1:]
    live = (inputs[1] != 0) & np.isfinite(inputs[1]) & (t >= 0)
    w = np.stack([uv[:, 0], uv[:, 1], 1 - uv[:, 0] - uv[:, 1]], 1).astype(np.float64)
    for k in range(3):
        np.add.at(mag, f[t[live], k], np.abs(w[live, k] * g[live]))
    assert (np.abs(gv - rv) <= 1e-5 * mag[:, None]).all()


def test_finite_differences_of_the_binary64_oracle():
    v, f = synth.icosphere(1)
    rng = np.random.default_rng(11)
    p = (rng.normal(size=(1000, 3)) * rng.uniform(0.3, 1.7, (1000, 1))).astype(np.float32)
    # the closest feature is unique by a margin: the point lies inside its triangle's face region by 1e-2 in weights
    # and every other triangle is farther by 2e-3, and the surface by 5e-3 (the step is 1e-3)
    truth = pq.query(pq.PointMesh(v, f), p, pq.TRUTH)
    c, d, t, uv = forward(v, f, p)
    w = np.stack([uv[:, 0], uv[:, 1], 1 - uv[:, 0] - uv[:, 1]], 1)
    all_d = np.sqrt(pq.all_d2(pq.PointMesh(v, f), p))
    all_d[np.arange(len(p)), t] = np.inf
    keep = (w.min(1) > 1e-2) & (all_d.min(1) - truth["distance"] > 2e-3) & (truth["distance"] > 5e-3)
    assert keep.sum() > 100
    g = keep.astype(np.float32)
    gp, gv = D.sim_grad(p, g, d, c, t, uv, f, len(v))

    def total(vv, pp):
        return float((pq.query(pq.PointMesh(vv, f), pp, pq.TRUTH)["distance"] * keep).sum())

    h = 1e-3
    for a in range(3):
        hi, lo = p.copy(), p.copy()
        hi[:, a] += h; lo[:, a] -= h
        dh = pq.query(pq.PointMesh(v, f), hi, pq.TRUTH)["distance"]
        dl = pq.query(pq.PointMesh(v, f), lo, pq.TRUTH)["distance"]
        fd = (dh - dl) / (hi[:, a].astype(np.float64) - lo[:, a])
        np.testing.assert_allclose(gp[keep, a], fd[keep], atol=1e-4)
    for j in range(len(v)):
        for a in range(3):
            hi, lo = v.copy(), v.copy()
            hi[j, a] += h; lo[j, a] -= h
            fd = (total(hi, p) - total(lo, p)) / (float(hi[j, a]) - float(lo[j, a]))
            assert abs(gv[j, a] - fd) <= 1e-4 * max(1.0, abs(fd)), (j, a, gv[j, a], fd)


def live_points(value, t):
    """the points that contribute: |value| positive and finite, and a triangle"""
    a = np.abs(np.asarray(value, np.float64))
    return (a > 0) & (a < np.inf) & (np.asarray(t) >= 0)


@pytest.mark.parametrize("window", [0, 1000, 777])
def test_summation_order_is_the_documented_tree(window):
    v, f = synth.cube(0.5)
    rng = np.random.default_rng(window)
    # 3000 points beyond one corner (runs of 3000 pairs: three levels) plus points around the cube
    corner = (v[6].astype(np.float64) + 0.2 + rng.uniform(0, 1, (3000, 3))).astype(np.float32)
    p = np.concatenate([corner, rng.uniform(-1, 1, (1500, 3)).astype(np.float32)])
    g = rng.normal(size=len(p)).astype(np.float32)
    gp, gv, (_, value, c, t, uv) = grads(v, f, p, g=g, window=window)
    bits_equal(gv, D.documented_order(gp, uv, live_points(value, t), t, f, len(v), window), f"window {window}")


def test_result_of_a_vertex_depends_on_its_own_list_only():
    v, f = synth.icosphere(3)
    rng = np.random.default_rng(5)
    p = sample_points(v, 2000, rng)[:150]
    gp, gv, _ = grads(v, f, p)
    # points that touch other vertices only, put in front: every run moves in the sorted array, no sum changes
    c, d, t, uv = forward(v, f, p)
    touched = np.unique(f[t])
    q = rng.uniform(-1.5, 1.5, (4000, 3)).astype(np.float32)
    _, _, tq, _ = forward(v, f, q)
    q = q[~np.isin(f[tq], touched).any(1)][:1000]
    assert len(q) > 10
    gp2, gv2, _ = grads(v, f, np.concatenate([q, p]))
    bits_equal(gp2[len(q):], gp, "grad_points")
    bits_equal(gv2[touched], gv[touched], "grad_vertices of the first batch's vertices")
    # one window per point: the sums are added point by point in order
    _, gv1, _ = grads(v, f, p[:200], window=1)
    _, gv0, inputs = grads(v, f, p[:200])
    bits_equal(gv1, D.documented_order(D.sim_grad(p[:200], *inputs, f, len(v))[0], inputs[4],
                                       live_points(inputs[1], inputs[3]), inputs[3], f, len(v), 1), "window 1")
    np.testing.assert_allclose(gv1, gv0, atol=1e-5)
