"""Pseudo-normal signed distance, CPU tier: the host simulator of rt_pseudonormal.cu and of the signed-distance
kernel (their own RT_HD code) against known answers in every Voronoi region, against the binary64 truth (distance
from the point oracle, inside from the winding-number oracle) on closed meshes at every scale, unwelded soups against
welded meshes bit for bit, the edge counts of open, non-manifold, inconsistent and degenerate meshes, and reversed
orientation.

Signs are compared with the truth only for points farther than TAU times the bounding-box diagonal from the surface:
nearer than that the binary32 closest point itself is uncertain at the scale of the distance."""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pseudonormal"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import hostsim  # noqa: E402
import pointquery as pq  # noqa: E402
import pseudonormal as P  # noqa: E402
from test_closest_point_logic import sample_points  # noqa: E402
from triro import synth  # noqa: E402

TAU = 1e-4


def closed_meshes():
    out = {"cube": synth.cube(0.5), "ico3": synth.icosphere(3), "ico5": synth.icosphere(5), "torus": P.torus(),
           "star": P.star_prism(), "notched": P.notched_cube()}
    ico, icf = synth.icosphere(4)
    for s, off in ((1e6, 0.0), (1e-6, 0.0), (1e4, 3e7)):
        out[f"ico4_s{s:g}_o{off:g}"] = ((ico.astype(np.float64) * s + off).astype(np.float32), icf)
    out["star_s1e4_o3e7"] = ((P.star_prism()[0].astype(np.float64) * 1e4 + 3e7).astype(np.float32), P.star_prism()[1])
    return out


CLOSED = closed_meshes()


def diagonal(v):
    good = v[np.isfinite(v).all(axis=1)].astype(np.float64)
    return float(np.linalg.norm(good.max(0) - good.min(0)))


def bits_equal(a, b, what):
    a = np.ascontiguousarray(a, dtype=np.float32); b = np.ascontiguousarray(b, dtype=np.float32)
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ (first at {np.argwhere(bad)[0]})"


def feature_points(v, f, scale, rng, per=4):
    """points around every vertex, every edge (at random parameters) and every face centroid, offset by up to `scale`
    in random directions, so that every Voronoi region of every feature is sampled from both sides"""
    tv = v[f].astype(np.float64)
    edges = np.concatenate([tv[:, [0, 1]], tv[:, [1, 2]], tv[:, [2, 0]]])
    t = rng.uniform(0.05, 0.95, (len(edges), per, 1))
    on_edges = (edges[:, None, 0] * (1 - t) + edges[:, None, 1] * t).reshape(-1, 3)
    base = np.concatenate([np.repeat(v.astype(np.float64), per, 0), on_edges, np.repeat(tv.mean(1), per, 0)])
    d = rng.normal(size=base.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return (base + d * rng.uniform(0.02, 1.0, (len(base), 1)) * scale).astype(np.float32)


def face_only_inside(v, f, p):
    """the sign a face normal alone gives: (p - c) . n_face < 0 for the closest triangle (mirror oracle)"""
    r = pq.query(pq.PointMesh(v, f), p, pq.MIRROR)
    tv = v[f[r["tri"]]].astype(np.float64)
    n = np.cross(tv[:, 1] - tv[:, 0], tv[:, 2] - tv[:, 0])
    return ((p - r["closest"]) * n).sum(1) < 0, r


# ------------------------------------------------------------------ known answers
def test_cube_known_answers():
    v, f = synth.cube(0.5)
    blob = hostsim.build_blob(v, f)
    rows, counts = P.sim_normals(blob)
    assert counts == (0, 0, 0)
    # every vertex normal is the corner direction times pi/2 (three right angles), every edge normal the sum of two unit
    # face normals (or 2 n on a face diagonal)
    vn = rows.reshape(-1, 6, 4)[:, :3, :3]
    np.testing.assert_allclose(np.abs(vn), np.pi / 2, rtol=1e-6)
    en = np.abs(rows.reshape(-1, 6, 4)[:, 3:, :3])
    assert np.isin(np.round(en, 6), [0.0, 1.0, 2.0]).all()
    p = np.array([[0, 0, 0], [0.3, -0.2, 0.1],                      # inside, face
                  [0.7, 0.1, 0.0], [0.1, 0.1, -0.9],                # outside, face
                  [0.7, 0.7, 0.0], [0.45, 0.45, 0.2],               # outside / inside, edge
                  [0.7, 0.7, 0.7], [0.49, 0.49, 0.49],              # outside / inside, vertex
                  [0.5, 0.5, -0.5]], np.float32)                    # at a vertex: exactly 0, +0
    sd = P.sim_signed_distance(blob, p)["sd"]
    want = [0.5, 0.2, -0.2, -0.4, -np.sqrt(0.08), 0.05, -np.sqrt(0.12), 0.01, 0.0]
    np.testing.assert_allclose(sd, want, rtol=1e-6, atol=1e-7)
    assert sd[-1] == 0.0 and not np.signbit(sd[-1])


def test_point_tri_regions():
    """point_tri reports the Voronoi region of the branch it took; in the zero-area branch the chosen segment's edge,
    or the vertex at its end when the parameter is 0 or 1"""
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    pts = {"face": [0.25, 0.25, 2.0], "ab": [0.5, -1.0, 0.0], "ac": [-1.0, 0.5, 0.0], "bc": [1.0, 1.0, 0.5],
           "a": [-1.0, -1.0, 0.0], "b": [2.0, -0.5, 0.0], "c": [-0.5, 2.0, 0.0]}
    for want, p in pts.items():
        assert P.sim_region(p, tri) == want
    seg = np.array([[0, 0, 0], [0, 0, 0], [1, 0, 0]], np.float32)       # a == b: segments ab (a point), ac, bc
    assert P.sim_region([0.5, 1.0, 0.0], seg) == "ac"
    assert P.sim_region([-1.0, 0.5, 0.0], seg) == "a"                   # t = 0 on ab
    assert P.sim_region([2.0, 0.5, 0.0], seg) == "c"                    # t = 1 on ac
    line = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0]], np.float32)      # collinear
    assert P.sim_region([1.5, 1.0, 0.0], line) == "ac"
    assert P.sim_region([3.0, 1.0, 0.0], line) == "c"


@pytest.mark.parametrize("name", ["cube", "star", "notched", "torus"])
def test_every_region_against_truth(name):
    """points around every feature of closed solids with convex, acute and reflex edges and saddle and concave
    vertices: the sign equals the truth beyond TAU, every Voronoi region of point_tri occurs, and on the star (acute
    tips) the face normal alone gets some of them wrong"""
    v, f = CLOSED[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    diag = diagonal(v)
    p = feature_points(v, f, 0.05 * diag, rng)
    d, inside = P.truth(v, f, p)
    clear = d > TAU * diag
    assert clear.sum() > 0.9 * len(p)
    sd = P.sim_signed_distance(hostsim.build_blob(v, f), p)["sd"]
    assert np.array_equal((sd > 0)[clear], inside[clear]), f"{int(((sd > 0) != inside)[clear].sum())} signs differ"
    face_only, r = face_only_inside(v, f, p)
    regions = {P.sim_region(p[i], v[f[r["tri"][i]]]) for i in range(len(p))}
    assert "face" in regions and regions & {"a", "b", "c"} and regions & {"ab", "ac", "bc"}, regions
    if name == "star":
        assert (face_only != inside)[clear].sum() > 0


def test_concave_vertex_and_reflex_edges():
    """directly off the concave vertex and the reflex edges of the notched cube, from inside and from the notch"""
    v, f = P.notched_cube()
    blob = hostsim.build_blob(v, f)
    p = np.array([[0.9, 0.9, 0.9],       # inside, nearest feature the concave vertex (1, 1, 1)
                  [0.9, 0.9, 1.5],       # inside, nearest the reflex edge x = y = 1
                  [1.5, 0.9, 0.9],       # inside, reflex edge y = z = 1
                  [1.2, 1.2, 1.2],       # in the notch: outside, faces at 0.2
                  [1.3, 1.1, 1.6]], np.float32)
    sd = P.sim_signed_distance(blob, p)["sd"]
    d, inside = P.truth(v, f, p)
    assert inside.tolist() == [True, True, True, False, False]
    np.testing.assert_allclose(np.abs(sd), d, rtol=1e-6)
    assert ((sd > 0) == inside).all()
    tri = pq.query(pq.PointMesh(v, f), p, pq.MIRROR)["tri"]
    assert P.sim_region(p[0], v[f[tri[0]]]) in ("a", "b", "c")
    assert P.sim_region(p[1], v[f[tri[1]]]) in ("ab", "ac", "bc")


# ------------------------------------------------------------------ simulator against the truth
@pytest.mark.parametrize("name", list(CLOSED))
def test_hostsim_sign_matches_truth(name):
    v, f = CLOSED[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()) + 1)
    p = sample_points(v, 1500, rng)
    blob = hostsim.build_blob(v, f)
    rows, counts = P.sim_normals(blob)
    assert counts == (0, 0, 0)
    s = P.sim_signed_distance(blob, p, rows)
    d, inside = P.truth(v, f, p)
    clear = d > TAU * diagonal(v)
    assert clear.sum() >= len(p) // 2
    bad = ((s["sd"] > 0) != inside) & clear
    assert not bad.any(), f"{name}: {int(bad.sum())} of {int(clear.sum())} signs differ from the truth"
    # |sd| is the closest-point distance of rt_point.cuh bit for bit
    bits_equal(np.abs(s["sd"]), pq.sim_closest_point(blob, p)["distance"], f"{name}: |sd| vs closest point")
    assert s["stats"]["points"] == len(p) and s["stats"]["found"] == len(p)


# ------------------------------------------------------------------ welding
@pytest.mark.parametrize("name", ["cube", "ico3", "torus", "star", "notched", "ico4_s10000_o3e+07"])
def test_unwelded_soup_equals_welded_mesh(name):
    v, f = CLOSED[name]
    sv, sf = P.soup(v, f)
    b, bs = hostsim.build_blob(v, f), hostsim.build_blob(sv, sf)
    (rw, cw), (rs, cs) = P.sim_normals(b), P.sim_normals(bs)
    assert cw == cs == (0, 0, 0)
    bits_equal(rs, rw, f"{name}: normals")
    p = sample_points(v, 800, np.random.default_rng(9))
    bits_equal(P.sim_signed_distance(bs, p)["sd"], P.sim_signed_distance(b, p)["sd"], f"{name}: signed distance")


def test_negative_zero_welds_with_positive_zero():
    v, f = synth.cube(0.5)
    v = v - np.float32([0.5, 0.0, 0.0])                      # x in {-1, 0}
    sv, sf = P.soup(v, f)
    neg = sv.copy()
    zeros = np.flatnonzero(neg[:, 0] == 0)
    neg[zeros[::2], 0] = -0.0
    assert np.signbit(neg[zeros, 0]).any() and not np.signbit(sv[zeros, 0]).any()
    rw, cw = P.sim_normals(hostsim.build_blob(sv, sf))
    rn, cn = P.sim_normals(hostsim.build_blob(neg, sf))
    assert cw == cn == (0, 0, 0)
    bits_equal(rn, rw, "normals with -0 coordinates")


# ------------------------------------------------------------------ edge counts
def counts_of(v, f):
    return P.sim_normals(hostsim.build_blob(v, f))[1]


def test_edge_counts():
    v, f = synth.cube(0.5)
    assert counts_of(v, f) == (0, 0, 0)
    assert counts_of(v, f[2:]) == (4, 0, 0)                                  # bottom face removed
    flipped = f.copy(); flipped[5] = flipped[5, ::-1]
    assert counts_of(v, flipped) == (0, 0, 3)                                # one face turned over
    fin_v = np.concatenate([v, [[0.0, 0.0, 1.5]]]).astype(np.float32)        # a fin on the edge (0.5, 0.5, z)
    fin_f = np.concatenate([f, [[2, 6, 8]]]).astype(np.int32)
    assert counts_of(fin_v, fin_f) == (2, 1, 0)
    iv, iff = synth.icosphere(3)
    assert counts_of(iv, iff) == (0, 0, 0)
    assert counts_of(*P.soup(iv, iff)) == (0, 0, 0)
    assert counts_of(*synth.heightfield(8, 4)) == (2 * (8 + 4), 0, 0)


def test_nan_and_zero_area_triangles():
    """a triangle with a non-finite vertex takes part in nothing: its rows are zero and the rest is as without it; a
    zero-area triangle takes part with zero normals, here making its two distinct edges non-manifold or boundary"""
    v, f = synth.cube(0.5)
    nv = np.concatenate([v, [[np.nan, 0, 0], [np.inf, 1, 1]]]).astype(np.float32)
    nf = np.concatenate([f, [[0, 8, 1], [8, 9, 2], [3, 9, 4]]]).astype(np.int32)
    b = hostsim.build_blob(nv, nf)
    rows, counts = P.sim_normals(b)
    assert counts == (0, 0, 0)
    tris = b[256:256 + 48 * len(nf)].view(np.float32).reshape(-1, 12)
    bad = ~np.isfinite(tris[:, [0, 1, 2, 4, 5, 6, 8, 9, 10]]).all(1)
    assert bad.sum() == 3 and (rows[bad] == 0).all() and (rows[~bad] != 0).any()
    p = sample_points(v, 600, np.random.default_rng(2))
    bits_equal(P.sim_signed_distance(b, p)["sd"], P.sim_signed_distance(hostsim.build_blob(v, f), p)["sd"],
               "signed distance with non-finite triangles")
    # zero area: a repeated vertex on the cube edge 0-1 (one more face on it) and a collinear triangle hanging off it
    zv = np.concatenate([v, [[0.0, -0.5, -0.5], [0.25, -0.5, -0.5]]]).astype(np.float32)
    zf = np.concatenate([f, [[0, 1, 1]]]).astype(np.int32)
    rows, counts = P.sim_normals(hostsim.build_blob(zv, zf))
    assert counts == (1, 1, 0)                                # edge 0-1 gets a third face; edge 1-1 is alone
    zf = np.concatenate([f, [[0, 8, 9]]]).astype(np.int32)   # collinear along the edge 0-1, sharing vertex 0
    assert counts_of(zv, zf) == (3, 0, 0)
    assert np.isfinite(P.sim_normals(hostsim.build_blob(zv, zf))[0]).all()


def test_empty_mesh_and_non_finite_points():
    empty = hostsim.build_blob(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    rows, counts = P.sim_normals(empty)
    assert rows.shape == (0, 24) and counts == (0, 0, 0)
    assert (P.sim_signed_distance(empty, [[0, 0, 0]])["sd"] == -np.inf).all()
    v, f = synth.cube(0.5)
    sd = P.sim_signed_distance(hostsim.build_blob(v, f), [[np.nan, 0, 0], [0, np.inf, 0], [0, 0, 0]])["sd"]
    assert sd.tolist() == [-np.inf, -np.inf, 0.5]


def test_reversed_orientation_flips_the_sign():
    v, f = synth.icosphere(3)
    r = np.ascontiguousarray(f[:, ::-1])
    assert counts_of(v, r) == (0, 0, 0)
    p = sample_points(v, 1500, np.random.default_rng(3))
    d, _ = P.truth(v, f, p)
    clear = d > TAU * diagonal(v)
    a = P.sim_signed_distance(hostsim.build_blob(v, f), p)["sd"]
    b = P.sim_signed_distance(hostsim.build_blob(v, r), p)["sd"]
    assert np.array_equal((a > 0)[clear], (b < 0)[clear])


def test_open_heightfield_is_the_side_of_the_orientation():
    """not inside/outside, but fully defined: the points high above the terrain get one sign, those far below the
    other, and the sign follows the faces' orientation"""
    v, f = synth.heightfield(32, 16)
    assert counts_of(v, f)[0] > 0
    xy = np.random.default_rng(4).uniform(-0.9, 0.9, (500, 2))
    top = np.concatenate([xy, np.full((500, 1), 0.6)], 1).astype(np.float32)
    bot = np.concatenate([xy, np.full((500, 1), -0.6)], 1).astype(np.float32)
    blob = hostsim.build_blob(v, f)
    n = np.cross(v[f[0, 1]] - v[f[0, 0]], v[f[0, 2]] - v[f[0, 0]])
    up = 1.0 if n[2] > 0 else -1.0                            # +1: the faces look up, "above" is outside
    assert (np.sign(P.sim_signed_distance(blob, top)["sd"]) == -up).all()
    assert (np.sign(P.sim_signed_distance(blob, bot)["sd"]) == up).all()
    flipped = hostsim.build_blob(v, np.ascontiguousarray(f[:, ::-1]))
    assert (np.sign(P.sim_signed_distance(flipped, top)["sd"]) == up).all()
