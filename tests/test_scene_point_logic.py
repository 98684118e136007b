"""Point queries on instanced scenes on the CPU: the host simulator of rt_scene.cuh (the kernels' own RT_HD code) with
and without the top-level tree against a brute-force loop over every triangle of every instance, and against the
single-mesh simulator on the scene flattened with the same binary32 vertices, bit for bit; the exhaustive check of
the instance walk's world bound; the singular-value bound; and the pseudo-normal sign against the binary64 truth."""
import os
import sys

import numpy as np
import pytest

_T = os.path.dirname(os.path.abspath(__file__))
for _d in ("scene", "pointquery", "pseudonormal"):
    sys.path.insert(0, os.path.join(_T, _d))
import pointquery as pq  # noqa: E402
import pseudonormal as pn  # noqa: E402
import scene as sc  # noqa: E402
import scenepoint as sp  # noqa: E402
import scene_cases as cases  # noqa: E402
import scene_point_cases as spc  # noqa: E402
from helpers import assert_bits_equal  # noqa: E402
from triro import synth  # noqa: E402


def _blobs(ms):
    return [sc.hostsim.build_blob(v, f) for v, f in ms]


def _same(a: dict, b: dict, what: str):
    assert a.keys() == b.keys()
    for k in a:
        assert_bits_equal(a[k], b[k], f"{what}.{k}")


def _face_offsets(ms, inst_mesh):
    return np.concatenate([[0], np.cumsum([len(ms[int(m)][1]) for m in inst_mesh])]).astype(np.int64)


@pytest.fixture(scope="module")
def big_scene():
    ms, inst_mesh, t = cases.scene(300, seed=0)
    blobs = _blobs(ms)
    s = sc.SimScene(blobs, inst_mesh, t)
    fv, ff, _, _ = sp.flatten_affine(ms, inst_mesh, t)
    lo, hi = spc.scene_box(fv)
    pts = {"uniform": spc.uniform_points(lo, hi, 400, seed=0), "surface": spc.surface_points(fv, ff, 400, seed=1),
           "special": spc.special_points(lo, hi)}
    return ms, inst_mesh, t, s, fv, ff, pts


@pytest.mark.parametrize("max_distance", [float("inf"), 0.5, 0.0])
def test_tree_equals_brute_force(big_scene, max_distance):
    ms, inst_mesh, t, s, fv, ff, pts = big_scene
    for name, p in pts.items():
        got = sp.closest_point(s, p, max_distance)
        _same(got, sp.closest_point(s, p, max_distance, mode="instances"), f"{name}/instances")
        _same(got, sp.closest_point(s, p, max_distance, mode="brute"), f"{name}/brute")
        bad = ~np.isfinite(p).all(1)
        assert (got["inst"][bad] == -1).all() and np.isinf(got["distance"][bad]).all()
    got = sp.closest_point(s, pts["uniform"])
    assert len(np.unique(got["inst"])) > 50
    assert not (got["inst"] == inst_mesh.tolist().index(3)).any(), "an instance of the empty mesh answered"
    if max_distance == 0.0:
        surf = sp.closest_point(s, pts["surface"], 0.0)
        assert ((surf["inst"] >= 0) == (surf["distance"] == 0)).all()


@pytest.mark.parametrize("max_distance", [float("inf"), 0.25])
def test_equals_flattened_mesh(big_scene, max_distance):
    ms, inst_mesh, t, s, fv, ff, pts = big_scene
    blob = sc.hostsim.build_blob(fv, ff)
    off = _face_offsets(ms, inst_mesh)
    for name, p in pts.items():
        got = sp.closest_point(s, p, max_distance)
        ref = pq.sim_closest_point(blob, p, max_distance)
        f = np.where(got["inst"] >= 0, off[np.maximum(got["inst"], 0)] + got["tri"], -1)
        np.testing.assert_array_equal(f, ref["tri"], err_msg=name)
        for k in ("closest", "distance", "uv"):
            assert_bits_equal(got[k], ref[k], f"{name}.{k}")


def test_identity_instance_equals_single_mesh():
    for v, f in (synth.icosphere(3), synth.triangle_soup(300, sigma=0.05, seed=4), pn.torus()):
        blob = sc.hostsim.build_blob(v, f)
        s = sc.SimScene([blob], [0], np.eye(4, dtype=np.float32)[None, :3])
        p = np.concatenate([spc.uniform_points(-1.5, 1.5, 500), spc.surface_points(v, f, 300),
                            spc.special_points([-1] * 3, [1] * 3)])
        got = sp.closest_point(s, p)
        ref = pq.sim_closest_point(blob, p)
        for k in ("closest", "distance", "tri", "uv"):
            assert_bits_equal(got[k], ref[k], k)
        rows, _ = pn.sim_normals(blob)
        sd = sp.closest_point(s, p, normals=[rows])["sd"]
        assert_bits_equal(sd, pn.sim_signed_distance(blob, p, rows)["sd"], "sd")


def _bound_scene(transforms, mesh):
    v, f = mesh
    blob = sc.hostsim.build_blob(v, f)
    t = np.asarray(transforms, np.float32)
    return sc.SimScene([blob], np.zeros(len(t), np.int32), t), sp.flatten_affine([(v, f)], np.zeros(len(t)), t)


def _transform(a, b):
    t = np.zeros((3, 4))
    t[:, :3], t[:, 3] = a, b
    return t


@pytest.mark.parametrize("case", ["random", "scale1e6", "scale1e-6", "offset3e7", "kappa1e4"])
def test_world_bound_exhaustive(case):
    rng = np.random.default_rng(7)
    rot = [spc.rotation(rng) for _ in range(3)]
    if case == "random":
        _, _, t = cases.scene(12, seed=3, coincident=0)
        mesh = synth.icosphere(2)
    else:
        mesh = synth.triangle_soup(200, sigma=0.05, seed=5)
        a = {"scale1e6": [r * 1e6 for r in rot], "scale1e-6": [r * 1e-6 for r in rot], "offset3e7": rot,
             "kappa1e4": [r @ np.diag([1.0, 1e-2, 1e2]) for r in rot]}[case]
        b = {"offset3e7": [np.array([3e7, -2e7, 1e7]) + 3.0 * k for k in range(3)]}.get(case)
        if b is None:
            sz = 1e6 if case == "scale1e6" else (1e-6 if case == "scale1e-6" else 1.0)
            b = [np.array([2.0 * k, -1.0, 0.5]) * sz for k in range(3)]
        t = np.stack([_transform(ai, bi) for ai, bi in zip(a, b)])
    s, (fv, ff, _, _) = _bound_scene(t, mesh)
    lo, hi = spc.scene_box(fv)
    size = float((hi - lo).max())
    p = np.concatenate([spc.uniform_points(lo - 0.2 * size, hi + 0.2 * size, 60, seed=2),
                        spc.surface_points(fv, ff, 60, seed=3, offset=1e-4)])
    viol, checked, worst = sp.bound_check(s, p)
    print(f"{case}: {checked} slot/subtree pairs, worst bound / d2 = {worst:.9f}")
    assert checked > 1000 and viol == 0
    assert worst < 1.0
    # and the walk still gives the brute-force answer
    _same(sp.closest_point(s, p), sp.closest_point(s, p, mode="brute"), case)


def test_sigma_bounds_singular_value():
    rng = np.random.default_rng(11)
    ts, rotations = [], []
    for k in range(200):
        r = spc.rotation(rng)
        if k % 2 == 0:
            a = r * float(10.0 ** rng.uniform(-6, 6)) * (-1.0 if k % 4 == 0 else 1.0)
            rotations.append(True)
        else:
            a = r @ np.diag(10.0 ** rng.uniform(-2, 2, size=3)) @ spc.rotation(rng)
            rotations.append(False)
        ts.append(_transform(a, rng.uniform(-10, 10, size=3)))
    _, inst_mesh, t = None, np.zeros(len(ts), np.int32), np.asarray(ts, np.float32)
    s = sc.SimScene([sc.hostsim.build_blob(*synth.icosphere(1))], inst_mesh, t)
    sigma = sp.point_side(s)[:, 0].astype(np.float64)
    smin = np.array([np.linalg.svd(x[:, :3].astype(np.float64), compute_uv=False).min() for x in t])
    assert (sigma <= smin).all()
    rot = np.asarray(rotations)
    assert (sigma[rot] >= (1.0 - 2.0 ** -20) * smin[rot]).all()
    assert (sigma[~rot] > 0.5 * smin[~rot]).all()


def test_side_of_identity_and_empty():
    ms, inst_mesh, t = cases.scene(20, seed=1, coincident=0)
    s = sc.SimScene(_blobs(ms), inst_mesh, t)
    side = sp.point_side(s)
    empty = inst_mesh == 3
    assert (side[empty] == 0).all() and (side[~empty, 0] > 0).all()
    s1 = sc.SimScene([sc.hostsim.build_blob(*synth.icosphere(1))], [0], np.eye(4, dtype=np.float32)[None, :3])
    assert 1.0 - 2.0 ** -24 <= sp.point_side(s1)[0, 0] <= 1.0   # rounded down below the exact 1


@pytest.fixture(scope="module")
def sign_case():
    ms, inst_mesh, t = spc.sign_scene(seed=0)
    s = sc.SimScene(_blobs(ms), inst_mesh, t)
    rows = [pn.sim_normals(b)[0] for b in s.blobs]
    fv, ff, fi, _ = sp.flatten_affine(ms, inst_mesh, t)
    p, owner = spc.sign_points(ms, inst_mesh, t, per_instance=100)
    d, inside = pn.truth(fv, spc.outward_faces(ff, fi, t), p)
    diag = np.array([np.linalg.norm(np.ptp(np.asarray(ms[int(m)][0], np.float64) @ t[i, :, :3].T, axis=0))
                     for i, m in enumerate(inst_mesh)])
    keep = d > 1e-4 * diag[owner]
    return s, rows, p[keep], inside[keep], d[keep]


def test_sign_matches_binary64_truth(sign_case):
    s, rows, p, inside, d = sign_case
    got = sp.closest_point(s, p, normals=rows)
    assert len(p) > 1000 and inside.sum() > 100 and (~inside).sum() > 100
    np.testing.assert_array_equal(got["sd"] > 0, inside)
    # binary32 world coordinates: the error scales with |p| as well as with d
    assert (np.abs(np.abs(got["sd"]) - d) <= 1e-4 * d + 1e-6 * np.abs(p).max(1)).all()
    _same(got, sp.closest_point(s, p, normals=rows, mode="brute"), "sign/brute")


def test_mirrored_instance_negative_outside_positive_inside():
    v, f = synth.icosphere(3)
    for a in (np.diag([-1.0, 1.0, 1.0]), np.diag([2.0, -2.0, -2.0]), -np.eye(3) * 0.5):
        s = sc.SimScene([sc.hostsim.build_blob(v, f)], [0], _transform(a, [1.0, 2.0, 3.0])[None].astype(np.float32))
        rows = [pn.sim_normals(s.blobs[0])[0]]
        r = float(abs(a[0, 0]))
        p = np.array([[1.0, 2.0, 3.0], [1.0 + 0.5 * r, 2.0, 3.0], [1.0 + 2 * r, 2.0, 3.0], [1.0, 2.0 - 3 * r, 3.0]],
                     np.float32)
        sd = sp.closest_point(s, p, normals=rows)["sd"]
        assert (sd[:2] > 0).all() and (sd[2:] < 0).all(), (a, sd)


def test_flatten_affine_matches_kernel_world_vertices(big_scene):
    ms, inst_mesh, t, s, fv, ff, pts = big_scene
    got = sp.closest_point(s, pts["surface"])
    ok = got["inst"] >= 0
    off = _face_offsets(ms, inst_mesh)
    tri = fv[ff[off[got["inst"][ok]] + got["tri"][ok]]]
    w = got["uv"][ok]
    approx = w[:, :1] * tri[:, 0] + w[:, 1:2] * tri[:, 1] + (1 - w.sum(1, keepdims=True)) * tri[:, 2]
    scale = np.abs(fv).max()
    np.testing.assert_allclose(approx, got["closest"][ok], atol=1e-5 * scale)
