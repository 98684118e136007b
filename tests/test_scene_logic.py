"""Instanced scenes on the CPU: the host simulator of rt_scene.cuh (the kernels' own RT_HD code) with its top-level
tree against the brute-force loop over every instance, bit for bit; one identity instance against the single-mesh
traversal; the flattened scene against the binary64 oracle; the transform arithmetic and the input checks."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "scene"))
import scene as sc  # noqa: E402
import scene_cases as cases  # noqa: E402
from helpers import assert_bits_equal, check_closest_vs_truth  # noqa: E402
from oracle import oracle  # noqa: E402


def _blobs(ms):
    return [sc.hostsim.build_blob(v, f) for v, f in ms]


def _same(a: dict, b: dict, what: str):
    assert a.keys() == b.keys()
    for k in a:
        assert_bits_equal(a[k], b[k], f"{what}.{k}")


@pytest.fixture(scope="module")
def big_scene():
    ms, inst_mesh, t = cases.scene(300, seed=0)
    blobs = _blobs(ms)
    return ms, blobs, inst_mesh, t, sc.SimScene(blobs, inst_mesh, t)


def _ray_sets(blobs, inst_mesh, t):
    return {"random": cases.rays(3000, seed=1), "camera": cases.camera_rays(64, 48),
            "box": cases.box_rays(blobs, inst_mesh, t, per_instance=12)}


@pytest.mark.parametrize("mode", ["closest", "any", "count"])
def test_tlas_equals_brute_force(big_scene, mode):
    ms, blobs, inst_mesh, t, s = big_scene
    for name, (o, d) in _ray_sets(blobs, inst_mesh, t).items():
        got = s.trace(mode, o, d)
        _same(got, s.trace(mode, o, d, brute=True), f"{name}/{mode}")
        key = "hit" if mode != "count" else "count"
        assert (got[key] > 0).sum() > len(o) // 20, f"{name}: too few hits to mean anything"
    if mode == "closest":
        res = s.trace("closest", *cases.rays(3000, seed=1))
        assert len(np.unique(res["inst"][res["hit"] == 1])) > 50
        assert not (res["inst"] == inst_mesh.tolist().index(3)).any(), "an instance of the empty mesh was hit"


def test_user_tmax_and_coincident_ties(big_scene):
    ms, blobs, inst_mesh, t, s = big_scene
    o, d = cases.rays(2000, seed=5)
    full = s.trace("closest", o, d)
    for mode in ("closest", "any", "count"):
        _same(s.trace(mode, o, d, tmax=4.0), s.trace(mode, o, d, tmax=4.0, brute=True), f"tmax/{mode}")
    short = s.trace("closest", o, d, tmax=4.0)
    keep = (full["hit"] == 1) & (np.linalg.norm(full["loc"] - o, axis=1) < 3.9)
    assert keep.any() and (short["inst"][keep] == full["inst"][keep]).all()
    # a coincident copy (same mesh, same transform) never wins: ties at equal t go to the smaller instance
    n = len(inst_mesh)
    assert not np.isin(full["inst"], np.arange(n - 8, n)).any()


def test_identity_instance_equals_single_mesh():
    ms = cases.meshes()[:3]
    o, d = cases.rays(4000, seed=7, radius=1.5)
    o[::7] = 0.0
    d[::5, 0] = -0.0
    d[::11, 1] = 0.0
    for v, f in ms:
        blob = sc.hostsim.build_blob(v, f)
        s = sc.SimScene([blob], [0], np.eye(4, dtype=np.float32)[None])
        for mode in ("closest", "any", "count"):
            got = s.trace(mode, o, d)
            ref = sc.hostsim.trace(blob, mode, o, d)
            for k in got:
                if k != "inst":
                    assert_bits_equal(got[k], ref[k], f"identity/{mode}.{k}")
            if mode == "closest":
                assert_bits_equal(got["inst"], np.where(ref["hit"] == 1, 0, -1).astype(np.int32), "identity inst")


def test_affine_row_identity_keeps_signed_zero_inf_nan():
    xyz = np.array([[-0.0, 1.0, np.inf], [0.0, -np.inf, np.nan], [np.nan, -0.0, 0.0], [1e-45, -3.0, 2.0]], np.float32)
    nz = np.float32(-0.0)
    for k in range(3):
        m = np.zeros(4, np.float32)
        m[k] = 1.0
        m[3] = nz
        assert_bits_equal(sc.affine_row(m, xyz), np.ascontiguousarray(xyz[:, k]), f"row {k}")


def test_prepared_records():
    ms = cases.meshes()
    blobs = _blobs(ms)
    t = cases.random_transforms(40, seed=4)
    inst_mesh = np.arange(40, dtype=np.int32) % 4
    s = sc.SimScene(blobs, inst_mesh, t)
    rec = s.records()
    flags = rec[:, 25].view(np.uint32)
    det = np.linalg.det(t[:, :, :3].astype(np.float64))
    assert ((flags & 1) == (det < 0)).all()
    assert ((flags & 2) != 0).tolist() == (inst_mesh == 3).tolist()
    inv = rec[:, 12:24].reshape(-1, 3, 4).astype(np.float64)
    a = t[:, :, :3].astype(np.float64)
    ref_inv = np.linalg.inv(a)
    assert np.abs(inv[:, :, :3] - ref_inv).max() <= 1e-6 * np.abs(ref_inv).max()
    ref_c = -np.einsum("nij,nj->ni", ref_inv, t[:, :, 3].astype(np.float64))
    assert np.abs(inv[:, :, 3] - ref_c).max() <= 1e-5 * max(1.0, np.abs(ref_c).max())
    # the world box holds the transformed mesh box; the top-level vertices are (lo, hi)
    lo, hi = rec[:, 26:29], rec[:, 29:32]
    assert_bits_equal(s.tlas_v[0::2], np.ascontiguousarray(lo), "tlas lo")
    assert_bits_equal(s.tlas_v[1::2], np.ascontiguousarray(hi), "tlas hi")
    for i, m in enumerate(inst_mesh):
        v = np.asarray(ms[m][0], np.float64)
        if len(v) == 0:
            assert_bits_equal(lo[i], t[i, :, 3], "empty box"); continue
        w = v @ a[i].T + t[i, :, 3]
        assert (w.min(0) >= lo[i]).all() and (w.max(0) <= hi[i]).all()
    assert (s.tlas_f == np.stack([2 * np.arange(40), 2 * np.arange(40) + 1, 2 * np.arange(40)], 1)).all()


def test_identity_offset_and_transform_are_exact():
    blob = sc.hostsim.build_blob(*cases.meshes()[0])
    s = sc.SimScene([blob], [0], np.eye(4, dtype=np.float32)[None])
    rec = s.records()[0]
    assert_bits_equal(rec[12:24], np.array([1, 0, 0, -0.0, 0, 1, 0, -0.0, 0, 0, 1, -0.0], np.float32), "identity inverse")


@pytest.mark.parametrize("bad", ["singular", "nan", "inf", "mesh", "overflow"])
def test_invalid_instances_are_refused(bad):
    blobs = _blobs(cases.meshes()[:1])
    t = np.eye(4, dtype=np.float32)[None, :3].copy()
    m = np.zeros(1, np.int32)
    if bad == "singular":
        t[0, 2, :3] = t[0, 0, :3] + t[0, 1, :3]
    elif bad == "nan":
        t[0, 1, 3] = np.nan
    elif bad == "inf":
        t[0, 0, 1] = np.inf
    elif bad == "mesh":
        m[0] = 1
    else:
        t[0, :, :3] *= np.float32(1e-39)
    with pytest.raises(ValueError):
        sc.SimScene(blobs, m, t)


def test_empty_scene_and_empty_mesh():
    blobs = _blobs(cases.meshes())
    o, d = cases.rays(500, seed=3)
    s = sc.SimScene(blobs, np.zeros(0, np.int32), np.zeros((0, 3, 4), np.float32))
    r = s.trace("closest", o, d)
    assert (r["hit"] == 0).all() and (r["inst"] == -1).all() and (r["tri"] == -1).all() and not r["loc"].any()
    assert (s.trace("count", o, d)["count"] == 0).all() and (s.trace("any", o, d)["hit"] == 0).all()
    s = sc.SimScene(blobs, np.array([3, 3], np.int32), np.tile(np.eye(4, dtype=np.float32)[:3], (2, 1, 1)))
    assert (s.trace("count", o, d)["count"] == 0).all()


def test_many_instances_of_one_mesh():
    v, f = cases.meshes()[0]
    blob = sc.hostsim.build_blob(v, f)
    n = 512
    g = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(8), indexing="ij"), -1).reshape(-1, 3) * 2.5 - 8.75
    t = np.tile(np.eye(4, dtype=np.float32)[:3], (n, 1, 1))
    t[:, :, 3] = g
    s = sc.SimScene([blob], np.zeros(n, np.int32), t)
    o, d = cases.rays(3000, seed=9, radius=12.0)
    for mode in ("closest", "count"):
        _same(s.trace(mode, o, d), s.trace(mode, o, d, brute=True), mode)
    r = s.trace("closest", o, d)
    assert len(np.unique(r["inst"][r["hit"] == 1])) > 100


@pytest.mark.parametrize("seed", [0, 1])
def test_flattened_scene_against_truth(seed):
    ms, inst_mesh, t = cases.scene(60, seed=seed, coincident=0)
    blobs = _blobs(ms)
    s = sc.SimScene(blobs, inst_mesh, t)
    fv, ff, fi, fr = sc.flatten(ms, inst_mesh, t)
    base = np.zeros(len(inst_mesh), np.int64)
    base[1:] = np.cumsum([len(ms[m][1]) for m in inst_mesh])[:-1]
    mesh = oracle.OracleMesh(fv, ff)
    for o, d in (cases.rays(3000, seed=11 + seed), cases.camera_rays(48, 32)):
        got = s.trace("closest", o, d)
        flat = dict(got)
        flat["tri"] = np.where(got["hit"] == 1, base[np.maximum(got["inst"], 0)] + got["tri"], -1).astype(np.int32)
        check_closest_vs_truth(flat, mesh, o, d)
        ref = oracle.query(mesh, o, d, oracle.TRUTH, want=("hit", "t", "flags", "count"))
        both = (ref["flags"] == 0) & (ref["hit"] == 1)
        t_got = np.linalg.norm(got["loc"][both] - o[both], axis=1) / np.linalg.norm(d[both], axis=1)
        assert np.abs(t_got - ref["t"][both]).max() <= 1e-5 * max(1.0, np.abs(fv).max())
        cnt = s.trace("count", o, d)["count"]
        clean = ref["flags"] == 0
        assert (cnt[clean] == ref["count"][clean]).all()
