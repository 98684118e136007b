"""Gradients of instanced-scene queries on the CPU (DESIGN.md §4.13): the host simulator of rt_scene_grad.cu (the
kernels' own RT_HD code) against a numpy restatement of the contract, bit for bit; against the single-mesh
simulators on the scene flattened with the kernels' binary32 world vertices, bit for bit; against central
differences of the binary64 contract; the translation and direction-scaling identities; and row windows."""
import os
import sys

import numpy as np
import pytest

_T = os.path.dirname(os.path.abspath(__file__))
for _d in ("scene", "scenegrad", "raygrad", "distgrad", "pseudonormal"):
    sys.path.insert(0, os.path.join(_T, _d))
import distgrad as dg  # noqa: E402
import pseudonormal as pn  # noqa: E402
import raygrad as rg  # noqa: E402
import scenegrad as sg  # noqa: E402
import scenepoint as sp  # noqa: E402
import scene_cases as cases  # noqa: E402
import scene_point_cases as spc  # noqa: E402
from helpers import assert_bits_equal  # noqa: E402
from triro import synth  # noqa: E402


@pytest.fixture(scope="module")
def big():
    """scene(300): non-uniform scales, mirrors, coincident copies and an empty mesh; its flattened mesh; hit rows
    of random and camera rays and point rows of uniform, surface and special points from the simulators."""
    ms, inst_mesh, t = cases.scene(300, seed=0)
    gs = sg.SimGradScene(ms, inst_mesh, t)
    fv, ff, fi, fr = sp.flatten_affine(ms, inst_mesh, t)
    off = np.concatenate([[0], np.cumsum([len(ms[int(m)][1]) for m in inst_mesh])]).astype(np.int64)
    vbase = np.concatenate([[0], np.cumsum([len(ms[int(m)][0]) for m in inst_mesh])]).astype(np.int64)
    o1, d1 = cases.rays(600, seed=5)
    o2, d2 = cases.camera_rays(24, 18, origin=(0.0, -2.0, 14.0))
    o, d = np.concatenate([o1, o2]), np.concatenate([d1, d2])
    hit = gs.sim.trace("closest", o, d)
    lo, hi = spc.scene_box(fv)
    pts = np.concatenate([spc.uniform_points(lo, hi, 300, seed=0), spc.surface_points(fv, ff, 300, seed=1),
                          spc.special_points(lo, hi)])
    cp = sp.closest_point(gs.sim, pts)
    return dict(ms=ms, inst_mesh=inst_mesh, t=t, gs=gs, fv=fv, ff=ff, off=off, vbase=vbase, o=o, d=d, hit=hit,
                pts=pts, cp=cp)


def _grads(rng, n, k):
    return rng.normal(size=(n, k)).astype(np.float32)


def _bad_point_rows(b, rng):
    """the point rows plus rows with inst / tri out of range, a NaN point and a value of 0 and of inf"""
    p, cp = b["pts"].copy(), {k: v.copy() for k, v in b["cp"].items()}
    n_inst = len(b["inst_mesh"])
    live = np.flatnonzero(cp["inst"] >= 0)[:6]
    cp["inst"][live[0]] = n_inst
    cp["tri"][live[1]] = 10 ** 6
    cp["inst"][live[2]] = -5
    p[live[3]] = np.nan
    cp["distance"][live[4]] = 0.0
    cp["distance"][live[5]] = np.inf
    return p, cp


@pytest.mark.parametrize("window", [0, 97])
def test_point_rows_equal_the_restated_contract(big, window):
    rng = np.random.default_rng(1)
    p, cp = _bad_point_rows(big, rng)
    g = rng.normal(size=len(p)).astype(np.float32)
    gs = big["gs"]
    got = gs.point_grad(p, g, cp["distance"], cp["closest"], cp["inst"], cp["tri"], cp["uv"], window=window)
    ref = sg.restate_point(gs, p, g, cp["distance"], cp["closest"], cp["inst"], cp["tri"], cp["uv"], window=window)
    for a, r, what in zip(got, ref, ("grad_points", "grad_transforms", "grad_vertices")):
        assert_bits_equal(a, r, what)
    assert np.abs(got[1]).sum() > 0 and np.abs(got[2]).sum() > 0
    assert np.isfinite(got[1]).all() and np.isfinite(got[2]).all()
    # the empty mesh's instance and the dead rows contribute nothing
    assert (got[1][big["inst_mesh"].tolist().index(3)] == 0).all()


def test_point_rows_equal_the_single_mesh_simulator_on_the_flattened_mesh(big):
    """grad_points is §4.9's bit for bit; the flattened vertex gradient, chained to each instance by
    sum_v grad_W (x) (v, 1), is the scene's transform gradient to float tolerance."""
    rng = np.random.default_rng(2)
    cp, p, gs = big["cp"], big["pts"], big["gs"]
    g = rng.normal(size=len(p)).astype(np.float32)
    gp, gt, _ = gs.point_grad(p, g, cp["distance"], cp["closest"], cp["inst"], cp["tri"], cp["uv"])
    f = np.where(cp["inst"] >= 0, big["off"][np.maximum(cp["inst"], 0)] + cp["tri"], -1).astype(np.int32)
    rp, rv = dg.sim_grad(p, g, cp["distance"], cp["closest"], f, cp["uv"], big["ff"], len(big["fv"]))
    assert_bits_equal(gp, rp, "grad_points")
    _check_chain(big, rv, gt)


def _check_chain(b, grad_w, gt):
    ref = np.zeros_like(gt, dtype=np.float64)
    for i, m in enumerate(b["inst_mesh"]):
        v = np.asarray(b["ms"][int(m)][0], np.float64).reshape(-1, 3)
        gw = np.asarray(grad_w[b["vbase"][i]:b["vbase"][i] + len(v)], np.float64)
        ref[i, :, :3] = gw.T @ v
        ref[i, :, 3] = gw.sum(0)
    scale = np.abs(ref).max()
    np.testing.assert_allclose(gt, ref, rtol=1e-4, atol=1e-5 * scale)


def _hit_rows(b, rng, extra=True):
    h = b["hit"]
    inst, tri = h["inst"].copy(), h["tri"].copy()
    if extra:
        live = np.flatnonzero(inst >= 0)[:3]
        inst[live[0]] = len(b["inst_mesh"])
        tri[live[1]] = -7
    n = len(inst)
    return inst, tri, _grads(rng, n, 3), _grads(rng, n, 2)


def test_hit_rows_equal_the_single_mesh_simulator_on_the_flattened_mesh(big):
    """lambda, t lambda, q, w and grad_o / grad_d of every row are rt_ray_grad's on the flattened mesh, bit for bit;
    x and q_obj are the restated binary32 sequences; grad [A|b] is the chained flattened vertex gradient."""
    rng = np.random.default_rng(3)
    inst, tri, gl, gu = _hit_rows(big, rng, extra=False)
    gs, o, d = big["gs"], big["o"], big["d"]
    f = np.where(inst >= 0, big["off"][np.maximum(inst, 0)] + tri, -1).astype(np.int32)
    rows = gs.hit_rows(o, d, inst, tri, gl, gu)
    lam, tlam, q, w, live = rg.sim_rows(o, d, f, gl, gu, big["fv"], big["ff"])
    for k, r in (("lam", lam), ("tlam", tlam), ("q", q), ("w", w)):
        assert_bits_equal(rows[k], r, k)
    np.testing.assert_array_equal(rows["live"], live)
    assert live.sum() > 300
    recs = gs.sim.records()
    for j in np.flatnonzero(live)[:200]:
        m = int(big["inst_mesh"][inst[j]])
        v = np.asarray(big["ms"][m][0], np.float32)[big["ms"][m][1][tri[j]]]
        w0, w1 = rows["w"][j]
        w2 = np.float32(np.float32(1.0 - w0) - w1)
        x = ((w0 * v[0]).astype(np.float32) + (w1 * v[1]).astype(np.float32)).astype(np.float32)
        x = (x + (w2 * v[2]).astype(np.float32)).astype(np.float32)
        assert_bits_equal(rows["x"][j], x, "x")
        fw = recs[inst[j], :12]
        qo = [sg._affine_row(fw[k], fw[4 + k], fw[8 + k], np.float32(-0.0), *rows["q"][j]) for k in range(3)]
        assert_bits_equal(rows["qo"][j], np.array(qo, np.float32), "q_obj")
    go, gd, gt, _ = gs.ray_grad(o, d, inst, tri, gl, gu)
    rgo, rgd, rgv = rg.sim_grad(o, d, f, gl, gu, big["fv"], big["ff"])
    assert_bits_equal(go, rgo, "grad_origins")
    assert_bits_equal(gd, rgd, "grad_directions")
    _check_chain(big, rgv, gt)


@pytest.mark.parametrize("window", [0, 50])
def test_hit_rows_and_windows_equal_the_restated_sums(big, window):
    """transform and vertex sums of hit rows (bad rows included, compacted with row_ray) from the simulator's own
    per-row factors, restated with numpy and distgrad's tree order per window, bit for bit"""
    rng = np.random.default_rng(4)
    inst, tri, gl, gu = _hit_rows(big, rng)
    keep = np.flatnonzero(big["hit"]["hit"] > 0)
    gs, o, d = big["gs"], big["o"], big["d"]
    row_ray = keep.astype(np.int32)
    inst, tri, gl, gu = inst[keep], tri[keep], gl[keep], gu[keep]
    _, _, gt, gv = gs.ray_grad(o, d, inst, tri, gl, gu, row_ray=row_ray, window=window)
    rows = gs.hit_rows(o, d, inst, tri, gl, gu, row_ray=row_ray)
    n_keys = gs.n_verts + 4 * gs.n_inst
    acc = np.zeros((n_keys, 3), np.float32)
    mesh_of = gs.sim.records()[:, 24].view(np.int32)
    h = len(tri)
    win = h if window <= 0 else window
    for base in range(0, h, win):
        lists = {}
        for j in range(base, min(h, base + win)):
            if not rows["live"][j]:
                continue
            m = int(mesh_of[inst[j]])
            idx = gs.meshes[m][1][tri[j]]
            w = rows["w"][j]
            ws = (w[0], w[1], np.float32(np.float32(1.0 - w[0]) - w[1]))
            for k in range(3):
                lists.setdefault(int(gs.base[m] + idx[k]), []).append((-ws[k] * rows["qo"][j]).astype(np.float32))
            for c in range(4):
                val = (-rows["x"][j][c] * rows["q"][j]).astype(np.float32) if c < 3 else -rows["q"][j]
                lists.setdefault(gs.n_verts + 4 * int(inst[j]) + c, []).append(val)
        for key, cs in lists.items():
            acc[key] = (acc[key] + sg.tree_sum(np.stack(cs))).astype(np.float32)
    assert_bits_equal(gv, acc[:gs.n_verts], "grad_vertices")
    assert_bits_equal(gt, acc[gs.n_verts:].reshape(-1, 4, 3).transpose(0, 2, 1), "grad_transforms")


def test_outputs_are_independent(big):
    """transforms alone, vertices alone and both give the same bits (each key's list is the same)"""
    rng = np.random.default_rng(5)
    inst, tri, gl, gu = _hit_rows(big, rng)
    gs, o, d = big["gs"], big["o"], big["d"]
    _, _, gt, gv = gs.ray_grad(o, d, inst, tri, gl, gu, outputs=3)
    _, _, gt1, gv1 = gs.ray_grad(o, d, inst, tri, gl, gu, outputs=sg.TRANSFORMS)
    _, _, gt2, gv2 = gs.ray_grad(o, d, inst, tri, gl, gu, outputs=sg.VERTICES)
    assert_bits_equal(gt, gt1, "transforms only")
    assert_bits_equal(gv, gv2, "vertices only")
    assert not gv1.any() and not gt2.any()


def test_scaling_directions_halves_grad_d_only(big):
    rng = np.random.default_rng(6)
    inst, tri, gl, gu = _hit_rows(big, rng)
    gs, o, d = big["gs"], big["o"], big["d"]
    a = gs.ray_grad(o, d, inst, tri, gl, gu)
    b = gs.ray_grad(o, 2 * d, inst, tri, gl, gu)
    assert_bits_equal(b[0], a[0], "grad_origins")
    assert_bits_equal(b[1], a[1] / 2, "grad_directions")
    assert_bits_equal(b[2], a[2], "grad_transforms")
    assert_bits_equal(b[3], a[3], "grad_vertices")


def test_translation_identities(big):
    """grad b_i = -sum grad_points over the instance's points; for hit rows grad b_i = sum (g_L - grad_o)"""
    rng = np.random.default_rng(7)
    gs, cp, p = big["gs"], big["cp"], big["pts"]
    g = rng.normal(size=len(p)).astype(np.float32)
    gp, gt, _ = gs.point_grad(p, g, cp["distance"], cp["closest"], cp["inst"], cp["tri"], cp["uv"])
    ref = np.zeros((gs.n_inst, 3))
    ok = cp["inst"] >= 0
    np.add.at(ref, cp["inst"][ok], -gp[ok].astype(np.float64))
    np.testing.assert_allclose(gt[:, :, 3], ref, rtol=1e-5, atol=1e-5)
    inst, tri, gl, gu = _hit_rows(big, rng, extra=False)
    go, _, gt, _ = gs.ray_grad(big["o"], big["d"], inst, tri, gl, gu)
    ref = np.zeros((gs.n_inst, 3))
    ok = inst >= 0
    np.add.at(ref, inst[ok], (gl[ok] - go[ok]).astype(np.float64))
    np.testing.assert_allclose(gt[:, :, 3], ref, rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------ finite differences of the binary64 contract
def _fd_scene(seed=0):
    """a star prism and a notched cube under a rotation, non-uniform scale, shear and mirror each"""
    rng = np.random.default_rng(seed)
    ms = [pn.star_prism(), pn.notched_cube()]
    ts = []
    for k in range(4):
        a = spc.rotation(rng) @ np.diag(rng.uniform(0.5, 2.0, 3))
        a = a @ np.array([[1, 0.3 * (k % 2), 0], [0, 1, 0.2], [0, 0, 1]])
        if k in (1, 2):
            a[:, 0] *= -1
        t = np.zeros((3, 4))
        t[:, :3], t[:, 3] = a, rng.uniform(-3, 3, 3) + 8.0 * k
        ts.append(t)
    return ms, np.array([0, 1, 0, 1], np.int32), np.asarray(ts, np.float32)


def _world(ms, inst_mesh, t64, verts64, i, tri):
    m = int(inst_mesh[i])
    v = verts64[m][np.asarray(ms[m][1])[tri]]
    return v @ t64[i, :, :3].T + t64[i, :, 3]


def _fd_check(analytic, f, x0, idx, eps_rel=1e-6):
    x0 = np.asarray(x0, np.float64)
    num = []
    for k in idx:
        h = eps_rel * max(1.0, abs(x0.flat[k]))
        xp, xm = x0.copy(), x0.copy()
        xp.flat[k] += h
        xm.flat[k] -= h
        num.append((f(xp) - f(xm)) / (2 * h))
    num = np.array(num)
    got = np.asarray(analytic, np.float64).reshape(-1)[idx]
    np.testing.assert_allclose(got, num, rtol=1e-4, atol=1e-4 * np.abs(num).max())


def test_point_gradients_match_central_differences():
    """distance to each point's fixed world triangle, interior rows only (barycentrics >= 0.05): grad A, grad b and
    the member vertices against binary64 central differences, relative tolerance 1e-4"""
    ms, inst_mesh, t = _fd_scene()
    gs = sg.SimGradScene(ms, inst_mesh, t)
    fv, ff, fi, fr = sp.flatten_affine(ms, inst_mesh, t)
    rng = np.random.default_rng(1)
    pts = spc.surface_points(fv, ff, 400, seed=4, offset=0.05)
    cp = sp.closest_point(gs.sim, pts)
    w2 = 1.0 - cp["uv"].sum(1)
    keep = (cp["inst"] >= 0) & (cp["uv"].min(1) > 0.05) & (w2 > 0.05) & (cp["distance"] > 1e-3)
    pts, cp = pts[keep], {k: v[keep] for k, v in cp.items()}
    assert len(pts) > 50
    g = rng.normal(size=len(pts)).astype(np.float32)
    _, gt, gv = gs.point_grad(pts, g, cp["distance"], cp["closest"], cp["inst"], cp["tri"], cp["uv"])
    verts64 = [np.asarray(v, np.float64) for v, _ in ms]
    p64 = pts.astype(np.float64)

    def loss(t64, vs):
        total = 0.0
        for j in range(len(pts)):
            w = _world(ms, inst_mesh, t64, vs, cp["inst"][j], cp["tri"][j])
            n = np.cross(w[1] - w[0], w[2] - w[0])
            total += g[j] * abs(np.dot(p64[j] - w[0], n)) / np.linalg.norm(n)
        return total

    t64 = t.astype(np.float64)
    _fd_check(gt, lambda x: loss(x.reshape(t.shape), verts64), t64, np.arange(t64.size))
    used = np.unique(np.concatenate([gs.base[int(inst_mesh[i])] + np.asarray(ms[int(inst_mesh[i])][1])[k]
                                     for i, k in zip(cp["inst"], cp["tri"])]))
    flat = np.concatenate(verts64)
    idx = (3 * rng.choice(used, 12, replace=False)[:, None] + np.arange(3)).reshape(-1)

    def vloss(x):
        xs = x.reshape(-1, 3)
        return loss(t64, [xs[gs.base[m]:gs.base[m + 1]] for m in range(len(ms))])

    _fd_check(gv, vloss, flat, idx)


def test_hit_gradients_match_central_differences():
    """world hit location and barycentrics on the fixed world triangle (binary64 Moeller-Trumbore of §4.10), rays
    aimed inside triangles (barycentrics >= 0.05, not grazing: |cos| > 0.3): grad A, grad b, member vertices, origins and directions against
    binary64 central differences, relative tolerance 1e-4"""
    ms, inst_mesh, t = _fd_scene(1)
    gs = sg.SimGradScene(ms, inst_mesh, t)
    fv, ff, fi, fr = sp.flatten_affine(ms, inst_mesh, t)
    rng = np.random.default_rng(2)
    faces = rng.choice(len(ff), 300)
    bary = rng.dirichlet([2, 2, 2], size=300)
    target = (bary[:, :, None] * fv[ff[faces]].astype(np.float64)).sum(1)
    o = (target + rng.normal(size=(300, 3)) * 4.0).astype(np.float32)
    d = (target - o) / np.linalg.norm(target - o, axis=1, keepdims=True)
    d = d.astype(np.float32)
    hit = gs.sim.trace("closest", o, d)
    off = np.concatenate([[0], np.cumsum([len(ms[int(m)][1]) for m in inst_mesh])])
    wt = fv[ff[off[np.maximum(hit["inst"], 0)] + hit["tri"]]].astype(np.float64)
    n = np.cross(wt[:, 1] - wt[:, 0], wt[:, 2] - wt[:, 0])
    cos = np.abs((n * d).sum(1)) / np.linalg.norm(n, axis=1)
    keep = (hit["inst"] >= 0) & (hit["uv"].min(1) > 0.05) & (1.0 - hit["uv"].sum(1) > 0.05) & (cos > 0.3)
    o, d = o[keep], d[keep]
    inst, tri = hit["inst"][keep], hit["tri"][keep]
    assert len(o) > 50
    gl, gu = _grads(rng, len(o), 3), _grads(rng, len(o), 2)
    go, gd, gt, gv = gs.ray_grad(o, d, inst, tri, gl, gu)
    verts64 = [np.asarray(v, np.float64) for v, _ in ms]

    def loss(t64, vs, oo, dd):
        w = np.stack([_world(ms, inst_mesh, t64, vs, inst[j], tri[j]) for j in range(len(o))])
        tt, b1, b2, _, _, _, _ = rg.hit64(oo, dd, w[:, 0], w[:, 1], w[:, 2])
        loc = w[:, 0] * (1 - b1 - b2)[:, None] + w[:, 1] * b1[:, None] + w[:, 2] * b2[:, None]
        uv = np.stack([1 - b1 - b2, b1], 1)
        return float((gl * loc).sum() + (gu * uv).sum())

    t64, o64, d64 = t.astype(np.float64), o.astype(np.float64), d.astype(np.float64)
    _fd_check(gt, lambda x: loss(x.reshape(t.shape), verts64, o64, d64), t64, np.arange(t64.size))
    _fd_check(go, lambda x: loss(t64, verts64, x.reshape(-1, 3), d64), o64, rng.choice(o64.size, 30, replace=False))
    _fd_check(gd, lambda x: loss(t64, verts64, o64, x.reshape(-1, 3)), d64, rng.choice(d64.size, 30, replace=False))
    used = np.unique(np.concatenate([gs.base[int(inst_mesh[i])] + np.asarray(ms[int(inst_mesh[i])][1])[k]
                                     for i, k in zip(inst, tri)]))
    idx = (3 * rng.choice(used, 12, replace=False)[:, None] + np.arange(3)).reshape(-1)

    def vloss(x):
        xs = x.reshape(-1, 3)
        return loss(t64, [xs[gs.base[m]:gs.base[m + 1]] for m in range(len(ms))], o64, d64)

    _fd_check(gv, vloss, np.concatenate(verts64), idx)


def test_det_zero_and_misses_contribute_nothing():
    """a degenerate member triangle (det = 0 for every ray), misses (inst -1) and an identity instance"""
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [2, 0, 0], [3, 0, 0], [4, 0, 0]], np.float32)
    f = np.array([[0, 1, 2], [3, 4, 5]], np.int32)
    t = np.zeros((1, 3, 4), np.float32)
    t[0, :, :3] = np.eye(3)
    gs = sg.SimGradScene([(v, f), (synth.icosphere(1))], np.array([0], np.int32), t)
    o = np.array([[0.2, 0.2, 1.0], [2.5, 0.0, 1.0], [9, 9, 9]], np.float32)
    d = np.array([[0, 0, -1], [0, 0, -1], [0, 0, 1]], np.float32)
    inst = np.array([0, 0, -1], np.int32)
    tri = np.array([0, 1, -1], np.int32)
    gl = np.ones((3, 3), np.float32)
    go, gd, gt, gv = gs.ray_grad(o, d, inst, tri, gl, None)
    assert go[0].any() and not go[1:].any() and not gd[1:].any()
    assert not gv[3:6].any() and gv[:3].any() and not gv[6:].any()
    rows = gs.hit_rows(o, d, inst, tri, gl, None)
    assert rows["live"].tolist() == [True, False, False]
