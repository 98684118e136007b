"""Point queries on instanced scenes on the GPU (rt_scene_point_prepare, rt_scene_closest_point,
rt_scene_signed_distance, RayMeshScene.closest_point / signed_distance): the side array and every output against the
host simulator of rt_scene.cuh bit for bit over batch layouts, windows and max_distance; one identity instance
against RayMeshIntersector; the 300-instance scene against a RayMeshIntersector of the mesh flattened with the
kernels' binary32 world vertices; signs against the binary64 truth; gradients; update() and the stale-member error;
empty scenes, device checks and repeatability."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

_T = os.path.dirname(os.path.abspath(__file__))
for _d in ("scene", "pseudonormal"):
    sys.path.insert(0, os.path.join(_T, _d))
import pseudonormal as pn  # noqa: E402
import scene as sc  # noqa: E402
import scenepoint as sp  # noqa: E402
import scene_cases as cases  # noqa: E402
import scene_point_cases as spc  # noqa: E402
from helpers import assert_bits_equal  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402
from triro.ray.scene import RayMeshScene  # noqa: E402

pytestmark = pytest.mark.gpu


def make(v, f):
    return RayMeshIntersector(vertices=torch.from_numpy(np.ascontiguousarray(v)), faces=torch.from_numpy(np.ascontiguousarray(f)))


def sim_of(scene: RayMeshScene) -> sc.SimScene:
    return sc.SimScene([m.as_wrapper.blob.cpu().numpy() for m in scene.meshes], scene.instance_mesh.numpy(),
                       scene.transforms.numpy())


def gpu_rows(scene: RayMeshScene):
    return [hops.pseudo_normals(m.as_wrapper)[0].cpu().numpy() for m in scene.meshes]


def np_closest(res) -> dict:
    closest, distance, inst, tri, uv = res
    return dict(closest=closest.cpu().numpy().reshape(-1, 3), distance=distance.cpu().numpy().reshape(-1),
                inst=inst.cpu().numpy().reshape(-1), tri=tri.cpu().numpy().reshape(-1), uv=uv.cpu().numpy().reshape(-1, 2))


def check_scene(scene, sim, points, what, max_distance=None, rows=None):
    """closest_point (with uv) and signed_distance of the scene against the simulator on the flattened batch"""
    pn_ = points.reshape(-1, 3).cpu().numpy()
    md = float("inf") if max_distance is None else max_distance
    ref = sp.closest_point(sim, pn_, md)
    got = np_closest(scene.closest_point(points, max_distance, return_uv=True))
    for k in ref:
        assert_bits_equal(got[k], ref[k], f"{what}: {k}")
    if rows is not None:
        sref = sp.closest_point(sim, pn_, normals=rows)
        assert_bits_equal(scene.signed_distance(points).cpu().numpy().reshape(-1), sref["sd"], f"{what}: sd")
    return ref


@pytest.fixture(scope="module")
def big(cuda_device):
    ms, inst_mesh, t = cases.scene(300, seed=0)
    scene = RayMeshScene([make(v, f) for v, f in ms], torch.from_numpy(inst_mesh), torch.from_numpy(t))
    sim = sim_of(scene)
    fv, ff, _, _ = sp.flatten_affine(ms, inst_mesh, t)
    lo, hi = spc.scene_box(fv)
    pts = np.concatenate([spc.uniform_points(lo, hi, 3000, seed=0), spc.surface_points(fv, ff, 3000, seed=1),
                          spc.special_points(lo, hi)])
    return scene, sim, ms, inst_mesh, t, fv, ff, pts


def test_side_array_matches_sim(big):
    scene, sim = big[:2]
    side, _ = scene._point_state(False)
    n = scene.instance_mesh.numel()
    got = side.cpu().numpy().view(np.float32)[: 4 * n].reshape(n, 4)
    assert_bits_equal(got, sp.point_side(sim), "side")


def test_kernels_match_sim(big):
    scene, sim, *_, pts = big
    rows = gpu_rows(scene)
    p = torch.from_numpy(pts).cuda()
    ref = check_scene(scene, sim, p, "dense", rows=rows)
    assert (ref["inst"] >= 0).sum() == len(pts) - 4
    for md in (0.0, 0.3, 2.0):
        check_scene(scene, sim, p, f"max_distance {md}", md)


def test_batch_layouts_and_windows(big):
    scene, sim, *_, pts = big
    rows = gpu_rows(scene)
    base = torch.from_numpy(pts[:4096]).cuda()
    strided = torch.zeros((4096, 5), device="cuda")
    strided[:, 1:4] = base
    check_scene(scene, sim, strided[:, 1:4], "strided", rows=rows)
    check_scene(scene, sim, base.reshape(4, 4, 16, 16, 3), "5-d", rows=rows)
    check_scene(scene, sim, base[7:8].expand(300, 3), "broadcast", rows=rows)
    check_scene(scene, sim, base.t().contiguous().t(), "column-major", 1.0, rows=rows)
    side, normals = scene._point_state(True)
    full = sp.closest_point(sim, pts[:4096], 1.5)
    full_sd = sp.closest_point(sim, pts[:4096], normals=rows)["sd"]
    for first, count in ((0, 100), (1000, 2000), (4000, -1)):
        got = np_closest(hops.scene_closest_point(scene._table, scene._tlas, side, base, 1.5, first, count))
        end = 4096 if count < 0 else first + count
        for k in full:
            assert_bits_equal(got[k], full[k][first:end], f"window {first}+{count}: {k}")
        sd = hops.scene_signed_distance(scene._table, scene._tlas, side, normals, base, first, count)
        assert_bits_equal(sd.cpu().numpy(), full_sd[first:end], f"window {first}+{count}: sd")


def test_identity_instance_equals_intersector(cuda_device):
    for v, f in (synth.icosphere(3), synth.triangle_soup(500, sigma=0.05, seed=2), pn.torus(), pn.notched_cube()):
        rmi = make(v, f)
        scene = RayMeshScene([rmi], [0], np.eye(4, dtype=np.float32)[None])
        lo, hi = v.min(0) - 0.5, v.max(0) + 0.5
        p = torch.from_numpy(np.concatenate([spc.uniform_points(lo, hi, 5000), spc.surface_points(v, f, 5000),
                                             spc.special_points(lo, hi)])).cuda()
        c, d, inst, tri, uv = scene.closest_point(p, return_uv=True)
        rc, rd, rt, ruv = rmi.closest_point(p, return_uv=True)
        for a, b, k in ((c, rc, "closest"), (d, rd, "distance"), (tri, rt, "tri"), (uv, ruv, "uv")):
            assert_bits_equal(a.cpu().numpy(), b.cpu().numpy(), k)
        assert ((inst == 0) == (tri >= 0)).all()
        assert_bits_equal(scene.signed_distance(p).cpu().numpy(), rmi.signed_distance(p, sign="pseudonormal").cpu().numpy(), "sd")


def test_agrees_with_flattened_intersector(big):
    scene, sim, ms, inst_mesh, t, fv, ff, pts = big
    flat = make(fv, ff)
    off = np.concatenate([[0], np.cumsum([len(ms[int(m)][1]) for m in inst_mesh])])
    p = torch.from_numpy(pts).cuda()
    for md in (None, 0.25):
        got = np_closest(scene.closest_point(p, md, return_uv=True))
        rc, rd, rt, ruv = flat.closest_point(p, md, return_uv=True)
        f = np.where(got["inst"] >= 0, off[np.maximum(got["inst"], 0)] + got["tri"], -1)
        assert_bits_equal(f.astype(np.int32), rt.cpu().numpy(), "face")
        for k, r in (("closest", rc), ("distance", rd), ("uv", ruv)):
            assert_bits_equal(got[k], r.cpu().numpy(), k)


def test_sign_matches_binary64_truth(cuda_device):
    ms, inst_mesh, t = spc.sign_scene(seed=0)
    scene = RayMeshScene([make(v, f) for v, f in ms], inst_mesh, t)
    fv, ff, fi, _ = sp.flatten_affine(ms, inst_mesh, t)
    p, owner = spc.sign_points(ms, inst_mesh, t, per_instance=100)
    d, inside = pn.truth(fv, spc.outward_faces(ff, fi, t), p)
    diag = np.array([np.linalg.norm(np.ptp(np.asarray(ms[int(m)][0], np.float64) @ t[i, :, :3].T, axis=0))
                     for i, m in enumerate(inst_mesh)])
    keep = d > 1e-4 * diag[owner]
    sd = scene.signed_distance(torch.from_numpy(p[keep]).cuda()).cpu().numpy()
    assert inside[keep].sum() > 100 and (~inside[keep]).sum() > 100
    np.testing.assert_array_equal(sd > 0, inside[keep])
    assert_bits_equal(sd, sp.closest_point(sim_of(scene), p[keep], normals=gpu_rows(scene))["sd"], "sd vs sim")


def test_mirrored_closed_mesh_negative_outside_positive_inside(cuda_device):
    v, f = synth.icosphere(3)
    for a in (np.diag([-1.0, 1.0, 1.0]), np.diag([2.0, -2.0, -2.0])):
        t = np.zeros((1, 3, 4), np.float32)
        t[0, :, :3], t[0, :, 3] = a, [1.0, 2.0, 3.0]
        scene = RayMeshScene([make(v, f)], [0], t)
        r = float(abs(a[0, 0]))
        p = torch.tensor([[1.0, 2.0, 3.0], [1.0 + 0.5 * r, 2.0, 3.0], [1.0 + 2 * r, 2.0, 3.0], [1.0, 2.0 - 3 * r, 3.0]],
                         device="cuda")
        sd = scene.signed_distance(p)
        assert (sd[:2] > 0).all() and (sd[2:] < 0).all(), (a, sd)


def test_gradients(big):
    scene, *_, pts = big
    p = torch.from_numpy(pts[:2000]).cuda()
    p[:5] = torch.tensor([[np.nan, 0.0, 0.0]] * 5)
    p.requires_grad_(True)
    g = torch.rand(2000, device="cuda")
    closest, distance, inst, tri = scene.closest_point(p)
    assert closest.grad_fn is None or not closest.requires_grad
    (gp,) = torch.autograd.grad((distance * g).sum(), p)
    pd = p.detach()
    ok = torch.isfinite(distance) & (distance > 0)
    want = torch.where(ok[:, None], g[:, None] * (pd - closest) / distance[:, None], torch.zeros_like(pd))
    torch.testing.assert_close(gp, want, rtol=1e-5, atol=1e-6)
    assert (gp[:5] == 0).all()
    sd = scene.signed_distance(p)
    (gs,) = torch.autograd.grad((sd * g).sum(), p)
    s = torch.where(sd < 0, -1.0, 1.0)
    ok = torch.isfinite(sd) & (sd != 0)
    want = torch.where(ok[:, None], (g * s)[:, None] * (pd - closest) / sd.abs()[:, None], torch.zeros_like(pd))
    torch.testing.assert_close(gs, want, rtol=1e-5, atol=1e-6)
    with torch.no_grad():
        assert scene.closest_point(p)[1].grad_fn is None and scene.signed_distance(p).grad_fn is None
    assert_bits_equal(scene.signed_distance(p).detach().cpu().numpy(), scene.signed_distance(pd).cpu().numpy(), "sd grad/no grad")


def test_update_refit_and_stale_members(cuda_device):
    ms = cases.meshes()[:3]
    members = [make(v, f) for v, f in ms]
    inst_mesh = np.arange(30) % 3
    scene = RayMeshScene(members, inst_mesh, cases.random_transforms(30, seed=8))
    p = torch.from_numpy(spc.uniform_points(-8, 8, 5000, seed=4)).cuda()
    before = np_closest(scene.closest_point(p, return_uv=True))
    scene.update(torch.from_numpy(cases.random_transforms(30, seed=9)))
    check_scene(scene, sim_of(scene), p, "new transforms", rows=gpu_rows(scene))
    assert not np.array_equal(np_closest(scene.closest_point(p, return_uv=True))["inst"], before["inst"])
    members[0].refit(torch.from_numpy(ms[0][0]).cuda() * 1.7)
    with pytest.raises(RuntimeError, match="update"):
        scene.closest_point(p)
    with pytest.raises(RuntimeError, match="update"):
        scene.signed_distance(p)
    scene.update()
    check_scene(scene, sim_of(scene), p, "after refit", rows=gpu_rows(scene))


def test_empty_scenes_devices_and_repeatability(cuda_device):
    p = torch.from_numpy(spc.uniform_points(-2, 2, 1000, seed=6)).cuda()
    for scene in (RayMeshScene([cases.meshes()[0]], np.zeros(0, np.int64), np.zeros((0, 3, 4), np.float32)),
                  RayMeshScene([cases.meshes()[3]], [0, 0], np.tile(np.eye(4, dtype=np.float32), (2, 1, 1)))):
        c, d, inst, tri, uv = scene.closest_point(p, return_uv=True)
        assert (inst == -1).all() and (tri == -1).all() and torch.isinf(d).all() and not c.any() and not uv.any()
        sd = scene.signed_distance(p)
        assert (sd == -float("inf")).all()
    scene = RayMeshScene([cases.meshes()[0]], [0], torch.eye(4)[None])
    e = torch.zeros((0, 3), device="cuda")
    assert scene.closest_point(e)[1].shape == (0,) and scene.signed_distance(e).shape == (0,)
    with pytest.raises(ValueError, match="device"):
        scene.closest_point(p.cpu())
    with pytest.raises(ValueError, match="pseudonormal"):
        scene.signed_distance(p, sign="winding")
    with pytest.raises(ValueError, match="max_distance"):
        scene.closest_point(p, -1.0)
    ms, inst_mesh, t = cases.scene(100, seed=2)
    scene = RayMeshScene([make(v, f) for v, f in ms], inst_mesh, t)
    q = torch.from_numpy(spc.uniform_points(-8, 8, 20000, seed=7)).cuda()
    a = np_closest(scene.closest_point(q, return_uv=True))
    sa = scene.signed_distance(q).cpu().numpy()
    for _ in range(2):
        b = np_closest(scene.closest_point(q, return_uv=True))
        for k in a:
            assert_bits_equal(b[k], a[k], f"repeat {k}")
        assert_bits_equal(scene.signed_distance(q).cpu().numpy(), sa, "repeat sd")
