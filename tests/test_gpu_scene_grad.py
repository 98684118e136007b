"""Gradients of instanced-scene queries on the GPU (rt_scene_ray_grad, rt_scene_distance_grad and the autograd of
RayMeshScene.intersects_closest / closest_point / signed_distance): every gradient against the host simulator of
rt_scene_grad.cu bit for bit over batch layouts, row windows and repeat runs; one identity instance against
RayMeshIntersector; autograd behaviour (leaf dtypes and devices, shared members, grad mode, double backward,
update() and in-place changes); empty cases; and two pose fits by gradient descent."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

_T = os.path.dirname(os.path.abspath(__file__))
for _d in ("scene", "scenegrad", "pseudonormal"):
    sys.path.insert(0, os.path.join(_T, _d))
import pseudonormal as pn  # noqa: E402
import scenegrad as sg  # noqa: E402
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


def sim_of(scene: RayMeshScene) -> sg.SimGradScene:
    return sg.SimGradScene([(m.mesh_vertices.cpu().numpy(), m.mesh_faces.cpu().numpy()) for m in scene.meshes],
                           scene.instance_mesh.numpy(), scene.transforms.numpy())


def np_(t):
    return None if t is None else t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def big(cuda_device):
    ms, inst_mesh, t = cases.scene(300, seed=0)
    scene = RayMeshScene([make(v, f) for v, f in ms], inst_mesh, torch.from_numpy(t))
    fv, ff, _, _ = sp.flatten_affine(ms, inst_mesh, t)
    o1, d1 = cases.rays(3000, seed=5)
    o2, d2 = cases.camera_rays(64, 48)
    o = torch.from_numpy(np.concatenate([o1, o2])).cuda()
    d = torch.from_numpy(np.concatenate([d1, d2])).cuda()
    lo, hi = spc.scene_box(fv)
    pts = np.concatenate([spc.uniform_points(lo, hi, 1500, seed=0), spc.surface_points(fv, ff, 1500, seed=1),
                          spc.special_points(lo, hi)])
    return scene, sim_of(scene), o, d, torch.from_numpy(pts).cuda()


def ray_args(scene):
    table, n_verts, _ = scene._grad_members()
    return scene._table, scene.instance_mesh.numel(), table, n_verts


def ray_case(scene, sim, o, d, compact, seed, workspace_bytes=None, window=0, what=""):
    hit, front, inst, tri, loc, uv = scene.intersects_closest(o, d)
    g = torch.Generator(device="cpu").manual_seed(seed)
    rows_ray = None
    inst, tri = inst.reshape(-1), tri.reshape(-1)
    if compact:
        _, rows_ray, tri, _, _ = hops.compact_closest(hit, front, tri, loc.reshape(-1, 3), uv.reshape(-1, 2))
        inst = inst[rows_ray.long()]
    h = tri.numel()
    gl = torch.randn((h, 3), generator=g).cuda()
    gu = torch.randn((h, 2), generator=g).cuda()
    got = hops.scene_ray_grad(*ray_args(scene), o, d, inst, tri, gl, gu, ray_idx=rows_ray,
                              workspace_bytes=workspace_bytes)
    ref = sim.ray_grad(np_(o).reshape(-1, 3), np_(d).reshape(-1, 3), np_(inst), np_(tri), np_(gl), np_(gu),
                       row_ray=np_(rows_ray), window=window)
    for a, r, k in zip(got, ref, ("grad_origins", "grad_directions", "grad_transforms", "grad_vertices")):
        assert_bits_equal(np_(a).reshape(r.shape), r, f"{what}: {k}")
    return got


def point_case(scene, sim, p, signed, seed, workspace_bytes=None, window=0, what=""):
    side, normals = scene._point_state(signed)
    if signed:
        value, closest, inst, tri, uv = hops.scene_signed_distance(scene._table, scene._tlas, side, normals, p,
                                                                   return_closest=True)
    else:
        closest, value, inst, tri, uv = hops.scene_closest_point(scene._table, scene._tlas, side, p)
    g = torch.randn(value.shape, generator=torch.Generator(device="cpu").manual_seed(seed)).cuda()
    got = hops.scene_point_grad(*ray_args(scene), p, g, value, closest, inst, tri, uv, workspace_bytes=workspace_bytes)
    ref = sim.point_grad(np_(p).reshape(-1, 3), np_(g).reshape(-1), np_(value).reshape(-1), np_(closest).reshape(-1, 3),
                         np_(inst).reshape(-1), np_(tri).reshape(-1), np_(uv).reshape(-1, 2), window=window)
    for a, r, k in zip(got, ref, ("grad_points", "grad_transforms", "grad_vertices")):
        assert_bits_equal(np_(a).reshape(r.shape), r, f"{what}: {k}")
    return got


def window_of(n, n_inst, n_verts, workspace_bytes):
    """the window the kernels pick: the largest whose workspace fits"""
    lo, hi = 1, n
    if hops.scene_grad_workspace_bytes(n, n_inst, n_verts, 3) <= workspace_bytes:
        return n
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if hops.scene_grad_workspace_bytes(mid, n_inst, n_verts, 3) <= workspace_bytes else (lo, mid)
    return lo


def test_kernels_equal_the_simulator(big):
    scene, sim, o, d, p = big
    for compact in (False, True):
        a = ray_case(scene, sim, o, d, compact, seed=1, what=f"rays compact={compact}")
        b = ray_case(scene, sim, o, d, compact, seed=1, what="repeat")
        for x, y in zip(a, b):
            assert torch.equal(x, y), "repeat run differs"
        assert a[2].abs().sum() > 0 and a[3].abs().sum() > 0
    for signed in (False, True):
        a = point_case(scene, sim, p, signed, seed=2, what=f"points signed={signed}")
        b = point_case(scene, sim, p, signed, seed=2, what="repeat")
        for x, y in zip(a, b):
            assert torch.equal(x, y), "repeat run differs"


def test_batch_layouts(big):
    scene, sim, o, d, p = big
    n = 2 * 3 * 5 * 40
    o5, d5 = o[:n].reshape(2, 3, 5, 40, 3), d[:n].reshape(2, 3, 5, 40, 3)
    ray_case(scene, sim, o5, d5, True, seed=3, what="5-d")
    ot = o[:n].t().contiguous().t()           # strided [n,3]
    ray_case(scene, sim, ot, d[:n], False, seed=3, what="strided")
    ob = torch.tensor([[0.0, -2.0, 14.0]], device="cuda").expand(n, 3)
    ray_case(scene, sim, ob, d[-n:], True, seed=3, what="broadcast origin")
    point_case(scene, sim, p[:n].reshape(2, 3, 5, 40, 3), False, seed=4, what="5-d points")
    point_case(scene, sim, p[:n].t().contiguous().t(), True, seed=4, what="strided points")


def test_windows(big):
    scene, sim, o, d, p = big
    n_inst, n_verts = scene.instance_mesh.numel(), scene._grad_members()[1]
    h = o.shape[0]
    for ws in (hops.scene_grad_workspace_bytes(1000, n_inst, n_verts, 3),
               hops.scene_grad_workspace_bytes(333, n_inst, n_verts, 3)):
        w = window_of(h, n_inst, n_verts, ws)
        assert w < h
        ray_case(scene, sim, o, d, False, seed=5, workspace_bytes=ws, window=w, what=f"ray window {w}")
        w = window_of(p.shape[0], n_inst, n_verts, ws)
        point_case(scene, sim, p, False, seed=6, workspace_bytes=ws, window=w, what=f"point window {w}")
    with pytest.raises(ValueError, match="workspace"):
        ray_case(scene, sim, o, d, False, seed=5, workspace_bytes=1024)


def test_autograd_equals_the_entry_points(big):
    scene, sim, o, d, p = big
    t = torch.from_numpy(cases.scene(300, seed=0)[2]).cuda().requires_grad_()
    scene.update(t)
    try:
        oo, dd = o.clone().requires_grad_(), d.clone().requires_grad_()
        hit, front, ray_idx, inst, tri, loc, uv = scene.intersects_closest(oo, dd, stream_compaction=True)
        g = torch.Generator(device="cpu").manual_seed(7)
        gl, gu = torch.randn(loc.shape, generator=g).cuda(), torch.randn(uv.shape, generator=g).cuda()
        ((loc * gl).sum() + (uv * gu).sum()).backward()
        ref = sim.ray_grad(np_(o), np_(d), np_(inst), np_(tri), np_(gl), np_(gu), row_ray=np_(ray_idx))
        assert_bits_equal(np_(oo.grad), ref[0], "origins")
        assert_bits_equal(np_(dd.grad), ref[1], "directions")
        assert_bits_equal(np_(t.grad), ref[2], "transforms")
        t.grad = None
        pp = p.clone().requires_grad_()
        sd = scene.signed_distance(pp)
        gs = torch.randn(sd.shape, generator=g).cuda()
        (sd * gs).sum().backward()
        _, closest, inst, tri, uv = hops.scene_signed_distance(scene._table, scene._tlas, *scene._point_state(True), p,
                                                               return_closest=True)
        ref = sim.point_grad(np_(p), np_(gs), np_(sd), np_(closest), np_(inst), np_(tri), np_(uv))
        assert_bits_equal(np_(pp.grad), ref[0], "points")
        assert_bits_equal(np_(t.grad), ref[1], "transforms (signed distance)")
    finally:
        scene.update(t.detach())


def test_identity_instance_equals_the_intersector(cuda_device):
    v, f = synth.icosphere(3)
    o, d = synth.readme_rays(64, device="cuda")
    o, d = o.reshape(-1, 3), d.reshape(-1, 3)
    eye = torch.eye(4)[None]
    for compact in (False, True):
        grads = []
        for use_scene in (False, True):
            verts = torch.from_numpy(v).cuda().requires_grad_()
            r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
            oo, dd = o.clone().requires_grad_(), d.clone().requires_grad_()
            q = RayMeshScene([r], [0], eye).intersects_closest if use_scene else r.intersects_closest
            out = q(oo, dd, stream_compaction=compact)
            loc, uv = out[-2], out[-1]
            g = torch.Generator(device="cpu").manual_seed(1)
            ((loc * torch.randn(loc.shape, generator=g).cuda()).sum() +
             (uv * torch.randn(uv.shape, generator=g).cuda()).sum()).backward()
            grads.append((oo.grad, dd.grad, verts.grad))
        for a, b, k in zip(*grads, ("origins", "directions", "vertices")):
            assert_bits_equal(np_(b), np_(a), f"compact={compact}: {k}")
    pts = torch.from_numpy(np.random.default_rng(0).uniform(-1.5, 1.5, (4000, 3)).astype(np.float32)).cuda()
    for signed in (False, True):
        grads = []
        for use_scene in (False, True):
            verts = torch.from_numpy(v).cuda().requires_grad_()
            r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
            pp = pts.clone().requires_grad_()
            target = RayMeshScene([r], [0], eye) if use_scene else r
            val = target.signed_distance(pp, sign="pseudonormal") if signed else target.closest_point(pp)[1]
            (val * torch.linspace(-1, 1, val.numel(), device="cuda")).sum().backward()
            grads.append((pp.grad, verts.grad))
        for a, b, k in zip(*grads, ("points", "vertices")):
            assert_bits_equal(np_(b), np_(a), f"signed={signed}: {k}")


def _small_scene(transforms):
    v, f = synth.icosphere(2)
    return RayMeshScene([make(v, f)], [0, 0], transforms), (v, f)


def _two_poses():
    t = np.zeros((2, 4, 4))
    t[:, 3, 3] = 1.0
    t[0, :3, :3] = np.diag([1.0, 0.7, 1.3])
    t[1, :3, :3] = spc.rotation(np.random.default_rng(0))
    t[0, :3, 3], t[1, :3, 3] = [-1.5, 0, 0], [1.5, 0.2, 0]
    return t


def test_transform_leaves_and_shared_members(cuda_device):
    """a float64 CPU [I,4,4] leaf and a CUDA float32 [I,3,4] leaf get the same gradient (zero last row for the 4x4);
    a member shared by two instances gets the sum of the gradients of two one-instance scenes"""
    t = _two_poses()
    pts = torch.from_numpy(np.random.default_rng(1).uniform(-3, 3, (3000, 3)).astype(np.float32)).cuda()
    t64 = torch.from_numpy(t).requires_grad_()
    t32 = torch.from_numpy(t[:, :3, :].astype(np.float32)).cuda().requires_grad_()
    grads = []
    for leaf in (t64, t32):
        scene, _ = _small_scene(leaf)
        scene.closest_point(pts)[1].sum().backward()
        grads.append(leaf.grad)
    assert t64.grad.dtype == torch.float64 and t64.grad.device.type == "cpu"
    assert (t64.grad[:, 3, :] == 0).all()
    assert_bits_equal(t64.grad[:, :3, :].float().numpy(), np_(t32.grad), "4x4 float64 leaf vs 3x4 float32 leaf")
    v, f = synth.icosphere(2)
    verts = torch.from_numpy(v).cuda().requires_grad_()
    scene = RayMeshScene([RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))], [0, 0], torch.from_numpy(t))
    scene.closest_point(pts)[1].sum().backward()
    both = verts.grad.clone()
    d0, d1 = scene.closest_point(pts)[2] == 0, scene.closest_point(pts)[2] == 1
    parts = torch.zeros_like(both)
    for i, mask in ((0, d0), (1, d1)):
        verts.grad = None
        s1 = RayMeshScene([RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))], [0],
                          torch.from_numpy(t[i:i + 1]))
        s1.closest_point(pts[mask])[1].sum().backward()
        parts += verts.grad
    torch.testing.assert_close(both, parts, rtol=1e-5, atol=1e-5)


def test_grad_mode_double_backward_update_and_in_place(cuda_device):
    t = torch.from_numpy(_two_poses()).requires_grad_()
    scene, _ = _small_scene(t)
    o, d = synth.readme_rays(32, device="cuda")
    with torch.no_grad():
        ref = scene.intersects_closest(o, d)
    out = scene.intersects_closest(o, d)
    assert out[-2].grad_fn is not None
    for a, b in zip(ref, out):
        assert a.grad_fn is None
        assert torch.equal(a, b.detach())
    with pytest.raises(RuntimeError):
        loc = out[-2]
        (g,) = torch.autograd.grad(loc.sum(), t, create_graph=True)
        g.sum().backward()
    # a backward after update() still differentiates the forward's pose
    pts = torch.from_numpy(np.random.default_rng(2).uniform(-3, 3, (500, 3)).astype(np.float32)).cuda()
    dist = scene.closest_point(pts)[1]
    (expect,) = torch.autograd.grad(scene.closest_point(pts)[1].sum(), t)
    with torch.no_grad():
        t[:, :3, 3] += 0.25
    scene.update(t)
    (after,) = torch.autograd.grad(dist.sum(), t)
    assert torch.equal(expect, after)
    # an in-place change without update() raises
    with torch.no_grad():
        t[:, :3, 3] -= 0.25
    with pytest.raises(RuntimeError, match="update"):
        scene.closest_point(pts)
    with pytest.raises(RuntimeError, match="update"):
        scene.intersects_closest(o, d)
    scene.update(t)
    scene.closest_point(pts)


def test_empty_cases(cuda_device):
    v, f = synth.icosphere(1)
    empty = (np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    verts = torch.from_numpy(v).cuda().requires_grad_()
    ev = torch.zeros((0, 3), device="cuda", requires_grad=True)
    t = torch.eye(4)[None].repeat(2, 1, 1)
    t[1, :3, 3] = 5.0
    t.requires_grad_()
    scene = RayMeshScene([RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f)),
                          RayMeshIntersector(vertices=ev, faces=torch.from_numpy(empty[1]))], [0, 1], t)
    o = torch.tensor([[0.0, 0.0, 50.0]], device="cuda").expand(100, 3).contiguous().requires_grad_()
    d = torch.tensor([[0.0, 0.0, 1.0]], device="cuda").expand(100, 3).contiguous()
    for compact in (False, True):
        out = scene.intersects_closest(o, d, stream_compaction=compact)       # every ray misses
        (out[-2].sum() + out[-1].sum()).backward()
        assert not t.grad.any() and not o.grad.any() and not verts.grad.any()
    pts = torch.tensor([[5.0, 5.0, 5.0]], device="cuda")
    scene.closest_point(pts)[1].sum().backward()
    assert t.grad[1].abs().sum() == 0 and t.grad[0].abs().sum() > 0
    none = RayMeshScene([RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))], np.zeros(0, np.int64),
                        torch.zeros((0, 3, 4), requires_grad=True))
    verts.grad = None
    none.closest_point(pts.requires_grad_())[1].sum().backward()
    assert not pts.grad.any() and not verts.grad.any()


def _rodrigues(w):
    th = torch.sqrt((w * w).sum() + 1e-20)
    k = w / th
    kx = torch.zeros((3, 3), dtype=w.dtype)
    kx[0, 1], kx[0, 2], kx[1, 0], kx[1, 2], kx[2, 0], kx[2, 1] = -k[2], k[1], k[2], -k[0], -k[1], k[0]
    return torch.eye(3, dtype=w.dtype) + torch.sin(th) * kx + (1 - torch.cos(th)) * (kx @ kx)


def _pose(w, b):
    return torch.cat([_rodrigues(w), b[:, None]], 1)[None]


def test_fit_a_rigid_pose_to_surface_points(cuda_device):
    """star prism, points sampled on its surface under a known pose; start 5 degrees and 5 % of the size off,
    minimise mean d^2 with Adam (cosine-annealed learning rate) over axis-angle + translation, update() every step:
    within 150 steps the rotation
    is within 0.2 degrees and the translation within 0.2 % of the size"""
    v, f = pn.star_prism()
    size = float(np.ptp(v, 0).max())
    rng = np.random.default_rng(0)
    w_true = torch.tensor([0.3, -0.2, 0.5], dtype=torch.float64)
    b_true = torch.tensor([0.4, -0.1, 0.2], dtype=torch.float64)
    a = _pose(w_true, b_true)[0].numpy()
    tri = rng.integers(0, len(f), 4000)
    bc = rng.dirichlet([1, 1, 1], 4000)
    obj = (bc[:, :, None] * np.asarray(v, np.float64)[np.asarray(f)[tri]]).sum(1)
    pts = torch.from_numpy((obj @ a[:, :3].T + a[:, 3]).astype(np.float32)).cuda()
    axis = np.array([1.0, 2.0, -1.0]) / np.sqrt(6)
    w = (w_true + torch.from_numpy(axis * np.deg2rad(5.0))).clone().requires_grad_()
    b = (b_true + torch.from_numpy(np.array([1.0, -1.0, 1.0]) / np.sqrt(3) * 0.05 * size)).clone().requires_grad_()
    scene = RayMeshScene([make(v, f)], [0], _pose(w, b))
    opt = torch.optim.Adam([w, b], lr=5e-3)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, 150)
    for step in range(150):
        opt.zero_grad()
        scene.update(_pose(w, b))
        loss = scene.closest_point(pts)[1].square().mean()
        loss.backward()
        opt.step()
        sched.step()
    r_err = torch.linalg.matrix_norm(_rodrigues(w.detach()) - _rodrigues(w_true)) / np.sqrt(2)
    assert float(np.rad2deg(float(r_err))) < 0.2, (w, w_true)
    assert float((b.detach() - b_true).norm()) < 0.002 * size, (b, b_true)


def test_fit_a_translation_to_a_depth_image(cuda_device):
    """an icosphere instance seen by an orthographic depth camera, moved 0.15 off the pose that rendered the target:
    Adam on the translation through intersects_closest's loc brings the mean squared depth error down by 100x and
    its depth within 0.01 in 80 steps"""
    v, f = synth.icosphere(3)
    s = np.linspace(-1.2, 1.2, 64)
    gx, gy = np.meshgrid(s, s)
    o = torch.from_numpy(np.stack([gx.ravel(), gy.ravel(), np.full(gx.size, 5.0)], 1).astype(np.float32)).cuda()
    d = torch.tensor([[0.0, 0.0, -1.0]], device="cuda").expand_as(o).contiguous()
    b_true = torch.tensor([0.1, -0.05, 0.2])
    t_true = torch.eye(4)[None].clone()
    t_true[0, :3, 3] = b_true
    target = RayMeshScene([make(v, f)], [0], t_true)
    hit_t, _, _, _, loc_t, _ = target.intersects_closest(o, d)
    b = (b_true + torch.tensor([0.15, 0.1, -0.1])).requires_grad_()
    scene = RayMeshScene([make(v, f)], [0], t_true)
    opt = torch.optim.Adam([b], lr=0.01)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, 80)
    losses = []
    for _ in range(80):
        opt.zero_grad()
        t = torch.cat([torch.eye(3), b[:, None]], 1)[None]
        scene.update(t)
        hit, _, _, _, loc, _ = scene.intersects_closest(o, d)
        m = hit & hit_t
        loss = (loc[:, 2] - loc_t[:, 2])[m].square().mean()
        loss.backward()
        losses.append(float(loss.detach()))
        opt.step()
        sched.step()
    assert losses[-1] * 100 < losses[0], losses
    assert float((b.detach() - b_true)[2].abs()) < 0.01, b
