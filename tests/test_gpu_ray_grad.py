"""Hit gradient on the GPU (rt_ray_grad and the autograd functions of RayMeshIntersector's ray queries): grad_origins,
grad_directions and grad_vertices against the host simulator bit for bit for dense, compacted and all-hits rows
(including the true-size config-2 and config-4 meshes, several row windows and deep-overlap scenes up to 64 hits per
ray), repeatability, batch layouts, a finite-difference check of a depth loss through the float32 kernels, unchanged
forward bits, double backward and a small fit."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "raygrad"))
import deep_overlap_cases as DO  # noqa: E402
import raygrad as R  # noqa: E402
from test_closest_point_logic import MESHES  # noqa: E402
from test_ray_grad_logic import random_rays  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

pytestmark = pytest.mark.gpu


def make(v, f, **kw):
    return RayMeshIntersector(vertices=torch.from_numpy(np.ascontiguousarray(v)),
                              faces=torch.from_numpy(np.ascontiguousarray(f)), **kw)


def bits_equal(a, b, what):
    a = np.ascontiguousarray(a, dtype=np.float32); b = np.ascontiguousarray(b, dtype=np.float32)
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ (first at {np.argwhere(bad)[0]})"


def same(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def rows_of(r, o, d, mode):
    """(tri [h], ray_idx [h] or None) of the forward in one of the three row layouts"""
    if mode == "allhits":
        _, ray_idx, tri = hops.intersects_location(r.as_wrapper, o, d, r.max_hits)
        return tri, ray_idx
    hit, front, tri, loc, uv = hops.intersects_closest(r.as_wrapper, o, d)
    if mode == "compact":
        _, ray_idx, tri, _, _ = hops.compact_closest(hit, front, tri, loc, uv)
        return tri, ray_idx
    return tri.reshape(-1), None


def gpu_vs_sim(r, o, d, mode, seed=0, workspace_bytes=None, window=0, what="", rows=None):
    ot, dt = torch.from_numpy(np.ascontiguousarray(o)).cuda(), torch.from_numpy(np.ascontiguousarray(d)).cuda()
    tri, ray_idx = rows_of(r, ot, dt, mode) if rows is None else rows
    h = tri.shape[0]
    rng = np.random.default_rng(seed)
    gl = rng.normal(size=(h, 3)).astype(np.float32)
    gu = None if mode == "allhits" else rng.normal(size=(h, 2)).astype(np.float32)
    go, gd, gv = hops.ray_grad(ot, dt, tri, torch.from_numpy(gl).cuda(), None if gu is None else torch.from_numpy(gu).cuda(),
                               r.mesh_vertices, r.mesh_faces, ray_idx=ray_idx, workspace_bytes=workspace_bytes)
    so, sd, sv = R.sim_grad(o, d, tri.cpu().numpy(), gl, gu, r.mesh_vertices.cpu().numpy(), r.mesh_faces.cpu().numpy(),
                            None if ray_idx is None else ray_idx.cpu().numpy(), window)
    bits_equal(go.cpu().numpy(), so, f"{what} {mode}: grad_origins")
    bits_equal(gd.cpu().numpy(), sd, f"{what} {mode}: grad_directions")
    bits_equal(gv.cpu().numpy(), sv, f"{what} {mode}: grad_vertices")
    return go, gd, gv


MODES = ["dense", "compact", "allhits"]


@pytest.mark.parametrize("name", list(MESHES))
@pytest.mark.parametrize("mode", MODES)
def test_cuda_matches_hostsim(cuda_device, name, mode):
    v, f = MESHES[name]
    o, d = random_rays(v, 4000, np.random.default_rng(7))
    gpu_vs_sim(make(v, f), o, d, mode, what=name)


@pytest.mark.parametrize("cfg", ["config2_icosphere", "config4_soup"])
def test_cuda_matches_hostsim_true_size(cuda_device, cfg):
    v, f = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000)}[cfg]()
    r = make(v, f)
    o, d = random_rays(v, 200_000, np.random.default_rng(17))
    for mode in MODES:
        gpu_vs_sim(r, o, d, mode, seed=18, what=cfg)


@pytest.mark.parametrize("scene", list(DO.SCENES))
@pytest.mark.parametrize("max_hits", [1, 8, 64])
def test_deep_overlap_all_hits(cuda_device, scene, max_hits):
    v, f = DO.scene(scene)
    o, d = DO.rays(scene, "pooled")
    r = make(v, f, max_hits=max_hits)
    gpu_vs_sim(r, o, d, "allhits", seed=max_hits, what=scene)
    if max_hits == 8:
        gpu_vs_sim(r, o, d, "compact", seed=3, what=scene)


def window_of(n, n_verts, workspace_bytes):
    """the window rt_ray_grad picks: the largest whose workspace fits"""
    lo, hi = 0, n + 1
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if hops.ray_grad_workspace_bytes(mid, n_verts) <= workspace_bytes else (lo, mid)
    return lo


def test_windows_and_repeatability(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f, max_hits=16)
    o, d = random_rays(v, 300_000, np.random.default_rng(3))
    for mode in ("dense", "allhits"):
        # the same rows twice (the all-hits forward lists a ray's hits in traversal order, which may vary by run)
        rows = rows_of(r, torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), mode)
        g1 = gpu_vs_sim(r, o, d, mode, seed=4, what="one window", rows=rows)
        g2 = gpu_vs_sim(r, o, d, mode, seed=4, what="again", rows=rows)
        assert all(same(a, b) for a, b in zip(g1, g2))
        n_rows = int(rows[0].shape[0])
        for ws in (hops.ray_grad_workspace_bytes(100_000, len(v)) + 1000, hops.ray_grad_workspace_bytes(7777, len(v))):
            w = window_of(n_rows, len(v), ws)
            assert w < n_rows
            gpu_vs_sim(r, o, d, mode, seed=4, workspace_bytes=ws, window=w, what=f"window {w}", rows=rows)
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    tri, _ = rows_of(r, ot, dt, "dense")
    with pytest.raises(ValueError, match="workspace"):
        hops.ray_grad(ot, dt, tri, torch.ones(len(o), 3, device="cuda"), None, r.mesh_vertices, r.mesh_faces,
                      workspace_bytes=1024)


def leaf(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda().requires_grad_()


def test_autograd_matches_ray_grad_and_forward_bits(cuda_device):
    v, f = synth.icosphere(4)
    verts = torch.from_numpy(v).cuda().requires_grad_()
    r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
    o, d = random_rays(v, 50_000, np.random.default_rng(5))
    ot, dt = leaf(o), leaf(d)
    plain = r.intersects_closest(ot.detach(), dt.detach())
    with torch.no_grad():
        nog = r.intersects_closest(ot, dt)
    tracked = r.intersects_closest(ot, dt)
    assert all(x.grad_fn is None for x in nog)
    assert tracked[3].grad_fn is not None and tracked[4].grad_fn is not None
    assert not any(x.requires_grad for x in tracked[:3])
    for a, b, c in zip(plain, nog, tracked):
        eq = same if a.dtype == torch.float32 else torch.equal
        assert eq(a, b) and eq(a, c.detach())
    gl = torch.randn_like(tracked[3])
    gu = torch.randn_like(tracked[4])
    ((tracked[3] * gl).sum() + (tracked[4] * gu).sum()).backward()
    want = hops.ray_grad(ot.detach(), dt.detach(), plain[2], gl, gu, verts.detach(), r.mesh_faces)
    assert same(ot.grad, want[0]) and same(dt.grad, want[1]) and same(verts.grad, want[2])
    # compacted: the same rows through ray_idx
    for x in (ot, dt, verts):
        x.grad = None
    hit, front, ray_idx, tri_c, loc_c, uv_c = r.intersects_closest(ot, dt, stream_compaction=True)
    assert torch.equal(loc_c.detach(), plain[3][plain[0]]) and torch.equal(uv_c.detach(), plain[4][plain[0]])
    (loc_c * gl[plain[0]]).sum().backward()
    want = hops.ray_grad(ot.detach(), dt.detach(), tri_c, gl[plain[0]].contiguous(), None, verts.detach(), r.mesh_faces,
                         ray_idx=ray_idx)
    assert same(ot.grad, want[0]) and same(dt.grad, want[1]) and same(verts.grad, want[2])
    # all hits through intersects_location and intersects_id
    for x in (ot, dt, verts):
        x.grad = None
    loc, ray_idx, tri = r.intersects_location(ot, dt)
    tri_i, ray_i, loc_i = r.intersects_id(ot, dt, return_locations=True)
    assert torch.equal(loc.detach(), loc_i.detach()) and torch.equal(ray_idx, ray_i) and torch.equal(tri, tri_i)
    g = torch.randn_like(loc)
    (loc * g).sum().backward()
    want = hops.ray_grad(ot.detach(), dt.detach(), tri, g, None, verts.detach(), r.mesh_faces, ray_idx=ray_idx)
    assert same(ot.grad, want[0]) and same(dt.grad, want[1]) and same(verts.grad, want[2])
    _, _, loc1 = r.intersects_id(ot, dt, return_locations=True, multiple_hits=False)
    assert loc1.grad_fn is not None and torch.equal(loc1.detach(), plain[3][plain[0]])
    # interpolate() is differentiable through uv
    for x in (ot, dt, verts):
        x.grad = None
    attr = torch.randn(len(v), 4, device="cuda")
    _, _, tri_d, _, uv_d = r.intersects_closest(ot, dt)
    m = tri_d >= 0
    r.interpolate(attr, tri_d[m], uv_d[m]).sum().backward()
    assert ot.grad is not None and torch.isfinite(ot.grad).all() and (ot.grad[~m] == 0).all() and ot.grad[m].abs().sum() > 0
    # the pinhole query has no gradient
    pin = r.intersects_closest_pinhole(torch.eye(3), torch.tensor([0.0, 0.0, 3.0]), 8, 8, 8.0)
    assert all(x.grad_fn is None for x in pin)


def test_batch_layouts(cuda_device):
    v, f = synth.icosphere(3)
    r = make(v, f)
    rng = np.random.default_rng(1)
    base_o = leaf(rng.uniform(-0.3, 0.3, (6, 5, 4, 3, 3)) + np.float32([0, 0, 3]))
    base_d = leaf(np.broadcast_to(np.float32([0.05, -0.02, -1]), (6, 5, 4, 3, 3)) + rng.normal(0, 0.1, (6, 5, 4, 3, 3)))
    r.intersects_closest(base_o, base_d)[3].square().sum().backward()
    ref_o, ref_d = base_o.grad.clone(), base_d.grad.clone()
    assert ref_o.abs().sum() > 0
    for name, view in (("strided", lambda x: x.transpose(1, 2)), ("sliced", lambda x: x[:, ::2, 1:])):
        base_o.grad = base_d.grad = None
        r.intersects_closest(view(base_o), view(base_d))[3].square().sum().backward()
        for got, ref in ((base_o.grad, ref_o), (base_d.grad, ref_d)):
            want = torch.zeros_like(ref)
            view(want).copy_(view(ref))
            assert same(got, want), name
    # one origin broadcast over many directions: autograd sums the rays' gradients
    one = leaf([0.01, 0.02, 3.0])
    dirs = leaf(np.float32([0, 0, -1]) + rng.normal(0, 0.15, (7, 9, 3)))
    loc = r.intersects_closest(one.expand(7, 9, 3), dirs)[3]
    loc.sum().backward()
    each = leaf(np.broadcast_to(np.float32([0.01, 0.02, 3.0]), (7, 9, 3)))
    r.intersects_closest(each, dirs.detach())[3].sum().backward()
    torch.testing.assert_close(one.grad, each.grad.sum((0, 1)), rtol=1e-5, atol=1e-5)
    empty_o, empty_d = leaf(np.zeros((0, 3))), leaf(np.zeros((0, 3)))
    r.intersects_closest(empty_o, empty_d)[3].sum().backward()
    assert empty_o.grad.shape == (0, 3)
    loc, _, _ = r.intersects_location(empty_o, empty_d)
    loc.sum().backward()


def test_rays_that_all_miss(cuda_device):
    """compacted and all-hits queries where no ray hits: zero rows (an empty ray_idx), all-zero gradients"""
    v, f = synth.icosphere(2)
    verts = torch.from_numpy(v).cuda().requires_grad_()
    r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
    o = leaf(np.tile(np.float32([[5.0, 0.0, 0.0]]), (100, 1)) + np.random.default_rng(8).normal(0, 0.1, (100, 3)))
    d = leaf(np.tile(np.float32([[1.0, 0.0, 0.0]]), (100, 1)))
    outs = {"compact": lambda: r.intersects_closest(o, d, stream_compaction=True)[4],
            "location": lambda: r.intersects_location(o, d)[0],
            "id all hits": lambda: r.intersects_id(o, d, return_locations=True)[2],
            "id closest": lambda: r.intersects_id(o, d, return_locations=True, multiple_hits=False)[2]}
    for name, fn in outs.items():
        for x in (o, d, verts):
            x.grad = None
        loc = fn()
        assert loc.shape == (0, 3) and loc.grad_fn is not None, name
        loc.sum().backward()
        for x in (o, d, verts):
            assert x.grad.shape == x.shape and (x.grad == 0).all() and not torch.signbit(x.grad).any(), name


def test_depth_loss_finite_differences(cuda_device):
    """d/d(o, d, V) of sum ((loc - o) . d) through the float32 kernels against central differences of the same
    kernels, on rays aimed at the middle of the large triangles of an icosahedron"""
    v, f = synth.icosphere(0)
    rng = np.random.default_rng(2)
    n = 2000
    tri = rng.integers(0, len(f), n)
    bc = rng.dirichlet([6, 6, 6], n)
    keep = (bc > 0.15).all(1)
    tgt = (bc[keep, :, None] * v[f[tri[keep]]].astype(np.float64)).sum(1)
    o = tgt * 2.5 + rng.normal(0, 0.1, tgt.shape)
    d = (tgt - o) / np.linalg.norm(tgt - o, axis=1, keepdims=True)
    verts = torch.from_numpy(v).cuda().requires_grad_()
    r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
    ot, dt = leaf(o), leaf(d)
    hit, _, tri_t, loc, _ = r.intersects_closest(ot, dt)
    assert hit.all() and torch.equal(tri_t.cpu(), torch.from_numpy(tri[keep].astype(np.int32)))
    ((loc - ot) * dt).sum(1).sum().backward()

    def depth(oo, dd, vv):
        r2 = RayMeshIntersector(vertices=vv, faces=torch.from_numpy(f))
        with torch.no_grad():
            _, _, t2, l2, _ = r2.intersects_closest(oo, dd)
            assert torch.equal(t2, tri_t)
            return ((l2 - oo) * dd).sum(1).double()

    h = 1e-3
    o0, d0, v0 = ot.detach(), dt.detach(), verts.detach()
    for a in range(3):
        e = torch.zeros(3, device="cuda"); e[a] = h
        fd_o = (depth(o0 + e, d0, v0) - depth(o0 - e, d0, v0)) / (2 * h)
        fd_d = (depth(o0, d0 + e, v0) - depth(o0, d0 - e, v0)) / (2 * h)
        torch.testing.assert_close(ot.grad[:, a].double(), fd_o, atol=2e-2, rtol=2e-2)
        torch.testing.assert_close(dt.grad[:, a].double(), fd_d, atol=2e-2, rtol=2e-2)
    for j in range(len(v)):
        for a in range(3):
            hi, lo = v0.clone(), v0.clone()
            hi[j, a] += h; lo[j, a] -= h
            fd = float((depth(o0, d0, hi) - depth(o0, d0, lo)).sum() / (2 * h))
            assert abs(float(verts.grad[j, a]) - fd) <= 2e-2 * max(1.0, abs(fd)), (j, a, float(verts.grad[j, a]), fd)


def test_double_backward_raises(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    o, d = random_rays(v, 200, np.random.default_rng(9))
    ot = leaf(o)
    w = torch.ones(len(o), 3, device="cuda", requires_grad=True)
    (go,) = torch.autograd.grad((r.intersects_closest(ot, torch.from_numpy(d).cuda())[3] * w).sum(), ot,
                                create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        go.sum().backward()


def test_adam_fit_to_an_ellipsoid_depth_image(cuda_device):
    """Vertices of an icosphere fitted with Adam and a refit per step to the depth image of an ellipsoid seen from three
    sides: the mean squared depth error over pixels that hit both meshes drops by at least 4x in 40 steps."""
    v, f = synth.icosphere(3)
    target = make((v * np.float32([1.2, 1.0, 0.8])).astype(np.float32), f)
    s = np.linspace(-1.0, 1.0, 48)
    gx, gy = np.meshgrid(s, s)
    o_list, d_list = [], []
    for axis in range(3):
        o = np.zeros((gx.size, 3)); d = np.zeros((gx.size, 3))
        o[:, (axis + 1) % 3] = gx.reshape(-1); o[:, (axis + 2) % 3] = gy.reshape(-1); o[:, axis] = 3.0
        d[:, axis] = -1.0
        o_list.append(o); d_list.append(d)
    o = torch.from_numpy(np.concatenate(o_list).astype(np.float32)).cuda()
    d = torch.from_numpy(np.concatenate(d_list).astype(np.float32)).cuda()
    hit_t, _, _, loc_t, _ = target.intersects_closest(o, d)
    depth_t = ((loc_t - o) * d).sum(1)
    verts = torch.from_numpy(v).cuda().requires_grad_()
    r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
    opt = torch.optim.Adam([verts], lr=0.01)
    losses = []
    for _ in range(41):
        opt.zero_grad()
        hit, _, _, loc, _ = r.intersects_closest(o, d)
        m = hit & hit_t
        loss = (((loc - o) * d).sum(1) - depth_t)[m].square().mean()
        loss.backward()
        losses.append(float(loss.detach()))
        opt.step()
        r.refit(verts)
    assert losses[-1] * 4 < losses[0], losses
