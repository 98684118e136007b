"""Distance gradient on the GPU (rt_distance_grad, rt_signed_distance_closest, the autograd functions of
RayMeshIntersector): grad_points and grad_vertices against the host simulator bit for bit (including the true-size
config-2 and config-4 meshes, several point windows and 2^24 points on one vertex), repeatability, all three sign
modes, batch layouts, float64 host vertices, refit, max_distance misses, |grad| = 1, unchanged forward bits, double
backward and a small fit."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "distgrad"))
import distgrad as D  # noqa: E402
from helpers import window_of  # noqa: E402
from test_closest_point_logic import MESHES, sample_points  # noqa: E402
from test_gpu_closest_point import distributions  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

pytestmark = pytest.mark.gpu


def make(v, f):
    return RayMeshIntersector(vertices=torch.from_numpy(np.ascontiguousarray(v)), faces=torch.from_numpy(np.ascontiguousarray(f)))


def bits_equal(a, b, what):
    a = np.ascontiguousarray(a, dtype=np.float32); b = np.ascontiguousarray(b, dtype=np.float32)
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ (first at {np.argwhere(bad)[0]})"


def same(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def gpu_vs_sim(r, p, g, signed=False, workspace_bytes=None, window=0, what=""):
    pt = torch.from_numpy(np.ascontiguousarray(p)).cuda()
    if signed:
        value, c, t, uv = hops.signed_distance_pseudonormal(r.as_wrapper, pt, return_closest=True)
    else:
        c, value, t, uv = hops.closest_point(r.as_wrapper, pt)
    gt = torch.from_numpy(g).cuda()
    nv = r.mesh_vertices.shape[0]
    gp, gv = hops.distance_grad(pt, gt, value, c, t, uv, r.mesh_faces, nv, workspace_bytes=workspace_bytes)
    sp, sv = D.sim_grad(p, g, value.cpu().numpy(), c.cpu().numpy(), t.cpu().numpy(), uv.cpu().numpy(),
                        r.mesh_faces.cpu().numpy(), nv, window)
    bits_equal(gp.cpu().numpy(), sp, f"{what}: grad_points")
    bits_equal(gv.cpu().numpy(), sv, f"{what}: grad_vertices")
    return gp, gv


@pytest.mark.parametrize("name", list(MESHES))
@pytest.mark.parametrize("signed", [False, True])
def test_cuda_matches_hostsim(cuda_device, name, signed):
    v, f = MESHES[name]
    rng = np.random.default_rng(7)
    p = sample_points(v, 4000, rng)
    gpu_vs_sim(make(v, f), p, rng.normal(size=len(p)).astype(np.float32), signed, what=name)


@pytest.mark.parametrize("cfg", ["config2_icosphere", "config4_soup"])
def test_cuda_matches_hostsim_true_size(cuda_device, cfg):
    v, f = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000)}[cfg]()
    r = make(v, f)
    p = np.concatenate(list(distributions(v, 100_000, np.random.default_rng(17)).values()))
    g = np.random.default_rng(18).normal(size=len(p)).astype(np.float32)
    gpu_vs_sim(r, p, g, False, what=cfg)
    gpu_vs_sim(r, p, g, True, what=cfg + " signed")


def test_windows_and_repeatability(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    rng = np.random.default_rng(3)
    p = np.concatenate([sample_points(v, 200_000, rng), rng.uniform(-3, 3, (100_000, 3)).astype(np.float32)])
    g = rng.normal(size=len(p)).astype(np.float32)
    gp1, gv1 = gpu_vs_sim(r, p, g, what="one window")
    pt, gt = torch.from_numpy(p).cuda(), torch.from_numpy(g).cuda()
    c, d, t, uv = hops.closest_point(r.as_wrapper, pt)
    gp2, gv2 = hops.distance_grad(pt, gt, d, c, t, uv, r.mesh_faces, len(v))
    assert same(gp1, gp2) and same(gv1, gv2)
    for ws in (hops.distance_grad_workspace_bytes(100_000, len(v)) + 1000, hops.distance_grad_workspace_bytes(7777, len(v))):
        w = window_of(len(p), lambda k: hops.distance_grad_workspace_bytes(k, len(v)), ws)
        assert w < len(p)
        gpu_vs_sim(r, p, g, workspace_bytes=ws, window=w, what=f"window {w}")
    with pytest.raises(ValueError, match="workspace"):
        hops.distance_grad(pt, gt, d, c, t, uv, r.mesh_faces, len(v), workspace_bytes=1024)


def test_every_point_on_one_vertex(cuda_device):
    v, f = synth.cube(0.5)
    r = make(v, f)
    rng = np.random.default_rng(4)
    n = 1 << 24
    p = (v[6].astype(np.float64) + 0.1 + rng.uniform(0, 2, (n, 3))).astype(np.float32)     # beyond (+, +, +)
    g = np.full(n, 1.0 / n, np.float32)
    gp, gv = gpu_vs_sim(r, p, g, what="2^24 points on one corner")
    gv = gv.cpu().numpy()
    assert (gv[np.arange(8) != 6] == 0).all()
    np.testing.assert_allclose(gv[6], -gp.double().sum(0).cpu().numpy(), rtol=1e-5)


def leaf(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda().requires_grad_()


@pytest.mark.parametrize("sign", ["contains", "winding", "pseudonormal"])
def test_sign_modes_and_unit_gradient(cuda_device, sign):
    v, f = synth.icosphere(4)
    r = make(v, f)
    rng = np.random.default_rng(5)
    p = leaf(rng.uniform(-1.5, 1.5, (50_000, 3)))
    sd = r.signed_distance(p, sign=sign)
    with torch.no_grad():
        assert same(sd, r.signed_distance(p, sign=sign))
    sd.sum().backward()
    c, d, t, uv = hops.closest_point(r.as_wrapper, p.detach())
    want = (p.detach() - c) / d[:, None] * torch.where(torch.signbit(sd.detach()), -1.0, 1.0)[:, None]
    torch.testing.assert_close(p.grad, want, atol=1e-6, rtol=0)
    pos = d > 0
    assert ((p.grad[pos].double().norm(dim=1) - 1).abs() < 1e-5).all()
    if sign == "pseudonormal":
        gp, _ = hops.distance_grad(p.detach(), torch.ones_like(sd), sd.detach(),
                                   *hops.signed_distance_pseudonormal(r.as_wrapper, p.detach(), return_closest=True)[1:],
                                   r.mesh_faces, len(v), vertices_grad=False)
        assert same(p.grad, gp)


def test_forward_bits_unchanged(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    p = leaf(np.random.default_rng(6).uniform(-1.3, 1.3, (100_000, 3)))
    plain = r.closest_point(p.detach(), return_uv=True)
    with torch.no_grad():
        nog = r.closest_point(p, return_uv=True)
    tracked = r.closest_point(p, return_uv=True)
    assert tracked[1].grad_fn is not None and nog[1].grad_fn is None
    for a, b, c in zip(plain, nog, tracked):
        assert same(a, b) and same(a, c.detach())
    assert not any(x.requires_grad for i, x in enumerate(tracked) if i != 1)
    sd = hops.signed_distance_pseudonormal(r.as_wrapper, p.detach())
    sd2, c2, t2, uv2 = hops.signed_distance_pseudonormal(r.as_wrapper, p.detach(), return_closest=True)
    assert same(sd, sd2) and same(c2, plain[0]) and same(t2, plain[2]) and same(uv2, plain[3])
    assert same(r.signed_distance(p, sign="pseudonormal").detach(), sd)
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    hops.signed_distance_pseudonormal(r.as_wrapper, p.detach(), counters=cnt, return_closest=True)
    cnt2 = torch.zeros(4, dtype=torch.int64, device="cuda")
    hops.signed_distance_pseudonormal(r.as_wrapper, p.detach(), counters=cnt2)
    assert cnt.tolist() == cnt2.tolist()


def test_batch_layouts(cuda_device):
    v, f = synth.icosphere(3)
    r = make(v, f)
    base = leaf(np.random.default_rng(1).uniform(-1.2, 1.2, (6, 5, 4, 3, 3)))
    r.closest_point(base)[1].square().sum().backward()
    ref = base.grad.clone()
    for name, view in (("strided", lambda x: x.transpose(1, 2)), ("sliced", lambda x: x[:, ::2, 1:])):
        base.grad = None
        r.signed_distance(view(base), sign="pseudonormal").square().sum().backward()
        want = torch.zeros_like(ref)
        view(want).copy_(view(ref))
        assert same(base.grad, want), name
    one = leaf([0.1, 0.2, 0.3])
    r.closest_point(one.expand(7, 9, 3))[1].sum().backward()
    single = leaf([[0.1, 0.2, 0.3]])
    r.closest_point(single)[1].sum().backward()
    torch.testing.assert_close(one.grad, 63 * single.grad[0], rtol=1e-6, atol=0)
    empty = leaf(np.zeros((0, 3)))
    r.closest_point(empty)[1].sum().backward()
    assert empty.grad.shape == (0, 3)


def test_host_float64_vertices_refit_and_misses(cuda_device):
    v, f = synth.icosphere(3)
    v64 = torch.from_numpy(v.astype(np.float64)).requires_grad_()
    r = RayMeshIntersector(vertices=v64, faces=torch.from_numpy(f))
    rng = np.random.default_rng(2)
    p = torch.from_numpy(rng.uniform(-2, 2, (20_000, 3)).astype(np.float32)).cuda()
    _, d, _ = r.closest_point(p, max_distance=0.5)
    miss = torch.isinf(d)
    assert miss.any() and not miss.all()
    d[~miss].sum().backward()
    assert v64.grad is not None and v64.grad.dtype == torch.float64 and not v64.grad.is_cuda
    c, d2, t, uv = hops.closest_point(r.as_wrapper, p, 0.5)
    g = (~miss).float()
    _, gv = hops.distance_grad(p, g, d2, c, t, uv, r.mesh_faces, len(v), points_grad=False)
    assert torch.equal(v64.grad, gv.double().cpu())
    pg = p.clone().requires_grad_()
    r.closest_point(pg, max_distance=0.5)[1][~miss].sum().backward()
    assert (pg.grad[miss] == 0).all()
    # refit to moved vertices, then backward: the gradients of a fresh intersector on the moved mesh
    v2 = torch.from_numpy((v * np.float32([1.2, 0.9, 1.1])).astype(np.float32)).cuda().requires_grad_()
    r.refit(v2)
    r.signed_distance(p, sign="pseudonormal").sum().backward()
    v3 = v2.detach().clone().requires_grad_()
    make_r = RayMeshIntersector(vertices=v3, faces=torch.from_numpy(f))
    make_r.signed_distance(p, sign="pseudonormal").sum().backward()
    assert same(v2.grad, v3.grad)


def test_double_backward_raises(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    p = leaf(np.random.default_rng(9).uniform(-1.5, 1.5, (100, 3)))
    w = torch.ones(100, device="cuda", requires_grad=True)        # a grad_out that itself requires grad
    (gp,) = torch.autograd.grad((r.closest_point(p)[1] * w).sum(), p, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gp.sum().backward()
    sd = r.signed_distance(p, sign="pseudonormal")
    (gp,) = torch.autograd.grad((sd * w).sum(), p, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gp.sum().backward()


def test_adam_fit_to_an_ellipsoid(cuda_device):
    """Vertices of an icosphere fitted to points on an ellipsoid with Adam and a refit per step: the mean squared
    distance drops by at least 50x in 40 steps (the host simulator of the same loop: ~180x)."""
    v, f = synth.icosphere(3)
    d = np.random.default_rng(0).normal(size=(20_000, 3))
    target = torch.from_numpy((d / np.linalg.norm(d, axis=1, keepdims=True) * [1.3, 1.0, 0.7]).astype(np.float32)).cuda()
    verts = torch.from_numpy(v).cuda().requires_grad_()
    r = RayMeshIntersector(vertices=verts, faces=torch.from_numpy(f))
    opt = torch.optim.Adam([verts], lr=0.01)
    losses = []
    for _ in range(41):
        opt.zero_grad()
        loss = r.closest_point(target)[1].square().mean()
        loss.backward()
        losses.append(float(loss.detach()))
        opt.step()
        r.refit(verts)
    assert losses[-1] * 50 < losses[0], losses
