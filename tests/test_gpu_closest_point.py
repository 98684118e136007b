"""Closest-point query on the GPU (rt_closest_point): CUDA against the binary32 MIRROR oracle and the host simulator
bit for bit, batch layouts, max_distance semantics, refit / save / load, the instrumented variant, signed distance,
interpolation at closest points and the numpy adapter."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import pointquery as pq  # noqa: E402
from test_closest_point_logic import MESHES, box_distance, sample_points  # noqa: E402
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


def gpu_query(r, p, max_distance=None):
    c, d, t, uv = r.closest_point(torch.from_numpy(np.ascontiguousarray(p)).cuda(), max_distance, return_uv=True)
    return dict(closest=c.cpu().numpy(), distance=d.cpu().numpy(), tri=t.cpu().numpy(), uv=uv.cpu().numpy())


def check_equal(got, ref, what):
    assert np.array_equal(got["tri"], ref["tri"]), f"{what}: {int((got['tri'] != ref['tri']).sum())} triangle ids differ"
    for k in ("closest", "distance", "uv"):
        bits_equal(got[k], ref[k], f"{what}.{k}")


def distributions(v, n, rng):
    """(a) jittered around the surface, (b) uniform in the 1.2x box, (c) a row-major grid over the 1.2x box."""
    good = v[np.isfinite(v).all(axis=1)].astype(np.float64)
    lo, hi = good.min(0), good.max(0)
    c, h = 0.5 * (lo + hi), 0.6 * (hi - lo)
    diag = float(np.linalg.norm(hi - lo))
    a = good[rng.integers(0, len(good), n)] + rng.normal(0.0, 0.01 * diag, (n, 3))
    b = rng.uniform(c - h, c + h, (n, 3))
    g = int(round(n ** (1 / 3)))
    axes = [np.linspace(c[k] - h[k], c[k] + h[k], g) for k in range(3)]
    grid = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3)
    return {"surface": a.astype(np.float32), "uniform": b.astype(np.float32), "grid": grid.astype(np.float32)}


@pytest.mark.parametrize("name", list(MESHES))
def test_cuda_matches_mirror_and_hostsim(cuda_device, name):
    v, f = MESHES[name]
    r = make(v, f)
    m = pq.PointMesh(v, f)
    rng = np.random.default_rng(5)
    pts = distributions(v, 60_000, rng)
    pts["vertices"] = sample_points(v, 4000, rng)
    blob = r.as_wrapper.blob.cpu().numpy()
    for kind, p in pts.items():
        got = gpu_query(r, p)
        check_equal(got, pq.query(m, p, pq.MIRROR), f"{name}/{kind} vs mirror")
        sim = pq.sim_closest_point(blob, p[:5000])
        check_equal({k: x[:5000] for k, x in got.items()}, sim, f"{name}/{kind} vs hostsim on the GPU blob")


@pytest.mark.parametrize("cfg", ["config2_icosphere", "config3_heightfield", "config4_soup"])
def test_cuda_matches_mirror_true_size(cuda_device, cfg):
    v, f = {"config2_icosphere": lambda: synth.icosphere(7), "config3_heightfield": lambda: synth.heightfield(2048, 1024),
            "config4_soup": lambda: synth.triangle_soup(1_000_000)}[cfg]()
    r = make(v, f)
    m = pq.PointMesh(v, f, use_bvh=True)
    rng = np.random.default_rng(17)
    for kind, p in distributions(v, 1_000_000 // 3, rng).items():
        check_equal(gpu_query(r, p), pq.query(m, p, pq.MIRROR), f"{cfg}/{kind}")


def same(a, b):
    """bitwise equality (float outputs compared as bit patterns)"""
    if a.dtype == torch.float32:
        a, b = a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)
    return a.shape == b.shape and torch.equal(a, b)


def test_batch_layouts(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    base = torch.from_numpy(np.random.default_rng(1).uniform(-1.5, 1.5, (6, 5, 4, 3, 3)).astype(np.float32)).cuda()
    ref = r.closest_point(base.contiguous(), return_uv=True)
    for name, x in (("5-d", base), ("strided", base.transpose(1, 2)), ("sliced", base[:, ::2, 1:, :, :])):
        got = r.closest_point(x, return_uv=True)
        want = r.closest_point(x.contiguous(), return_uv=True)
        assert got[0].shape == (*x.shape[:-1], 3) and got[1].shape == x.shape[:-1] and got[3].shape == (*x.shape[:-1], 2)
        for g, w in zip(got, want):
            assert same(g, w), name
    one = torch.tensor([0.3, 1.2, -0.4], device="cuda")
    bc = one.broadcast_to(7, 9, 3)
    got = r.closest_point(bc)
    single = r.closest_point(one[None])
    assert torch.equal(got[2], single[2].expand(7, 9)) and torch.equal(got[1], single[1].expand(7, 9))
    # a window of the flattened batch equals the same slice of the whole
    c, d, t, uv = hops.closest_point(r.as_wrapper, base, ray_first=100, ray_count=57)
    flat = [x.reshape(360, -1) for x in ref]
    assert torch.equal(t, flat[2][100:157].reshape(-1)) and torch.equal(d, flat[1][100:157].reshape(-1))
    del c, uv


def test_empty_inputs_and_miss_convention(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    c, d, t = r.closest_point(torch.zeros(0, 3, device="cuda"))
    assert c.shape == (0, 3) and d.shape == (0,) and t.shape == (0,)
    p = torch.tensor([[np.nan, 0, 0], [0, np.inf, 0], [0.1, 0.2, 3.0]], dtype=torch.float32, device="cuda")
    c, d, t, uv = r.closest_point(p, return_uv=True)
    assert t.tolist()[:2] == [-1, -1] and t.tolist()[2] >= 0
    assert d[:2].cpu().tolist() == [np.inf, np.inf] and not c[:2].any() and not uv[:2].any()
    empty = RayMeshIntersector(vertices=torch.zeros(0, 3), faces=torch.zeros(0, 3, dtype=torch.int32))
    c, d, t, uv = empty.closest_point(p, return_uv=True)
    assert t.tolist() == [-1, -1, -1] and bool(torch.isinf(d).all()) and not c.any() and not uv.any()


def test_max_distance_semantics(cuda_device):
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    r = make(v, np.array([[0, 1, 2]], np.int32))
    p = torch.tensor([[0.25, 0.25, 2.0]], device="cuda")
    assert r.closest_point(p)[2].tolist() == [0]
    assert r.closest_point(p, float("inf"))[2].tolist() == [0]
    assert r.closest_point(p, 2.0)[2].tolist() == [0]
    c, d, t = r.closest_point(p, float(np.nextafter(np.float32(2.0), np.float32(0))))
    assert t.tolist() == [-1] and d.tolist() == [float("inf")]
    for bad in (float("nan"), -1.0):
        with pytest.raises(ValueError):
            r.closest_point(p, bad)
    # the cut-off follows d2 <= fl(m * m) exactly as the mirror does, on a whole batch
    v, f = synth.icosphere(4)
    r = make(v, f)
    pts = np.random.default_rng(2).uniform(-1.4, 1.4, (20000, 3)).astype(np.float32)
    md = 0.2
    check_equal(gpu_query(r, pts, md), pq.query(pq.PointMesh(v, f), pts, pq.MIRROR, md), "max_distance 0.2")


def test_refit_and_save_load(cuda_device, tmp_path):
    v, f = synth.icosphere(4)
    r = make(v, f)
    pts = torch.from_numpy(np.random.default_rng(3).uniform(-1.5, 1.5, (30000, 3)).astype(np.float32)).cuda()
    before = r.closest_point(pts, return_uv=True)
    path = str(tmp_path / "bvh.pt")
    r.save_bvh(path)
    loaded = hops.AccelStructure().load(path)
    after = hops.closest_point(loaded, pts)
    for a, b in zip(before, (after[0], after[1], after[2], after[3])):
        assert torch.equal(a, b)
    v2 = (v * np.float32(1.3) + np.float32(0.1)).astype(np.float32)
    r.refit(torch.from_numpy(v2))
    fresh = make(v2, f)
    for a, b in zip(r.closest_point(pts, return_uv=True), fresh.closest_point(pts, return_uv=True)):
        assert torch.equal(a, b)


def test_repeatable_and_counters(cuda_device):
    v, f = synth.triangle_soup(50000)
    r = make(v, f)
    pts = torch.from_numpy(np.random.default_rng(4).uniform(-1.2, 1.2, (200000, 3)).astype(np.float32)).cuda()
    a = hops.closest_point(r.as_wrapper, pts)
    b = hops.closest_point(r.as_wrapper, pts)
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    c = hops.closest_point(r.as_wrapper, pts, counters=cnt)
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y) and torch.equal(x, z)
    nodes, tris, npts, found = cnt.tolist()
    assert npts == 200000 and found == 200000 and nodes >= npts and tris >= npts
    sim = pq.sim_closest_point(r.as_wrapper.blob.cpu().numpy(), pts[:2000].cpu().numpy())
    hops.closest_point(r.as_wrapper, pts[:2000], counters=cnt)
    assert cnt.tolist() == [sim["stats"]["nodes"], sim["stats"]["tris"], 2000, 2000]   # same traversal, same counts


def test_signed_distance(cuda_device):
    v, f = synth.cube(0.5)
    r = make(v, f)
    p = torch.from_numpy(np.random.default_rng(6).uniform(-1.5, 1.5, (50000, 3)).astype(np.float32)).cuda()
    sd = r.signed_distance(p)
    _, d, _ = r.closest_point(p)
    inside = r.contains_points(p)
    assert torch.equal(sd.abs(), d)
    nz = d != 0
    assert torch.equal((sd[nz] > 0), inside[nz])
    ref = -box_distance(p.cpu().numpy(), 0.5)
    clear = np.abs(ref) > 1e-4
    np.testing.assert_allclose(sd.cpu().numpy()[clear], ref[clear], rtol=1e-6, atol=1e-7)
    corner = torch.tensor([[0.5, 0.5, 0.5]], device="cuda")   # a vertex: distance exactly 0, contains_points says outside
    assert not r.contains_points(corner).item()
    z = r.signed_distance(corner)
    assert z.item() == 0.0 and not torch.signbit(z).item()
    v, f = synth.icosphere(4)
    r = make(v, f)
    q = np.random.default_rng(8).uniform(-1.3, 1.3, (4000, 3)).astype(np.float32)
    sd = r.signed_distance(torch.from_numpy(q).cuda())
    bits_equal(np.abs(sd.cpu().numpy()), pq.query(pq.PointMesh(v, f), q, pq.MIRROR)["distance"], "|signed distance| vs mirror")
    inside = r.contains_points(torch.from_numpy(q).cuda())
    assert torch.equal(sd > 0, inside)


def test_interpolate_reproduces_closest(cuda_device):
    v, f = synth.heightfield(128, 128)
    r = make(v, f)
    p = torch.from_numpy(np.random.default_rng(9).uniform(-1.1, 1.1, (50000, 3)).astype(np.float32)).cuda()
    c, d, t, uv = r.closest_point(p, return_uv=True)
    back = r.interpolate(r.mesh_vertices, t, uv)
    assert float((back - c).abs().max()) <= 1e-6 * max(1.0, float(r.mesh_vertices.abs().max()))


def test_numpy_adapter(cuda_device):
    from triro.ray.ray_numpy import RayMeshIntersector as NumpyRMI

    v, f = synth.icosphere(3)
    r = NumpyRMI(vertices=v, faces=f)
    p = np.random.default_rng(10).uniform(-1.5, 1.5, (1000, 3))
    c, d, t = r.closest_point(p)
    assert c.dtype == np.float64 and d.dtype == np.float64 and t.dtype == np.int64
    assert c.shape == (1000, 3) and d.shape == (1000,) and t.shape == (1000,)
    sd = r.signed_distance(p)
    assert sd.dtype == np.float64 and sd.shape == (1000,)
    np.testing.assert_array_equal(np.abs(sd), d)
