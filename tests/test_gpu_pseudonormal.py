"""Pseudo-normal signed distance on the GPU (rt_pseudonormals, rt_signed_distance): normals, edge counts, signed
distances and counters against the host simulator bit for bit (including the true-size config-2/3/4 meshes),
|sd| against closest_point, the sign against the binary64 truth and sign="winding", batch layouts, edge inputs,
refit / save / load / adopt, repeatability and the numpy adapter."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pseudonormal"))
import pseudonormal as P  # noqa: E402
from test_closest_point_logic import sample_points  # noqa: E402
from test_gpu_closest_point import distributions  # noqa: E402
from test_pseudonormal_logic import CLOSED, TAU, diagonal  # noqa: E402
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


def check_against_sim(r, p, what):
    blob = r.as_wrapper.blob.cpu().numpy()
    normals, counts = hops.pseudo_normals(r.as_wrapper)
    rows, hcounts = P.sim_normals(blob)
    bits_equal(normals.cpu().numpy(), rows, f"{what}: normals")
    assert tuple(counts.tolist()) == hcounts, f"{what}: edge counts"
    pt = torch.from_numpy(np.ascontiguousarray(p)).cuda()
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    got = hops.signed_distance_pseudonormal(r.as_wrapper, pt, counters=cnt)
    sim = P.sim_signed_distance(blob, p, rows)
    bits_equal(got.cpu().numpy(), sim["sd"], f"{what}: signed distance")
    s = sim["stats"]
    assert cnt.tolist() == [s["nodes"], s["tris"], s["points"], s["found"]], f"{what}: counters"
    plain = r.signed_distance(pt, sign="pseudonormal")
    assert same(plain, got), f"{what}: plain vs instrumented kernel"
    _, d, _ = r.closest_point(pt)
    assert same(plain.abs(), d), f"{what}: |sd| vs closest_point"
    return got.cpu().numpy(), hcounts


MESHES = dict(CLOSED)
MESHES["cube_open"] = (synth.cube(0.5)[0], np.ascontiguousarray(synth.cube(0.5)[1][2:]))
MESHES["hf64"] = synth.heightfield(64, 64)
MESHES["soup20k"] = synth.triangle_soup(20000, seed=5)
MESHES["torus_soup"] = P.soup(*P.torus())


@pytest.mark.parametrize("name", list(MESHES))
def test_cuda_matches_hostsim(cuda_device, name):
    v, f = MESHES[name]
    r = make(v, f)
    p = sample_points(v, 4000, np.random.default_rng(5))
    sd, counts = check_against_sim(r, p, name)
    if name in CLOSED:
        assert counts == (0, 0, 0) and r.is_watertight and r.is_winding_consistent
        d, inside = P.truth(v, f, p)
        clear = d > TAU * diagonal(v)
        assert np.array_equal((sd > 0)[clear], inside[clear]), f"{name}: sign vs binary64 truth"


@pytest.mark.parametrize("cfg", ["config2_icosphere", "config3_heightfield", "config4_soup"])
def test_cuda_matches_hostsim_true_size(cuda_device, cfg):
    v, f = {"config2_icosphere": lambda: synth.icosphere(7), "config3_heightfield": lambda: synth.heightfield(2048, 1024),
            "config4_soup": lambda: synth.triangle_soup(1_000_000)}[cfg]()
    r = make(v, f)
    pts = distributions(v, 3000, np.random.default_rng(17))
    check_against_sim(r, np.concatenate(list(pts.values())), cfg)


def test_sign_agrees_with_winding_away_from_the_surface(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    q = torch.from_numpy(np.random.default_rng(8).uniform(-1.3, 1.3, (50000, 3)).astype(np.float32)).cuda()
    clear = (q.norm(dim=1) - 1).abs() > 0.02
    pn = r.signed_distance(q, sign="pseudonormal")
    assert torch.equal(pn[clear] > 0, r.signed_distance(q, sign="winding")[clear] > 0)
    assert torch.equal(pn[clear] > 0, q.norm(dim=1)[clear] < 1)


def test_batch_layouts(cuda_device):
    v, f = P.star_prism()
    r = make(v, f)
    base = torch.from_numpy(np.random.default_rng(1).uniform(-1.2, 1.2, (6, 5, 4, 3, 3)).astype(np.float32)).cuda()
    ref = r.signed_distance(base.contiguous(), sign="pseudonormal")
    assert ref.shape == base.shape[:-1]
    for name, x in (("5-d", base), ("strided", base.transpose(1, 2)), ("sliced", base[:, ::2, 1:, :, :])):
        got = r.signed_distance(x, sign="pseudonormal")
        assert got.shape == x.shape[:-1], name
        assert same(got, r.signed_distance(x.contiguous(), sign="pseudonormal")), name
    one = torch.tensor([0.1, 0.2, 0.3], device="cuda")
    got = r.signed_distance(one.broadcast_to(7, 9, 3), sign="pseudonormal")
    assert same(got, r.signed_distance(one[None], sign="pseudonormal").expand(7, 9))
    w = hops.signed_distance_pseudonormal(r.as_wrapper, base, ray_first=100, ray_count=57)
    assert same(w, ref.reshape(-1)[100:157])


def test_edge_inputs(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    assert r.signed_distance(torch.zeros(0, 3, device="cuda"), sign="pseudonormal").shape == (0,)
    cnt = torch.ones(4, dtype=torch.int64, device="cuda")
    assert hops.signed_distance_pseudonormal(r.as_wrapper, torch.zeros(2, 0, 3, device="cuda"), counters=cnt).shape == (2, 0)
    assert cnt.tolist() == [0, 0, 0, 0]
    p = torch.tensor([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.0, 0.0, 0.0], [3.0, 0, 0]], device="cuda")
    sd = r.signed_distance(p, sign="pseudonormal").cpu().numpy()
    assert (sd[:3] == -np.inf).all() and sd[3] > 0.9 and sd[4] < -1.9
    at_vertex = torch.from_numpy(v[:5]).cuda()
    z = r.signed_distance(at_vertex, sign="pseudonormal")
    assert (z == 0).all() and not bool(torch.signbit(z).any())
    empty = RayMeshIntersector(vertices=torch.zeros(0, 3), faces=torch.zeros(0, 3, dtype=torch.int32))
    assert (empty.signed_distance(p[3:], sign="pseudonormal") == -np.inf).all()
    assert not empty.is_watertight and not empty.is_winding_consistent
    with pytest.raises(ValueError, match="pseudonormal"):
        r.signed_distance(p, sign="normals")
    lib = hops.get_module()
    nb, wb = hops.C.c_size_t(), hops.C.c_size_t()
    assert lib.rt_pseudonormals_sizes((1 << 30) // 3 + 1, hops.C.byref(nb), hops.C.byref(wb)) == -1
    assert lib.rt_pseudonormals_sizes((1 << 30) // 3, hops.C.byref(nb), hops.C.byref(wb)) == 0


def test_open_and_inconsistent_meshes(cuda_device):
    v, f = synth.cube(0.5)
    flipped = f.copy(); flipped[5] = flipped[5, ::-1]
    fin_v = np.concatenate([v, [[0.0, 0.0, 1.5]]]).astype(np.float32)
    for (vv, ff), want in (((v, f[2:]), (4, 0, 0)), ((v, flipped), (0, 0, 3)),
                           ((fin_v, np.concatenate([f, [[2, 6, 8]]]).astype(np.int32)), (2, 1, 0))):
        r = make(vv, ff)
        assert hops.edge_counts(r.as_wrapper) == want
        assert r.is_watertight == (want[0] == 0 and want[1] == 0) and r.is_winding_consistent == (want[2] == 0)
        check_against_sim(r, sample_points(vv, 2000, np.random.default_rng(2)), f"counts {want}")


def test_refit_drops_the_cached_normals(cuda_device):
    v, f = P.torus()
    r = make(v, f)
    p = sample_points(v, 3000, np.random.default_rng(3))
    pt = torch.from_numpy(p).cuda()
    before = r.signed_distance(pt, sign="pseudonormal")
    v2 = (v * np.float32([1.3, 0.8, 1.1]) + np.float32(0.1)).astype(np.float32)
    r.refit(torch.from_numpy(v2))
    check_against_sim(r, p, "refit")
    after = r.signed_distance(pt, sign="pseudonormal")
    assert not torch.equal(before, after)
    fresh = make(v2, f)
    assert same(after, fresh.signed_distance(pt, sign="pseudonormal"))


def test_save_load_and_adopt(cuda_device, tmp_path):
    v, f = synth.icosphere(5)
    r = make(v, f)
    pt = torch.from_numpy(np.random.default_rng(4).uniform(-1.2, 1.2, (50000, 3)).astype(np.float32)).cuda()
    ref = r.signed_distance(pt, sign="pseudonormal")
    path = str(tmp_path / "bvh.pt")
    r.save_bvh(path)
    loaded = hops.AccelStructure().load(path)
    assert same(hops.signed_distance_pseudonormal(loaded, pt), ref)
    adopted = hops.AccelStructure().adopt(r.as_wrapper._inner.used().clone())
    assert same(hops.signed_distance_pseudonormal(adopted, pt), ref)
    assert same(hops.pseudo_normals(adopted)[0], hops.pseudo_normals(r.as_wrapper)[0])
    assert hops.edge_counts(adopted) == (0, 0, 0)


def test_repeatable(cuda_device):
    v, f = P.soup(*synth.heightfield(256, 256))
    r = make(v, f)
    pt = torch.from_numpy(np.random.default_rng(6).uniform(-1.2, 1.2, (200000, 3)).astype(np.float32)).cuda()
    a = r.signed_distance(pt, sign="pseudonormal")
    b = r.signed_distance(pt, sign="pseudonormal")
    n1 = hops.pseudo_normals(r.as_wrapper)[0].clone()
    r.as_wrapper._inner.pseudo_normals = None              # recompute the normals: same bits
    c = r.signed_distance(pt, sign="pseudonormal")
    assert same(a, b) and same(a, c) and same(n1, hops.pseudo_normals(r.as_wrapper)[0])


def test_numpy_adapter(cuda_device):
    from triro.ray.ray_numpy import RayMeshIntersector as NumpyRMI

    v, f = P.notched_cube()
    r = NumpyRMI(vertices=v, faces=f)
    p = np.random.default_rng(10).uniform(-0.5, 2.5, (1000, 3))
    sd = r.signed_distance(p, sign="pseudonormal")
    assert sd.dtype == np.float64 and sd.shape == (1000,)
    _, d, _ = r.closest_point(p)
    np.testing.assert_array_equal(np.abs(sd), d)
    assert r.is_watertight and r.is_winding_consistent
    o = NumpyRMI(vertices=v, faces=f[1:])
    assert not o.is_watertight and o.is_winding_consistent
