"""Generalized winding number on the GPU (rt_winding_moments, rt_winding_number): moments and winding numbers against
the host simulator of rt_winding.cuh bit for bit, counters, batch layouts, edge inputs, refit / save / load / adopt,
repeatability, signed_distance(sign="winding") and the numpy adapter."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "winding"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import pointquery as pq  # noqa: E402
import winding as W  # noqa: E402
from test_closest_point_logic import sample_points  # noqa: E402
from test_gpu_closest_point import distributions  # noqa: E402
from test_winding_logic import WMESHES  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

pytestmark = pytest.mark.gpu
INF = float("inf")


def make(v, f):
    return RayMeshIntersector(vertices=torch.from_numpy(np.ascontiguousarray(v)), faces=torch.from_numpy(np.ascontiguousarray(f)))


def bits_equal(a, b, what):
    a = np.ascontiguousarray(a, dtype=np.float32); b = np.ascontiguousarray(b, dtype=np.float32)
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ (first at {np.argwhere(bad)[0]})"


def check_against_sim(r, p, what, betas=(2.0, INF)):
    blob = r.as_wrapper.blob.cpu().numpy()
    nn = r.as_wrapper.header["n_nodes"]
    gm = hops.winding_moments(r.as_wrapper)[:nn].cpu().numpy()
    hm = W.sim_moments(blob)
    bits_equal(gm, hm, f"{what}: moments")
    pt = torch.from_numpy(np.ascontiguousarray(p)).cuda()
    for beta in betas:
        cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
        got = hops.winding_number(r.as_wrapper, pt, beta, counters=cnt).cpu().numpy()
        sim = W.sim_winding(blob, p, beta)
        bits_equal(got, sim["w"], f"{what}: beta {beta}")
        s = sim["stats"]
        assert cnt.tolist() == [s["nodes"], s["tris"], s["points"], s["far"]], f"{what}: counters at beta {beta}"
        plain = r.winding_number(pt, beta).cpu().numpy()
        bits_equal(plain, got, f"{what}: plain vs instrumented kernel")


@pytest.mark.parametrize("name", list(WMESHES))
def test_cuda_matches_hostsim(cuda_device, name):
    v, f = WMESHES[name]
    r = make(v, f)
    p = sample_points(v, 4000, np.random.default_rng(5))
    check_against_sim(r, p, name)


@pytest.mark.parametrize("cfg", ["config2_icosphere", "config3_heightfield", "config4_soup"])
def test_cuda_matches_hostsim_true_size(cuda_device, cfg):
    v, f = {"config2_icosphere": lambda: synth.icosphere(7), "config3_heightfield": lambda: synth.heightfield(2048, 1024),
            "config4_soup": lambda: synth.triangle_soup(1_000_000)}[cfg]()
    r = make(v, f)
    rng = np.random.default_rng(17)
    pts = distributions(v, 3000, rng)
    check_against_sim(r, np.concatenate(list(pts.values())), cfg, betas=(2.0,))
    # the whole distributions on the GPU: finite and in a sane range
    for kind, p in distributions(v, 300_000, rng).items():
        w = r.winding_number(torch.from_numpy(p).cuda())
        assert bool(torch.isfinite(w).all()), f"{cfg}/{kind}"


def same(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def test_batch_layouts(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    base = torch.from_numpy(np.random.default_rng(1).uniform(-1.5, 1.5, (6, 5, 4, 3, 3)).astype(np.float32)).cuda()
    ref = r.winding_number(base.contiguous())
    assert ref.shape == base.shape[:-1]
    for name, x in (("5-d", base), ("strided", base.transpose(1, 2)), ("sliced", base[:, ::2, 1:, :, :])):
        got = r.winding_number(x)
        assert got.shape == x.shape[:-1], name
        assert same(got, r.winding_number(x.contiguous())), name
    one = torch.tensor([0.3, 0.2, -0.4], device="cuda")
    got = r.winding_number(one.broadcast_to(7, 9, 3))
    assert same(got, r.winding_number(one[None]).expand(7, 9))
    w = hops.winding_number(r.as_wrapper, base, 2.0, ray_first=100, ray_count=57)
    assert same(w, ref.reshape(-1)[100:157])


def test_edge_inputs(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    assert r.winding_number(torch.zeros(0, 3, device="cuda")).shape == (0,)
    cnt = torch.ones(4, dtype=torch.int64, device="cuda")
    assert hops.winding_number(r.as_wrapper, torch.zeros(2, 0, 3, device="cuda"), counters=cnt).shape == (2, 0)
    assert cnt.tolist() == [0, 0, 0, 0]
    p = torch.tensor([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.0, 0.0, 0.0], [3.0, 0, 0]], device="cuda")
    w = r.winding_number(p, INF).cpu().numpy()
    assert np.isnan(w[:3]).all() and abs(w[3] - 1.0) < 1e-5 and abs(w[4]) < 1e-5
    empty = RayMeshIntersector(vertices=torch.zeros(0, 3), faces=torch.zeros(0, 3, dtype=torch.int32))
    for beta in (2.0, INF):
        w = empty.winding_number(p[3:], beta)
        assert (w == 0).all() and not bool(torch.signbit(w).any())
    for bad in (0.999, 0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            r.winding_number(p, bad)
    lib = hops.get_module()
    rd, _ = hops.make_ray_desc(p, None)
    m = hops.winding_moments(r.as_wrapper)
    out = torch.empty(5, device="cuda")
    rc = lib.rt_winding_number(hops._ptr(r.as_wrapper.blob), hops._ptr(m), hops.C.byref(rd), None, 0.5, hops._ptr(out),
                               None, None, None)
    assert rc == -1 and b"beta" in lib.rt_last_error()


def test_refit_drops_the_cached_moments(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    p = sample_points(v, 3000, np.random.default_rng(3))
    pt = torch.from_numpy(p).cuda()
    before = r.winding_number(pt)
    v2 = (v * np.float32(1.3) + np.float32(0.1)).astype(np.float32)
    r.refit(torch.from_numpy(v2))
    check_against_sim(r, p, "refit")
    assert not torch.equal(before, r.winding_number(pt))


def test_save_load_and_adopt(cuda_device, tmp_path):
    v, f = synth.triangle_soup(20000, seed=5)
    r = make(v, f)
    pt = torch.from_numpy(np.random.default_rng(4).uniform(-1.2, 1.2, (50000, 3)).astype(np.float32)).cuda()
    ref = r.winding_number(pt)
    path = str(tmp_path / "bvh.pt")
    r.save_bvh(path)
    loaded = hops.AccelStructure().load(path)
    assert same(hops.winding_number(loaded, pt), ref)
    adopted = hops.AccelStructure().adopt(r.as_wrapper._inner.used().clone())
    assert same(hops.winding_number(adopted, pt), ref)
    nn = r.as_wrapper.header["n_nodes"]
    assert same(hops.winding_moments(adopted)[:nn], hops.winding_moments(r.as_wrapper)[:nn])


def test_repeatable(cuda_device):
    v, f = synth.heightfield(256, 256)
    r = make(v, f)
    pt = torch.from_numpy(np.random.default_rng(6).uniform(-1.2, 1.2, (200000, 3)).astype(np.float32)).cuda()
    a = r.winding_number(pt)
    r.as_wrapper._inner.winding_moments = None              # recompute the moments: same bits
    b = r.winding_number(pt)
    c = r.winding_number(pt, INF)
    assert same(a, b) and not same(a, c)


def test_signed_distance_with_winding_sign(cuda_device):
    for v, f in (synth.icosphere(4), WMESHES["cube_open"], synth.triangle_soup(5000, seed=2)):
        r = make(v, f)
        p = torch.from_numpy(np.random.default_rng(7).uniform(-1.3, 1.3, (20000, 3)).astype(np.float32)).cuda()
        sd = r.signed_distance(p, sign="winding")
        _, d, _ = r.closest_point(p)
        w = r.winding_number(p)
        assert torch.equal(sd.abs(), d)
        nz = d != 0
        assert torch.equal(sd[nz] > 0, w[nz] > 0.5)
        assert same(r.signed_distance(p), r.signed_distance(p, sign="contains"))
    with pytest.raises(ValueError):
        r.signed_distance(p, sign="parity")
    # on a closed mesh both signs agree away from the surface
    v, f = synth.icosphere(4)
    r = make(v, f)
    q = torch.from_numpy(np.random.default_rng(8).uniform(-1.3, 1.3, (20000, 3)).astype(np.float32)).cuda()
    clear = (q.norm(dim=1) - 1).abs() > 0.02
    assert torch.equal(r.signed_distance(q, sign="winding")[clear], r.signed_distance(q)[clear])
    ref = pq.query(pq.PointMesh(v, f), q.cpu().numpy(), pq.MIRROR)["distance"]
    bits_equal(r.signed_distance(q, sign="winding").abs().cpu().numpy(), ref, "|signed distance| vs mirror")


def test_numpy_adapter(cuda_device):
    from triro.ray.ray_numpy import RayMeshIntersector as NumpyRMI

    v, f = synth.icosphere(3)
    r = NumpyRMI(vertices=v, faces=f)
    p = np.random.default_rng(10).uniform(-1.5, 1.5, (1000, 3))
    w = r.winding_number(p)
    assert w.dtype == np.float64 and w.shape == (1000,)
    assert r.winding_number(p, beta=float("inf")).dtype == np.float64
    sd = r.signed_distance(p, sign="winding")
    assert sd.dtype == np.float64 and sd.shape == (1000,)
    _, d, _ = r.closest_point(p)
    np.testing.assert_array_equal(np.abs(sd), d)
    np.testing.assert_array_equal(sd > 0, (w > 0.5) & (d > 0))
