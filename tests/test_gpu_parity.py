"""GPU parity tests: the CUDA path (through the Python mirror of the reference API, i.e. through
the C ABI) against the oracle on identical seeded inputs.

Bars: bit-exact for masks / indices / counts and — against the oracle's binary32 mirror — for
locations and uv as well; against the binary64 truth, exact outside the documented grazing set
and within 1e-5 relative for locations.
"""
import numpy as np
import pytest
import torch

import hostsim
from helpers import assert_bits_equal, check_closest_vs_mirror, check_closest_vs_truth, closest_to_numpy
from oracle import oracle
from triro import synth
from triro.backend import ops as hops
from triro.ray.ray_optix import RayMeshIntersector

pytestmark = pytest.mark.gpu


def make(v, f):
    return RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))


def flat(t):
    return t.detach().cpu().numpy().reshape(-1, 3)


# ---------------------------------------------------------------- builder pieces
@pytest.mark.parametrize("n", [1, 2, 33, 4096, 4097, 100_003, 1_500_000])
def test_onesweep_sort_matches_numpy_stable_sort(cuda_device, n):
    rng = np.random.default_rng(n)
    bits = 63 if n % 2 else 20           # few distinct keys -> exercises stability
    keys = rng.integers(0, 2 ** bits, size=n, dtype=np.uint64)
    vals = np.arange(n, dtype=np.int32)
    k = torch.from_numpy(keys.view(np.int64)).to(cuda_device)
    v = torch.from_numpy(vals).to(cuda_device)
    hops.sort_pairs_u64(k, v)
    torch.cuda.synchronize()
    order = np.argsort(keys, kind="stable")
    assert_bits_equal(k.cpu().numpy().view(np.uint64), keys[order], "sorted keys")
    assert_bits_equal(v.cpu().numpy(), vals[order], "sorted values (stability)")


@pytest.mark.parametrize("mesh", ["tri1", "tri2", "tri3", "tri5", "ico0", "ico3", "ico5", "soup20k", "hf64"])
def test_bvh_blob_is_valid_and_conservative(cuda_device, mesh):
    v, f = named_mesh(mesh)
    rmi = make(v, f)
    blob = rmi.as_wrapper.blob.cpu().numpy()
    code, info = hostsim.check_blob(blob)
    assert code == 0, f"blob check failed with code {code}"
    assert info["tris"] == len(f)
    prims = hostsim.blob_prims(blob, len(f))
    assert np.array_equal(np.sort(prims), np.arange(len(f))), "triangle records are not a permutation of the faces"
    hdr = rmi.as_wrapper.header
    assert hdr["n_tris"] == len(f) and hdr["depth"] == info["depth"]


def test_build_is_deterministic_in_topology(cuda_device):
    v, f = synth.icosphere(4)
    a, b = make(v, f), make(v, f)
    o, d = synth.random_rays(50_000, seed=5, device=cuda_device, box=True)
    ra = a.intersects_location(o * 1.5, d)
    rb = b.intersects_location(o * 1.5, d)
    for x, y in zip(ra, rb):
        assert torch.equal(x, y)


def named_mesh(name):
    if name.startswith("tri"):
        n = int(name[3:])
        rng = np.random.default_rng(n)
        v = rng.uniform(-1, 1, size=(3 * n, 3)).astype(np.float32)
        return v, np.arange(3 * n, dtype=np.int32).reshape(n, 3)
    if name.startswith("ico"):
        return synth.icosphere(int(name[3:]))
    if name == "soup20k":
        return synth.triangle_soup(20_000, sigma=0.02, seed=11)
    if name == "hf64":
        return synth.heightfield(64, 32)
    raise KeyError(name)


# ---------------------------------------------------------------- reference known answers (test/test.py)
def test_k1_k2_single_triangle(cuda_device):
    v = np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0]], np.float32)
    f = np.array([[0, 1, 2]], np.int32)
    r = make(v, f)
    o = torch.tensor([[0, 0, 4], [10, 10, 10]], dtype=torch.float32, device=cuda_device)
    d = torch.tensor([[0, 0, -1], [0, 1, 0]], dtype=torch.float32, device=cuda_device)
    assert r.intersects_any(o, d).tolist() == [True, False]           # K1
    assert r.intersects_first(o, d).tolist() == [0, -1]               # K2
    assert r.intersects_any(o, d).dtype == torch.bool and r.intersects_first(o, d).dtype == torch.int32


def test_k3_k4_readme_quickstart(cuda_device):
    v, f = synth.icosphere(3)                                           # trimesh default icosphere: 1 280 faces
    r = make(v, f)
    o, d = synth.readme_rays(800, device=cuda_device)
    assert o.stride()[:2] == (0, 0)                                     # stride-0 broadcast origin
    hit, front, ray_idx, tri_idx, loc, uv = r.intersects_closest(o, d, stream_compaction=True)
    assert hit.shape == (800, 800) and hit.dtype == torch.bool
    h = int(hit.sum())
    assert front.shape == (h,) and ray_idx.shape == (h,) and tri_idx.shape == (h,) and loc.shape == (h, 3) and uv.shape == (h, 2)
    assert ray_idx.dtype == torch.int32 and tri_idx.dtype == torch.int32
    assert 0.095 < h / hit.numel() < 0.101                              # K3: disc x^2+y^2 <= 1/8 of the grid
    assert bool(front.all())                                            # outward CCW sphere seen from outside
    nrm = loc.norm(dim=1)
    assert float(nrm.min()) > 0.985 and float(nrm.max()) <= 1.0 + 1e-6
    assert torch.equal(ray_idx.long(), torch.nonzero(hit.reshape(-1)).reshape(-1))
    # K4: uv[:,0] weights vertex 0, uv[:,1] vertex 1 (test/test.py:41)
    vt = torch.from_numpy(v).to(cuda_device)
    ft = torch.from_numpy(f).to(cuda_device).long()
    tv = vt[ft[tri_idx.long()]]
    rec = uv[:, :1] * tv[:, 0] + uv[:, 1:] * tv[:, 1] + (1 - uv[:, :1] - uv[:, 1:]) * tv[:, 2]
    assert float((rec - loc).abs().max()) < 1e-5


def test_k5_k6_stacked_triangles(cuda_device):
    v = np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0], [0.5, -0.5, -1], [0, 0.5, -1], [-0.5, -0.5, -1]], np.float32)
    f = np.array([[0, 1, 2], [3, 4, 5]], np.int32)
    r = make(v, f)
    o = torch.tensor([[0, 0, -4], [0, 0.1, 4]], dtype=torch.float32, device=cuda_device)
    d = torch.tensor([[0, 0, 1], [0, 0, -1]], dtype=torch.float32, device=cuda_device)
    loc, ray_idx, tri_idx = r.intersects_location(o, d)
    got = sorted((int(a), int(b), tuple(round(float(x), 6) for x in l)) for a, b, l in zip(ray_idx, tri_idx, loc))
    assert got == [(0, 0, (0.0, 0.0, 0.0)), (0, 1, (0.0, 0.0, -1.0)), (1, 0, (0.0, 0.1, 0.0)), (1, 1, (0.0, 0.1, -1.0))]   # K5
    assert r.intersects_count(o, d).tolist() == [2, 2]                 # K6
    tri, ray = r.intersects_id(o, d)
    assert torch.equal(tri, tri_idx) and torch.equal(ray, ray_idx)


def test_k7_contains_point_under_vertex(cuda_device):
    v, f = synth.icosphere(3)
    r = make(v, f)
    assert r.contains_points(torch.tensor([[0, 0, 0.999]], dtype=torch.float32, device=cuda_device)).tolist() == [True]


# ---------------------------------------------------------------- closest hit vs oracle
@pytest.mark.parametrize("mesh,nray", [("ico3", 60_000), ("ico5", 60_000), ("soup20k", 60_000), ("hf64", 60_000), ("tri5", 5_000)])
def test_closest_random_rays_vs_mirror_and_truth(cuda_device, mesh, nray):
    v, f = named_mesh(mesh)
    r = make(v, f)
    o, d = synth.random_rays(nray, seed=42, device=cuda_device, box=True)
    o = o * 1.3
    got = closest_to_numpy(r.intersects_closest(o, d))
    om = oracle.OracleMesh(v, f)
    check_closest_vs_mirror(got, om, flat(o), flat(d))
    check_closest_vs_truth(got, om, flat(o), flat(d))
    first = r.intersects_first(o, d).cpu().numpy()
    assert_bits_equal(first, got["tri"], "intersects_first vs intersects_closest")
    anyh = r.intersects_any(o, d).cpu().numpy().astype(np.uint8)
    assert_bits_equal(anyh, got["hit"], "intersects_any vs intersects_closest")


def test_closest_brute_force_small(cuda_device):
    """Oracle without its BVH (all rays x all triangles)."""
    v, f = synth.icosphere(2)
    r = make(v, f)
    o, d = synth.readme_rays(160, device=cuda_device)
    got = closest_to_numpy(r.intersects_closest(o, d))
    om = oracle.OracleMesh(v, f, use_bvh=False)
    check_closest_vs_mirror(got, om, flat(o), flat(d))
    check_closest_vs_truth(got, om, flat(o), flat(d))


def test_closest_config2_camera_subsample(cuda_device):
    """BASELINE config 2 geometry (icosphere subdiv 7, 327 680 triangles), pinhole camera at
    reduced resolution so the oracle finishes in seconds."""
    v, f = synth.icosphere(7)
    r = make(v, f)
    o, d = synth.pinhole_rays(480, 270, device=cuda_device)
    got = closest_to_numpy(r.intersects_closest(o, d))
    assert 0.30 < got["hit"].mean() < 0.38
    om = oracle.OracleMesh(v, f)
    check_closest_vs_mirror(got, om, flat(o), flat(d))
    check_closest_vs_truth(got, om, flat(o), flat(d))


# ---------------------------------------------------------------- strided / broadcast / batched inputs
def test_strided_and_broadcast_inputs(cuda_device):
    v, f = synth.icosphere(3)
    r = make(v, f)
    base_o, base_d = synth.random_rays(6 * 7 * 5, seed=9, device=cuda_device, box=True)
    base_o = base_o * 2
    ref = closest_to_numpy(r.intersects_closest(base_o, base_d))
    # 3 batch dims
    o3, d3 = base_o.reshape(6, 7, 5, 3), base_d.reshape(6, 7, 5, 3)
    got = r.intersects_closest(o3, d3)
    assert got[0].shape == (6, 7, 5) and got[3].shape == (6, 7, 5, 3) and got[4].shape == (6, 7, 5, 2)
    for k, x in closest_to_numpy(got).items():
        assert_bits_equal(x, ref[k], f"3-d batch {k}")
    # non-contiguous: transposed batch dims, channel-first storage, padded rows
    oc = o3.permute(3, 0, 1, 2).contiguous().permute(1, 2, 3, 0)          # last-dim stride != 1
    pad = torch.zeros(6, 7, 5, 8, device=cuda_device)
    pad[..., 2:5] = d3
    dc = pad[..., 2:5]                                                      # row pitch 8, offset 2
    assert not oc.is_contiguous() and not dc.is_contiguous()
    for k, x in closest_to_numpy(r.intersects_closest(oc, dc)).items():
        assert_bits_equal(x, ref[k], f"strided {k}")
    # transposed view: compare with an explicit contiguous copy
    ot, dt = o3.transpose(0, 2), d3.transpose(0, 2)
    a = closest_to_numpy(r.intersects_closest(ot, dt))
    b = closest_to_numpy(r.intersects_closest(ot.contiguous(), dt.contiguous()))
    for k in a:
        assert_bits_equal(a[k], b[k], f"transposed {k}")
    # negative-free flip via index arithmetic is not expressible in torch; broadcast both ways instead
    one_o = torch.tensor([0.1, -0.2, 2.5], device=cuda_device).broadcast_to(base_d.shape)
    a = closest_to_numpy(r.intersects_closest(one_o, base_d))
    b = closest_to_numpy(r.intersects_closest(one_o.contiguous(), base_d))
    for k in a:
        assert_bits_equal(a[k], b[k], f"broadcast origin {k}")
    one_d = torch.tensor([0.0, 0.0, -1.0], device=cuda_device).broadcast_to(base_o.shape)
    a = r.intersects_count(base_o, one_d)
    b = r.intersects_count(base_o, one_d.contiguous())
    assert torch.equal(a, b)


def test_input_validation(cuda_device):
    v, f = synth.icosphere(1)
    r = make(v, f)
    o = torch.zeros(4, 3, device=cuda_device)
    with pytest.raises(ValueError):
        r.intersects_any(o.cpu(), o.cpu())
    with pytest.raises(ValueError):
        r.intersects_any(o.double(), o.double())
    with pytest.raises(ValueError):
        r.intersects_any(o, torch.zeros(5, 3, device=cuda_device))
    # more than 3 batch dims (reference limit MAX_SIZE_LENGTH = 4, silently wrong there): merged, same answers
    o5, d5 = synth.random_rays(2 * 3 * 4 * 5, seed=3, device=cuda_device, box=True)
    o5 = (o5 * 2).reshape(2, 3, 4, 5, 3); d5 = d5.reshape(2, 3, 4, 5, 3)
    a5 = r.intersects_closest(o5, d5)
    b5 = r.intersects_closest(o5.reshape(-1, 3), d5.reshape(-1, 3))
    assert a5[0].shape == (2, 3, 4, 5) and a5[3].shape == (2, 3, 4, 5, 3)
    for x, y in zip(a5, b5):
        assert torch.equal(x.reshape(y.shape), y)
    a5t = r.intersects_count(o5.transpose(0, 3), d5.transpose(0, 3))                 # non-mergeable strides -> copy
    assert torch.equal(a5t, r.intersects_count(o5, d5).transpose(0, 3))
    with pytest.raises(ValueError):
        RayMeshIntersector(foo=1)
    with pytest.raises(ValueError):
        make(v, f + 1000)


def test_empty_and_degenerate_inputs(cuda_device):
    v, f = synth.icosphere(1)
    r = make(v, f)
    e = torch.zeros(0, 3, device=cuda_device)
    assert r.intersects_any(e, e).shape == (0,)
    assert r.intersects_count(e, e).shape == (0,)
    res = r.intersects_closest(e, e, stream_compaction=True)
    assert [tuple(x.shape) for x in res] == [(0,), (0,), (0,), (0,), (0, 3), (0, 2)]
    loc, ri, ti = r.intersects_location(e, e)
    assert loc.shape == (0, 3) and ri.shape == (0,) and ti.shape == (0,)
    # NaN / zero-direction rays miss (SURVEY A.2)
    o = torch.tensor([[0.05, 0.03, 3], [0, 0, 3], [float("nan"), 0, 3], [0, 0, 3]], dtype=torch.float32, device=cuda_device)
    d = torch.tensor([[0, 0, -1], [0, 0, 0], [0, 0, -1], [float("nan"), 0, -1]], dtype=torch.float32, device=cuda_device)
    assert r.intersects_any(o, d).tolist() == [True, False, False, False]
    assert r.intersects_count(o, d).tolist() == [2, 0, 0, 0]
    hit, front, tri, loc, uv = r.intersects_closest(o, d)
    assert hit.tolist() == [True, False, False, False]
    assert tri[1:].tolist() == [-1, -1, -1] and float(loc[1:].abs().sum()) == 0.0 and float(uv[1:].abs().sum()) == 0.0
    assert front[1:].tolist() == [False, False, False]
    # empty mesh: everything misses
    r0 = RayMeshIntersector(vertices=torch.zeros(0, 3), faces=torch.zeros(0, 3, dtype=torch.int32))
    assert r0.intersects_any(o, d).tolist() == [False] * 4
    # mesh with degenerate (zero-area) and NaN triangles next to a good one
    vv = np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0], [1, 1, 1], [1, 1, 1], [1, 1, 1], [np.nan, 0, 0], [0, 1, 0], [1, 0, 0]], np.float32)
    ff = np.array([[0, 1, 2], [3, 4, 5], [6, 7, 8]], np.int32)
    r1 = make(vv, ff)
    o1 = torch.tensor([[0, 0, 4], [1, 1, 4]], dtype=torch.float32, device=cuda_device)
    d1 = torch.tensor([[0, 0, -1], [0, 0, -1]], dtype=torch.float32, device=cuda_device)
    assert r1.intersects_first(o1, d1).tolist() == [0, -1]


def test_interval_is_open_at_zero_and_bounded_by_tmax(cuda_device):
    v = np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0]], np.float32)
    f = np.array([[0, 1, 2]], np.int32)
    r = make(v, f)
    o = torch.tensor([[0, 0, 0], [0, 0, -1], [0, 0, 2e7], [0, 0, 0.5e7]], dtype=torch.float32, device=cuda_device)
    d = torch.tensor([[0, 0, -1], [0, 0, -1], [0, 0, -1], [0, 0, -1]], dtype=torch.float32, device=cuda_device)
    # origin on the triangle (t = 0) -> no hit; behind -> no hit; beyond 1e7 -> no hit; within -> hit
    assert r.intersects_any(o, d).tolist() == [False, False, False, True]
    # unnormalised direction: t is measured in units of |d|
    o2 = torch.tensor([[0, 0, 4]], dtype=torch.float32, device=cuda_device)
    d2 = torch.tensor([[0, 0, -1e-7]], dtype=torch.float32, device=cuda_device)   # t = 4e7 > tmax
    assert r.intersects_any(o2, d2).tolist() == [False]
    d3 = torch.tensor([[0, 0, -1e-6]], dtype=torch.float32, device=cuda_device)   # t = 4e6 < tmax
    assert r.intersects_any(o2, d3).tolist() == [True]
    # back face is hit, front flag false
    o4 = torch.tensor([[0, 0, -4]], dtype=torch.float32, device=cuda_device)
    d4 = torch.tensor([[0, 0, 1]], dtype=torch.float32, device=cuda_device)
    hit, front, *_ = r.intersects_closest(o4, d4)
    hit2, front2, *_ = r.intersects_closest(o2, -d4)
    # triangle (0.5,-0.5),(0,0.5),(-0.5,-0.5) is counter-clockwise seen from +z
    assert hit.tolist() == [True] and front.tolist() == [False]
    assert hit2.tolist() == [True] and front2.tolist() == [True]


# ---------------------------------------------------------------- count / all hits / compaction
@pytest.mark.parametrize("mesh", ["ico4", "soup20k", "hf64"])
def test_count_and_location_vs_oracle(cuda_device, mesh):
    v, f = named_mesh(mesh)
    r = make(v, f)
    o, d = synth.random_rays(40_000, seed=77, device=cuda_device, box=True)
    o = o * 1.2
    cnt = r.intersects_count(o, d).cpu().numpy()
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR)
    oloc, ori, oti, ocount, raw = oi.intersects_location(flat(o), flat(d))
    assert_bits_equal(cnt, ocount, "intersects_count vs mirror")
    truth = oracle.query(oracle.OracleMesh(v, f), flat(o), flat(d), oracle.TRUTH, want=("count", "flags"))
    clean = truth["flags"] == 0
    assert (truth["flags"] != 0).mean() < 0.02
    assert np.array_equal(cnt[clean], truth["count"][clean]), "count differs from the binary64 truth outside the grazing set"
    loc, ri, ti = r.intersects_location(o, d)
    loc, ri, ti = loc.cpu().numpy(), ri.cpu().numpy(), ti.cpu().numpy()
    # rays ascending, per-ray group sizes = min(count, 8)
    assert np.all(np.diff(ri) >= 0)
    sizes = np.bincount(ri, minlength=len(cnt))
    assert np.array_equal(sizes, np.minimum(cnt, 8))
    # per-ray SET equality of (tri, loc bits) for rays with <= 8 hits; valid distinct hits beyond
    start = np.concatenate([[0], np.cumsum(sizes)])
    ostart = np.concatenate([[0], np.cumsum(np.minimum(ocount, 8))])
    for i in np.nonzero(sizes)[0]:
        mine = sorted(zip(ti[start[i]:start[i + 1]].tolist(), map(bytes, loc[start[i]:start[i + 1]])))
        if cnt[i] <= 8:
            theirs = sorted(zip(oti[ostart[i]:ostart[i + 1]].tolist(), map(bytes, oloc[ostart[i]:ostart[i + 1]])))
            assert mine == theirs, f"ray {i}: hit set differs"
        else:
            k = raw["list_n"][i]
            allowed = dict(zip(raw["list_tri"][i, :k].tolist(), map(bytes, raw["list_loc"][i, :k])))
            assert len({t for t, _ in mine}) == 8
            if k >= cnt[i]:   # the oracle listed every hit of this ray
                assert all(t in allowed and allowed[t] == l for t, l in mine)
    # intersects_id re-orders the same arrays
    t2, r2, l2 = r.intersects_id(o, d, return_locations=True)
    assert np.array_equal(t2.cpu().numpy(), ti) and np.array_equal(r2.cpu().numpy(), ri)
    assert_bits_equal(l2.cpu().numpy(), loc, "intersects_id locations")


def test_more_than_eight_hits(cuda_device):
    """40 stacked quads: every ray through the stack has 80 triangle candidates, 40 hits."""
    n = 40
    quads = []
    for k in range(n):
        z = -k * 0.1
        quads += [[-1, -1, z], [1, -1, z], [1, 1, z], [-1, 1, z]]
    v = np.array(quads, np.float32)
    f = np.concatenate([[[4 * k, 4 * k + 1, 4 * k + 2], [4 * k, 4 * k + 2, 4 * k + 3]] for k in range(n)]).astype(np.int32)
    r = make(v, f)
    o = torch.tensor([[0.3, 0.2, 5.0], [-0.5, 0.1, 5.0], [3, 3, 5.0]], dtype=torch.float32, device=cuda_device)
    d = torch.tensor([[0, 0, -1.0]] * 3, dtype=torch.float32, device=cuda_device)
    assert r.intersects_count(o, d).tolist() == [40, 40, 0]
    loc, ri, ti = r.intersects_location(o, d)
    assert ri.tolist() == [0] * 8 + [1] * 8
    for ray in (0, 1):
        tris = ti[ri == ray].tolist()
        assert len(set(tris)) == 8
        for t, l in zip(tris, loc[ri == ray].tolist()):
            assert abs(l[2] - (-(t // 2) * 0.1)) < 1e-6 and abs(l[0] - float(o[ray, 0])) < 1e-6


@pytest.mark.parametrize("shape", [(1,), (2047,), (2048,), (2049,), (300, 333), (7, 11, 13)])
def test_stream_compaction_matches_boolean_mask_semantics(cuda_device, shape):
    v, f = synth.icosphere(3)
    r = make(v, f)
    n = int(np.prod(shape))
    o, d = synth.random_rays(n, seed=n, device=cuda_device, box=True)
    o, d = (o * 2).reshape(*shape, 3), d.reshape(*shape, 3)
    hit, front, tri, loc, uv = r.intersects_closest(o, d)
    chit, cfront, cray, ctri, cloc, cuv = r.intersects_closest(o, d, stream_compaction=True)
    assert torch.equal(chit, hit)
    # reference semantics, ray_optix.py:142-144
    ray_idx = torch.arange(0, hit.numel(), device=cuda_device).int()[hit.reshape(-1)]
    assert torch.equal(cray, ray_idx) and torch.equal(cfront, front[hit]) and torch.equal(ctri, tri[hit])
    assert torch.equal(cloc, loc[hit]) and torch.equal(cuv, uv[hit])
    t2, r2, l2 = r.intersects_id(o, d, return_locations=True, multiple_hits=False)
    assert torch.equal(t2, tri[hit]) and torch.equal(r2, ray_idx) and torch.equal(l2, loc[hit])
    t3, r3 = r.intersects_id(o, d, multiple_hits=False)
    assert torch.equal(t3, t2) and torch.equal(r3, r2)


# ---------------------------------------------------------------- contains_points
def test_contains_points_vs_oracle_and_analytic(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    g = torch.Generator(device=cuda_device); g.manual_seed(3)
    p = (torch.rand((50_000, 3), generator=g, device=cuda_device) * 2 - 1) * 1.1
    got = r.contains_points(p).cpu().numpy()
    rad = p.norm(dim=1).cpu().numpy()
    sure_in, sure_out = rad < 0.99, rad > 1.0
    assert got[sure_in].all() and not got[sure_out].any()
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR)
    inside, cp, cm = oi.contains_core(p.cpu().numpy(), oi.DEFAULT_DIRECTION)
    core = inside & (cp % 2 == 1) & (cm % 2 == 1)
    broken = ~((cp % 2 == 1) & (cm % 2 == 1)) & ((cp == 0) | (cm == 0))
    # outside the (random-direction) retry set the answer is the deterministic core
    assert np.array_equal(got[~broken], core[~broken])
    contain, brk, flags = hops.contains_parity(r.as_wrapper, p, oi.DEFAULT_DIRECTION, *r._aabb_host)
    assert np.array_equal(contain.cpu().numpy(), core) and np.array_equal(brk.cpu().numpy(), broken)
    assert flags.tolist() == [int(inside.any()), int(broken.any())]


def test_contains_points_reference_quirks(cuda_device):
    """Truth table of SURVEY Appendix A.6 on the unit cube."""
    v, f = synth.cube(0.5)
    r = make(v, f)
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR, use_bvh=False)
    pts = torch.tensor([[0.1, 0.2, 0.3], [0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [0.2, -0.3, 0.4]], dtype=torch.float32, device=cuda_device)
    torch.manual_seed(0)
    got = r.contains_points(pts).tolist()
    torch.manual_seed(0)
    exp = oi.contains_points(pts.cpu().numpy()).tolist()
    assert got == exp
    # explicit direction + an outside ("broken") point -> the reference returns all False
    xdir = torch.tensor([1.0, 0.0, 0.0], device=cuda_device)
    assert r.contains_points(pts, xdir).tolist() == oi.contains_points(pts.cpu().numpy(), [1, 0, 0]).tolist() == [False] * 4
    # explicit direction, only inside points -> correct answers
    inside_pts = pts[[0, 3]]
    assert r.contains_points(inside_pts, xdir).tolist() == [True, True]
    # nothing inside the AABB -> all False without tracing
    far = torch.tensor([[5.0, 5, 5], [0.5, 0.5, 0.5]], dtype=torch.float32, device=cuda_device)   # second is ON the box
    assert r.contains_points(far).tolist() == [False, False]


# ---------------------------------------------------------------- update_raw / host path / stats
def test_update_raw_rebuilds(cuda_device):
    v, f = synth.icosphere(2)
    r = make(v, f)
    o = torch.tensor([[0, 0, 3.0]], device=cuda_device); d = torch.tensor([[0, 0, -1.0]], device=cuda_device)
    assert abs(float(r.intersects_closest(o, d)[3][0, 2]) - 1.0) < 2e-2
    r.update_raw(torch.from_numpy(v * 0.5), torch.from_numpy(f))
    assert abs(float(r.intersects_closest(o, d)[3][0, 2]) - 0.5) < 1e-2
    assert torch.allclose(r.mesh_aabb[1], torch.full((3,), 0.5, device=cuda_device), atol=1e-2)


def test_host_buffer_entry_point_matches_device_path(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    o, d = synth.pinhole_rays(1500, 900, device="cpu")          # 1.35 M rays -> two chunks
    d = d.reshape(-1, 3).contiguous().pin_memory()
    o1 = torch.tensor([0.0, 0.0, 3.0]).pin_memory()
    out = hops.host_closest(r.as_wrapper, o1, d)
    dev = closest_to_numpy(r.intersects_closest(o1.to(cuda_device).broadcast_to(d.shape), d.to(cuda_device)))
    assert_bits_equal(out["hit"].numpy().astype(np.uint8), dev["hit"], "host hit")
    assert_bits_equal(out["tri"].numpy(), dev["tri"], "host tri")
    assert_bits_equal(out["loc"].numpy(), dev["loc"], "host loc")
    assert_bits_equal(out["uv"].numpy(), dev["uv"], "host uv")
    # per-ray origins
    o2 = o1.broadcast_to(d.shape).contiguous().pin_memory()
    out2 = hops.host_closest(r.as_wrapper, o2, d)
    assert_bits_equal(out2["tri"].numpy(), dev["tri"], "host tri (per-ray origins)")


def test_trace_stats_counts_agree_with_host_simulation(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    o, d = synth.readme_rays(200, device=cuda_device)
    # the direct (triangles-in-step) schedule visits nodes in exactly the order of the host simulation; the other
    # schedules test triangles later and may visit a few more nodes (later tmax shrink)
    old = hops.set_knobs(schedule=hops.SCHED_DIRECT)
    try:
        st = hops.trace_stats(r.as_wrapper, o, d, "closest")
    finally:
        hops.set_knobs(**old)
    sim = hostsim.trace(r.as_wrapper.blob.cpu().numpy(), "closest", flat(o), flat(d))
    assert st["rays"] == 40_000 and st["nodes"] == sim["stats"]["nodes"] and st["tris"] == sim["stats"]["tris"]
    assert st["hits"] == sim["stats"]["hits"]
    sq = hops.trace_stats(r.as_wrapper, o.contiguous(), d, "closest")          # per-ray origins -> incoherent schedule
    assert sq["rays"] == 40_000 and sq["hits"] == st["hits"] and sq["nodes"] >= st["nodes"]


def test_coherent_and_incoherent_auto_schedules_give_identical_results(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    o, d = synth.pinhole_rays(640, 360, device=cuda_device)
    a = closest_to_numpy(r.intersects_closest(o, d))                            # broadcast origin: coop_coherent
    b = closest_to_numpy(r.intersects_closest(o.contiguous(), d))               # materialised origins: coop_incoherent
    for k in a:
        assert_bits_equal(a[k], b[k], f"coherent vs incoherent {k}")
    assert torch.equal(r.intersects_count(o, d), r.intersects_count(o.contiguous(), d))
    assert torch.equal(r.intersects_any(o, d), r.intersects_any(o.contiguous(), d))


# ---------------------------------------------------------------- golden fixture (reference's own host logic)
def test_golden_fixture_from_reference_host_logic(cuda_device):
    """tests/golden/host_logic.npz was produced by executing the reference's unmodified
    triro/ray/ray_optix.py (with the oracle standing in for OptiX); the CUDA path must reproduce
    every array: tuple orders, dtypes, compaction, intersects_id, contains_points quirks."""
    import os

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_logic.npz"))
    r = make(g["ico_v"], g["ico_f"])
    o = torch.from_numpy(g["ico_o"]).to(cuda_device); d = torch.from_numpy(g["ico_d"]).to(cuda_device)
    for x, name in zip(r.intersects_closest(o, d), ("hit", "front", "tri", "loc", "uv")):
        exp = g[f"ico_dense_{name}"]
        assert x.cpu().numpy().dtype == exp.dtype and x.shape == exp.shape
        assert_bits_equal(x.cpu().numpy(), exp, f"golden dense {name}")
    for x, name in zip(r.intersects_closest(o, d, stream_compaction=True), ("hit", "front", "ray", "tri", "loc", "uv")):
        exp = g[f"ico_comp_{name}"]
        assert x.cpu().numpy().dtype == exp.dtype
        assert_bits_equal(x.cpu().numpy(), exp, f"golden compact {name}")
    t, ri, l = r.intersects_id(o, d, return_locations=True, multiple_hits=False)
    assert_bits_equal(t.cpu().numpy(), g["ico_id1_tri"]); assert_bits_equal(ri.cpu().numpy(), g["ico_id1_ray"])
    assert_bits_equal(l.cpu().numpy(), g["ico_id1_loc"])
    t, ri, l = r.intersects_id(o, d, return_locations=True, multiple_hits=True)
    # all-hits: same rays / group sizes; per-ray sets equal (order within a ray is unspecified in the reference)
    assert_bits_equal(ri.cpu().numpy(), g["ico_idm_ray"])
    mine = sorted(zip(ri.tolist(), t.tolist(), map(bytes, l.cpu().numpy())))
    theirs = sorted(zip(g["ico_idm_ray"].tolist(), g["ico_idm_tri"].tolist(), map(bytes, g["ico_idm_loc"])))
    assert mine == theirs
    assert_bits_equal(r.intersects_any(o, d).cpu().numpy(), g["ico_any"])
    assert_bits_equal(r.intersects_first(o, d).cpu().numpy(), g["ico_first"])
    assert_bits_equal(r.intersects_count(o, d).cpu().numpy(), g["ico_count"])
    assert_bits_equal(r.mesh_aabb[0].cpu().numpy(), g["ico_aabb_lo"]); assert_bits_equal(r.mesh_aabb[1].cpu().numpy(), g["ico_aabb_hi"])
    rc = make(g["cube_v"], g["cube_f"])
    pts = torch.from_numpy(g["cube_pts"]).to(cuda_device)
    torch.manual_seed(1234)
    assert_bits_equal(rc.contains_points(pts).cpu().numpy(), g["cube_default"], "cube default direction")
    xdir = torch.tensor([1.0, 0.0, 0.0], device=cuda_device)
    assert_bits_equal(rc.contains_points(torch.from_numpy(g["cube_inside_pts"]).to(cuda_device), xdir).cpu().numpy(), g["cube_inside_xdir"])
    assert_bits_equal(rc.contains_points(pts, xdir).cpu().numpy(), g["cube_mixed_xdir"], "explicit direction quirk")
    assert_bits_equal(rc.contains_points(torch.from_numpy(g["cube_far_pts"]).to(cuda_device)).cpu().numpy(), g["cube_far"])
    rs = make(g["sph_v"], g["sph_f"])
    torch.manual_seed(99)
    assert_bits_equal(rs.contains_points(torch.from_numpy(g["sph_pts"]).to(cuda_device)).cpu().numpy(), g["sph_default"], "sphere")


# ---------------------------------------------------------------- SURVEY 8(f): refit and blob serialisation
def test_refit_matches_rebuild_and_oracle(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    rng = np.random.default_rng(3)
    v2 = (v * np.array([1.2, 0.7, 1.1], np.float32) + rng.normal(0, 0.004, size=v.shape).astype(np.float32)).astype(np.float32)
    r.refit(torch.from_numpy(v2))
    blob = r.as_wrapper.blob.cpu().numpy()
    assert hostsim.check_blob(blob)[0] == 0
    o, d = synth.random_rays(60_000, seed=12, device=cuda_device, box=True)
    o = o * 1.5
    got = closest_to_numpy(r.intersects_closest(o, d))
    om = oracle.OracleMesh(v2, f)
    check_closest_vs_mirror(got, om, flat(o), flat(d))
    fresh = make(v2, f)
    ref = closest_to_numpy(fresh.intersects_closest(o, d))
    for k in got:
        assert_bits_equal(got[k], ref[k], f"refit vs rebuild {k}")
    assert torch.equal(r.intersects_count(o, d), fresh.intersects_count(o, d))
    assert torch.allclose(r.mesh_aabb[1], fresh.mesh_aabb[1])
    with pytest.raises(ValueError):
        r.as_wrapper._inner.refit(r.mesh_vertices, r.mesh_faces[:-1])


def test_blob_save_load_roundtrip(cuda_device, tmp_path):
    v, f = synth.icosphere(4)
    r = make(v, f)
    path = str(tmp_path / "bvh.pt")
    r.save_bvh(path)
    acc = hops.AccelStructure().load(path, device=cuda_device)
    o, d = synth.random_rays(20_000, seed=2, device=cuda_device, box=True)
    a = hops.intersects_closest(r.as_wrapper, o, d)
    b = hops.intersects_closest(acc, o, d)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_numpy_adapter_follows_trimesh_ray_conventions(cuda_device):
    """SURVEY 8(f) rank 2: the call the reference benchmarks against, mesh.ray.intersects_location(o, d,
    multiple_hits=False) with numpy float64 in / numpy out (test/performance_test.py:75)."""
    from types import SimpleNamespace

    from triro.ray.ray_numpy import RayMeshIntersector as NumpyRMI

    v, f = synth.icosphere(3)
    mesh = SimpleNamespace(vertices=v.astype(np.float64), faces=f.astype(np.int64))
    ray = NumpyRMI(mesh)
    o, d = synth.random_rays(5000, seed=6, box=True)
    o64, d64 = (o * 2).numpy().astype(np.float64), d.numpy().astype(np.float64)
    loc, index_ray, index_tri = ray.intersects_location(o64, d64, multiple_hits=False)
    assert loc.dtype == np.float64 and index_ray.dtype == np.int64 and index_tri.dtype == np.int64
    r = make(v, f)
    hit, _, tri, tloc, _ = r.intersects_closest((o * 2).to(cuda_device), d.to(cuda_device))
    assert np.array_equal(index_ray, np.nonzero(hit.cpu().numpy())[0]) and np.array_equal(index_tri, tri[hit].cpu().numpy())
    assert np.allclose(loc, tloc[hit].cpu().numpy())
    loc_m, ray_m, tri_m = ray.intersects_location(o64, d64)
    assert len(loc_m) == int(r.intersects_count((o * 2).to(cuda_device), d.to(cuda_device)).clamp(max=8).sum())
    assert np.array_equal(ray.intersects_first(o64, d64), tri.cpu().numpy()) and ray.intersects_first(o64, d64).dtype == np.int64
    assert np.array_equal(ray.intersects_any(o64, d64), hit.cpu().numpy())
    t2, r2 = ray.intersects_id(o64, d64, multiple_hits=False)
    assert np.array_equal(t2, index_tri) and np.array_equal(r2, index_ray)
    assert ray.contains_points(np.array([[0, 0, 0.999], [0, 0, 1.5]])).tolist() == [True, False]


# ---------------------------------------------------------------- property test: arbitrary strided views
def test_random_strided_views_equal_their_contiguous_copies(cuda_device):
    """SURVEY §4 (4): the kernels read rays through shape[4]/stride[4] exactly like the reference's getRay
    (shaders.cu:27-63); any view must give the answer of its contiguous copy."""
    from hypothesis import given, settings, strategies as st

    v, f = synth.icosphere(2)
    r = make(v, f)
    base_o = (torch.rand((6, 5, 4, 7, 3), generator=torch.Generator().manual_seed(1)) * 4 - 2).to(cuda_device)
    base_d = torch.randn((6, 5, 4, 7, 3), generator=torch.Generator().manual_seed(2)).to(cuda_device)

    @settings(max_examples=40, deadline=None)
    @given(st.integers(1, 3), st.permutations([0, 1, 2]), st.integers(0, 3), st.integers(1, 2), st.booleans(), st.integers(0, 2),
           st.booleans())
    def run(ndim, perm, start, step, bcast_o, chan_off, neg):
        # carve a [*b, 3] view out of the 5-D base: drop leading dims, permute batch dims, slice with a step,
        # take 3 of the 7 channels with stride 2 (non-unit last-dim stride)
        def view(t):
            x = t[0] if ndim < 3 else t                       # [5,4,7,3] or [6,5,4,7,3]
            x = x[..., chan_off::2, 0][..., :3] if not neg else x[..., chan_off:chan_off + 3, 1]   # last dim 3, stride 6 or 3
            if ndim == 1:
                x = x[0, start::step]                         # [k,3]
            elif ndim == 2:
                x = x[:, start::step].transpose(0, 1)          # [k,5,3] transposed
            else:
                x = x.permute(*perm, 3)[:, start::step]
            return x
        o, d = view(base_o), view(base_d)
        if bcast_o:
            o = torch.tensor([0.3, -0.2, 2.0], device=cuda_device).broadcast_to(d.shape)
        assert o.shape == d.shape and o.shape[-1] == 3 and 1 <= o.dim() - 1 <= 3
        a = r.intersects_closest(o, d)
        b = r.intersects_closest(o.contiguous(), d.contiguous())
        for x, y in zip(a, b):
            assert x.shape == y.shape and torch.equal(x, y)
        assert torch.equal(r.intersects_count(o, d), r.intersects_count(o.contiguous(), d.contiguous()))

    run()


def test_more_than_2_to_31_rays_use_64_bit_indexing(cuda_device):
    """The reference's `int float_idx = idx * 3` overflows at 715 M rays (shaders.cu:37) and OptiX launches are
    limited to 2^30; here ray indices are 64-bit.  2.19 G rays as stride-0 broadcast views (no input memory),
    any-hit output 2.19 GB; the result must be the 27 000-ray answer tiled."""
    v, f = synth.icosphere(2)
    r = make(v, f)
    k = 27_000
    o1, d1 = synth.random_rays(k, seed=77, device=cuda_device, box=True)
    o1 = o1 * 2
    small = r.intersects_any(o1, d1)
    o = o1.unsqueeze(0).unsqueeze(0).expand(3, k, k, 3)          # strides (0, 0, 3, 1)
    d = d1.unsqueeze(0).unsqueeze(0).expand(3, k, k, 3)
    assert o.numel() // 3 > 2 ** 31
    big = r.intersects_any(o, d)
    assert big.shape == (3, k, k)
    assert torch.equal(big[0, 0], small) and torch.equal(big[2, k - 1], small) and torch.equal(big[1, 12345], small)
    assert int(big.sum()) == 3 * k * int(small.sum())


def test_fused_pinhole_generation_matches_explicit_rays(cuda_device):
    """SURVEY 8(f) rank 3: rays of the reference benchmark's camera (test/performance_test.py:10-36, its cam_mat and
    the 640x360 / f = 444 set-up) generated inside the kernel vs the explicit gen_rays tensors.  Ray directions agree to
    rounding (the kernel and torch associate the 3x3 product differently), so masks / indices must agree except on a
    handful of edge-grazing pixels and locations to 1e-5."""
    cam_mat = torch.tensor([[5.6272650e-01, 2.7091104e-01, 7.8099048e-01], [8.2602328e-01, -1.4769979e-01, -5.4393965e-01],
                            [3.2007132e-02, -9.5120555e-01, 3.0689341e-01]])
    w, h, f = 640, 360, float(int(640 * 25 / 36))
    v, fa = synth.icosphere(5)
    # put the sphere in front of that camera: camera looks along -z of cam space = -cam_mat[:, 2]
    origin = (cam_mat[:, 2] * 3.0)
    r = make(v, fa)
    dirs = synth.gen_rays(cam_mat, w, h, f, device=cuda_device)
    o = origin.to(cuda_device).broadcast_to(dirs.shape)
    exp = r.intersects_closest(o, dirs)
    got = r.intersects_closest_pinhole(cam_mat, origin, w, h, f)
    assert got[0].shape == (h, w) and got[3].shape == (h, w, 3)
    assert 0.2 < float(exp[0].float().mean()) < 0.9
    differ = (got[0] != exp[0]) | (got[2] != exp[2])
    assert int(differ.sum()) <= 1e-4 * w * h, int(differ.sum())
    same = ~differ & exp[0]
    # 1-ulp differences in the directions are amplified at silhouette pixels (grazing incidence)
    assert float((got[3][same] - exp[3][same]).abs().max()) < 5e-5
    assert float((got[3][same] - exp[3][same]).abs().mean()) < 1e-6
    assert torch.equal(got[1][same], exp[1][same])
    # compaction variant and the demo's normal interpolation post-op (test/test.py:35-42)
    c = r.intersects_closest_pinhole(cam_mat, origin, w, h, f, stream_compaction=True)
    assert torch.equal(c[0], got[0]) and torch.equal(c[3], got[2][got[0]])
    normals = torch.from_numpy(v).to(cuda_device)                      # unit sphere: vertex normal = position
    n = r.interpolate(normals, c[3], c[5])
    assert float((n - c[4]).abs().max()) < 1e-5                        # interpolated position attribute == hit location


def test_tmax_and_max_hits_extensions_keep_reference_defaults(cuda_device):
    """SURVEY 8(f) rank 4: tmax (reference: hard-coded 1e7, shaders.cu:86) and max_hits (reference: 8,
    LaunchParams.h:8) are constructor keywords; two intersectors with different settings coexist."""
    n = 40
    quads = []
    for k in range(n):
        z = -k * 0.1
        quads += [[-1, -1, z], [1, -1, z], [1, 1, z], [-1, 1, z]]
    v = torch.tensor(quads, dtype=torch.float32)
    f = torch.tensor([[4 * k + a, 4 * k + b, 4 * k + c] for k in range(n) for (a, b, c) in ((0, 1, 2), (0, 2, 3))], dtype=torch.int32)
    ref = RayMeshIntersector(vertices=v, faces=f)                               # reference defaults
    short = RayMeshIntersector(vertices=v, faces=f, tmax=5.55, max_hits=16)     # reaches z >= -0.55 from z = 5
    o = torch.tensor([[0.3, 0.2, 5.0]], device=cuda_device); d = torch.tensor([[0.0, 0.0, -1.0]], device=cuda_device)
    assert ref.intersects_count(o, d).tolist() == [40] and short.intersects_count(o, d).tolist() == [6]
    assert ref.intersects_count(o, d).tolist() == [40]                          # switching back and forth
    assert len(ref.intersects_location(o, d)[0]) == 8
    far = RayMeshIntersector(vertices=v, faces=f, max_hits=16)
    loc, ri, ti = far.intersects_location(o, d)
    assert len(loc) == 16 and len(set(ti.tolist())) == 16
    assert short.intersects_any(torch.tensor([[0.3, 0.2, 6.0]], device=cuda_device), d).tolist() == [False]   # first quad at t = 6 > tmax
    assert ref.intersects_any(torch.tensor([[0.3, 0.2, 6.0]], device=cuda_device), d).tolist() == [True]
    with pytest.raises(ValueError):
        RayMeshIntersector(vertices=v, faces=f, max_hits=65)
    with pytest.raises(ValueError):
        RayMeshIntersector(vertices=v, faces=f, tmax=-1.0)


@pytest.mark.parametrize("scale,offset", [(1e6, 0.0), (1e-6, 0.0), (1e4, 3e7)])
def test_extreme_scales_and_offsets_on_the_gpu(cuda_device, scale, offset):
    v, f = synth.icosphere(4)
    v = (v.astype(np.float64) * scale + offset).astype(np.float32)
    r = make(v, f)
    assert hostsim.check_blob(r.as_wrapper.blob.cpu().numpy())[0] == 0
    o, d = synth.random_rays(30_000, seed=11, box=True)
    o = torch.from_numpy(((o.numpy().astype(np.float64) * 2.0) * scale + offset).astype(np.float32)).to(cuda_device)
    d = d.to(cuda_device)
    got = closest_to_numpy(r.intersects_closest(o, d))
    check_closest_vs_mirror(got, oracle.OracleMesh(v, f), flat(o), flat(d))
    ref = oracle.query(oracle.OracleMesh(v, f), flat(o), flat(d), oracle.MIRROR, want=("count",))
    assert_bits_equal(r.intersects_count(o, d).cpu().numpy(), ref["count"], "count at extreme scale")


def test_readme_quickstart_reproduces_the_reference_published_figure(cuda_device):
    """README.md:24-51 run verbatim (modulo matplotlib) against the reference's published result assets/location.png
    (fixture tests/golden/readme_location_png.npz): same hit disc, same location colours."""
    from helpers import compare_with_readme_figure

    v, f = synth.icosphere(3)                                                   # trimesh.creation.icosphere()
    intersector = make(v, f)
    y, x = torch.meshgrid([torch.linspace(1, -1, 800), torch.linspace(-1, 1, 800)], indexing="ij")
    z = -torch.ones_like(x)
    ray_directions = torch.stack([x, y, z], dim=-1).cuda()
    ray_origins = torch.Tensor([0, 0, 3]).cuda().broadcast_to(ray_directions.shape)
    hit, front, ray_idx, tri_idx, location, uv = intersector.intersects_closest(ray_origins, ray_directions, stream_compaction=True)
    locs = torch.zeros((800, 800, 3)).cuda()
    locs[hit] = location
    iou, diff = compare_with_readme_figure(locs.cpu().numpy())
    assert iou > 0.985 and diff < 0.01, (iou, diff)


@pytest.mark.parametrize("tilt", [0.0, 0.3])
def test_watertight_no_leaks_on_the_gpu(cuda_device, tilt):
    """Rays aimed exactly at the vertices, edge midpoints and cell centres of a flat 128 x 128 grid: every one must hit
    (no cracks between triangles that share an edge or a vertex), bit-identical to the mirror."""
    n = 128
    v, f = synth.heightfield(n, n, amplitude=0.0)
    xs = np.linspace(-1, 1, 2 * n + 1, dtype=np.float64)[1:-1]
    gx, gy = np.meshgrid(xs, xs, indexing="xy")
    targets = np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size)], axis=1)
    origins = targets + np.array([tilt, -0.5 * tilt, 1.0]) * 2.0
    o = torch.from_numpy(origins.astype(np.float32)).to(cuda_device)
    d = torch.from_numpy((targets - origins).astype(np.float32)).to(cuda_device)
    r = make(v, f)
    hit, front, tri, loc, uv = r.intersects_closest(o, d)
    assert bool(hit.all()), f"{int((~hit).sum())} rays leaked"
    assert float(loc[:, 2].abs().max()) < 1e-6 and bool(front.all())
    got = closest_to_numpy((hit, front, tri, loc, uv))
    check_closest_vs_mirror(got, oracle.OracleMesh(v, f), flat(o), flat(d))
    assert int(r.intersects_count(o, d).min()) >= 1
    # the same through the any-hit early exit (per-ray origins: the incoherent schedule, like the queries above)
    assert bool(r.intersects_any(o, d).all())
