"""GPU tests added in round 2: every traversal schedule gives the same bits, ray windows, bounded all-hits
staging, the masked contains retry, the compacting host-buffer entry point, blob validation / refit of adopted
blobs — and parity against the oracle's binary32 mirror on the TRUE-SIZE meshes of BASELINE configs 3, 4 and 5
(>= 1 M-ray subsamples; the oracle walks its own binned-SAH BVH2 of the full mesh on the host cores).
"""
import numpy as np
import pytest
import torch

import hostsim
from helpers import assert_bits_equal, check_closest_vs_mirror, closest_to_numpy
from oracle import oracle
from triro import synth
from triro.backend import ops as hops
from triro.ray.ray_optix import RayMeshIntersector

pytestmark = pytest.mark.gpu

# SCHED_QUEUED and SCHED_SLOTS name removed schedules: ABI v2 callers that still pass them must get the same bits
SCHEDULES = {"direct": hops.SCHED_DIRECT, "coop_coherent": hops.SCHED_COOP_COHERENT, "coop_incoherent": hops.SCHED_COOP_INCOHERENT,
             "legacy_queued": hops.SCHED_QUEUED, "legacy_slots": hops.SCHED_SLOTS}


def make(v, f, **kw):
    return RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f), **kw)


def flat(t):
    return t.detach().cpu().numpy().reshape(-1, 3)


class knobs:
    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.old = hops.set_knobs(**self.kw)

    def __exit__(self, *a):
        hops.set_knobs(**self.old)


# ---------------------------------------------------------------- schedules
@pytest.mark.parametrize("scene", ["camera_ico5", "random_soup20k"])
def test_all_schedules_give_identical_results(cuda_device, scene):
    """direct (per-lane triangle tests, round 1), the two warp-cooperative schedules and the legacy numbers must agree bit
    for bit on every query, for any pair-list threshold: the closest hit is resolved by (t, primitive index),
    never by test order."""
    if scene == "camera_ico5":
        v, f = synth.icosphere(5)
        o, d = synth.pinhole_rays(640, 360, device=cuda_device)
        pts = (torch.rand((50_000, 3), device=cuda_device, generator=torch.Generator(cuda_device).manual_seed(3)) * 2 - 1) * 1.1
    else:
        v, f = synth.triangle_soup(20_000, sigma=0.02, seed=5)
        o, d = synth.random_rays(300_000, seed=6, device=cuda_device, box=True)
        pts = o[:50_000].contiguous()
    r = make(v, f)
    base = None
    for name, sched in SCHEDULES.items():
        for thr in ((0,) if sched == hops.SCHED_DIRECT else (0, 1, 7, 96)):
            with knobs(schedule=sched, tri_threshold=thr):
                got = dict(closest=closest_to_numpy(r.intersects_closest(o, d)), first=r.intersects_first(o, d).cpu().numpy(),
                           any=r.intersects_any(o, d).cpu().numpy(), count=r.intersects_count(o, d).cpu().numpy())
                c, b, fl = r.contains_parity(pts, [0.3, 0.5, 0.8])
                got["contains"] = (c.cpu().numpy(), b.cpu().numpy(), fl.cpu().numpy())
            if base is None:
                base = got
                continue
            for k in base["closest"]:
                assert_bits_equal(got["closest"][k], base["closest"][k], f"{name}/{thr} closest.{k}")
            for k in ("first", "any", "count"):
                assert np.array_equal(got[k], base[k]), f"{name}/{thr} {k}"
            for a, b_ in zip(got["contains"], base["contains"]):
                assert np.array_equal(a, b_), f"{name}/{thr} contains"
    om = oracle.OracleMesh(v, f)
    check_closest_vs_mirror(base["closest"], om, flat(o), flat(d))


@pytest.mark.parametrize("n_rays", [1, 33, 5_000, 200_000])
def test_lane_sharing_in_the_launch_tail_changes_no_bit(cuda_device, n_rays):
    """Lanes of a warp that can draw no more rays walk parts of their neighbours' traversal stacks (rt_trace_coop.cuh,
    step 1b).  Small launches on a soup are nearly all tail: with sharing on (default), off
    (RT_OPT_NO_LANE_SHARING) and under the per-lane round-1 kernel every query must give the same bits, and the
    closest hit must equal the oracle's."""
    v, f = synth.triangle_soup(30_000, sigma=0.03, seed=11)
    o, d = synth.random_rays(n_rays, seed=12, device=cuda_device, box=True)
    pts = o[: min(n_rays, 20_000)].contiguous()
    r = make(v, f)
    res = []
    for kw in (dict(), dict(no_lane_sharing=1), dict(schedule=hops.SCHED_COOP_COHERENT), dict(schedule=hops.SCHED_DIRECT)):
        with knobs(**kw):
            got = dict(closest=closest_to_numpy(r.intersects_closest(o, d)), first=r.intersects_first(o, d).cpu().numpy(),
                       any=r.intersects_any(o, d).cpu().numpy(), count=r.intersects_count(o, d).cpu().numpy())
            c, b, fl = r.contains_parity(pts, [0.3, 0.5, 0.8])
            got["contains"] = (c.cpu().numpy(), b.cpu().numpy(), fl.cpu().numpy())
            loc, ray_idx, tri_idx = r.intersects_location(o, d)
            key = np.lexsort((tri_idx.cpu().numpy(), ray_idx.cpu().numpy()))
            got["location"] = (ray_idx.cpu().numpy()[key], tri_idx.cpu().numpy()[key], loc.cpu().numpy()[key])
        res.append(got)
    cnt = res[0]["count"]
    for got in res[1:]:
        for k in got["closest"]:
            assert_bits_equal(got["closest"][k], res[0]["closest"][k], f"closest.{k}")
        for k in ("first", "any", "count"):
            assert np.array_equal(got[k], res[0][k]), k
        for a, b_ in zip(got["contains"], res[0]["contains"]):
            assert np.array_equal(a, b_), "contains"
        if cnt.max(initial=0) <= 8:          # beyond max_hits the recorded subset is test order (reference: traversal order)
            for a, b_ in zip(got["location"], res[0]["location"]):
                assert_bits_equal(a, b_, "location")
    om = oracle.OracleMesh(v, f)
    check_closest_vs_mirror(res[0]["closest"], om, flat(o), flat(d))


@pytest.mark.parametrize("shape", [(64, 96), (4, 8), (36, 40), (30, 64), (64, 36), (3, 32, 64), (1, 2048)])
def test_tile_work_order_of_image_batches_changes_no_bit(cuda_device, shape):
    """Coherent image batches [H, W, 3] with H % 4 == 0 and W % 8 == 0 are traced in 8x4-pixel tiles per warp (rt_trace.cu
    tile_order); other shapes and batches of several images keep the row order.  Results are indexed by ray: tile order
    on / off (RT_OPT_NO_TILE_ORDER) and the oracle must agree on every bit, whatever the shape."""
    v, f = synth.icosphere(4)
    g = torch.Generator().manual_seed(21)
    d = torch.randn((*shape, 3), generator=g)
    d[..., 2] = -d[..., 2].abs() - 0.3
    d = d.to(cuda_device)
    o = torch.tensor([0.05, -0.02, 3.0], device=cuda_device).broadcast_to(d.shape)
    r = make(v, f)
    res = []
    for kw in (dict(), dict(no_tile_order=1), dict(schedule=hops.SCHED_DIRECT)):
        with knobs(**kw):
            got = dict(closest=closest_to_numpy(r.intersects_closest(o, d)), first=r.intersects_first(o, d).cpu().numpy(),
                       any=r.intersects_any(o, d).cpu().numpy(), count=r.intersects_count(o, d).cpu().numpy())
            h6 = r.intersects_closest(o, d, stream_compaction=True)
            got["compact"] = tuple(x.cpu().numpy() for x in h6)
            loc, ray_idx, tri_idx = r.intersects_location(o, d)
            key = np.lexsort((tri_idx.cpu().numpy(), ray_idx.cpu().numpy()))
            got["location"] = (ray_idx.cpu().numpy()[key], tri_idx.cpu().numpy()[key], loc.cpu().numpy()[key])
        res.append(got)
    assert res[0]["count"].shape == tuple(shape)
    for got in res[1:]:
        for k in got["closest"]:
            assert_bits_equal(got["closest"][k], res[0]["closest"][k], f"closest.{k}")
        for k in ("first", "any", "count"):
            assert np.array_equal(got[k], res[0][k]), k
        for a, b_ in zip(got["compact"], res[0]["compact"]):
            assert_bits_equal(a, b_, "compact")
        for a, b_ in zip(got["location"], res[0]["location"]):
            assert_bits_equal(a, b_, "location")
    om = oracle.OracleMesh(v, f)
    check_closest_vs_mirror(res[0]["closest"], om, flat(o), flat(d))


@pytest.mark.parametrize("mesh", ["cube", "flat_plane", "slab_heightfield", "far_offset_cube"])
def test_root_frame_pretest_rejects_only_rays_that_hit_nothing(cuda_device, mesh):
    """Pooled kernels test every ray against the box that bounds the root's children before it may take a lane, and
    write the miss of a rejected ray at once (rt_trace_coop.cuh fill_pool_frame / rt_core.cuh frame_missed).  Rays that
    graze that box - along faces, through edges and corners, starting on it, inside a zero-thickness frame - must come
    out exactly as the oracle's brute-force mirror says: closest hit, count and any."""
    if mesh in ("cube", "far_offset_cube"):
        c = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], np.float32)
        f = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5], [0, 4, 7], [0, 7, 3]], np.int32)
        v = c + (np.array([1000.25, -2000.5, 3000.125], np.float32) if mesh == "far_offset_cube" else 0)
    elif mesh == "flat_plane":
        v, f = synth.heightfield(8, 8)
        v = v.copy(); v[:, 2] = 0.25                       # zero-thickness root frame
    else:
        v, f = synth.heightfield(64, 32)
    lo, hi = v.min(0), v.max(0)
    g = np.random.default_rng(31)
    n = 40_000
    o = np.empty((n, 3), np.float32); d = np.empty((n, 3), np.float32)
    # origins on / just off the bounding planes, directions along the axes, the face diagonals, towards corners, random
    grid = np.stack([lo, (lo + hi) / 2, hi, lo - (hi - lo + 1) * 0.5, hi + (hi - lo + 1) * 0.5])      # 5 x 3 coordinates per axis
    o[:] = grid[g.integers(0, 5, (n, 3)), np.arange(3)]
    kind = g.integers(0, 4, n)
    axes = np.eye(3, dtype=np.float32)[g.integers(0, 3, n)] * g.choice([-1.0, 1.0], (n, 1))
    diag = g.choice([-1.0, 0.0, 1.0], (n, 3)).astype(np.float32)
    diag[(diag == 0).all(1)] = [1, 0, 0]
    corner = grid[g.integers(0, 3, (n, 3)), np.arange(3)] - o
    corner[(corner == 0).all(1)] = [0, 0, 1]
    rnd = g.normal(size=(n, 3)).astype(np.float32)
    d[:] = np.where((kind == 0)[:, None], axes, np.where((kind == 1)[:, None], diag, np.where((kind == 2)[:, None], corner, rnd)))
    jitter = g.integers(0, 3, n)                            # a third of the origins move by one ulp
    o = np.where((jitter == 1)[:, None], np.nextafter(o, np.float32(np.inf)), np.where((jitter == 2)[:, None], np.nextafter(o, np.float32(-np.inf)), o)).astype(np.float32)
    ot, dt = torch.from_numpy(o).to(cuda_device), torch.from_numpy(d.astype(np.float32)).to(cuda_device)
    r = make(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=False)
    got = closest_to_numpy(r.intersects_closest(ot, dt))
    check_closest_vs_mirror(got, om, o, d.astype(np.float32))
    ref = oracle.query(om, o, d.astype(np.float32), oracle.MIRROR, want=("count",))["count"]
    assert np.array_equal(r.intersects_count(ot, dt).cpu().numpy(), ref), "count vs mirror"
    assert np.array_equal(r.intersects_any(ot, dt).cpu().numpy(), ref > 0), "any vs mirror"
    with knobs(schedule=hops.SCHED_DIRECT):                # the per-lane kernel has no pre-test
        assert np.array_equal(r.intersects_count(ot, dt).cpu().numpy(), ref)
    assert 0.02 < (ref > 0).mean() < 0.98


def test_trace_stats_direct_equals_host_simulation_and_coop_never_skips(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    o, d = synth.readme_rays(200, device=cuda_device)
    sim = hostsim.trace(r.as_wrapper.blob.cpu().numpy(), "closest", flat(o), flat(d))
    with knobs(schedule=hops.SCHED_DIRECT):
        st = hops.trace_stats(r.as_wrapper, o, d, "closest")
    assert st["rays"] == 40_000 and st["nodes"] == sim["stats"]["nodes"] and st["tris"] == sim["stats"]["tris"]
    # the cooperative schedule tests triangles a little later (tmax shrinks later): never fewer visits, same hits
    sc = hops.trace_stats(r.as_wrapper, o, d, "closest")
    assert sc["rays"] == 40_000 and sc["hits"] == st["hits"] and sc["nodes"] >= st["nodes"] and sc["tris"] >= st["tris"]
    assert sc["nodes"] <= 1.25 * st["nodes"]


# ---------------------------------------------------------------- ray windows / bounded staging
def test_ray_window_equals_slice_of_the_full_result(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    o, d = synth.random_rays(7 * 11 * 13, seed=21, device=cuda_device, box=True)
    big = torch.zeros((7, 11, 13, 5), device=cuda_device)
    big[..., :3] = d.reshape(7, 11, 13, 3)
    dv = big[..., :3]                                     # strided view (row pitch 5 floats)
    ov = (o * 1.4).reshape(7, 11, 13, 3)
    full = closest_to_numpy(r.intersects_closest(ov, dv))
    n = 7 * 11 * 13
    for lo, cnt in ((0, 1), (5, 100), (333, n - 333), (n - 1, 1), (17, 0)):
        got = closest_to_numpy(hops.intersects_closest(r.as_wrapper, ov, dv, lo, cnt))
        for k in full:
            assert_bits_equal(got[k], full[k][lo:lo + cnt], f"window [{lo}, +{cnt}) {k}")
    with pytest.raises(ValueError):
        hops.intersects_closest(r.as_wrapper, ov, dv, n - 3, 10)
    # broadcast origin: the window needs no materialised copy of the origins
    oc, dc = synth.pinhole_rays(300, 200, device=cuda_device)
    fullc = closest_to_numpy(r.intersects_closest(oc, dc))
    got = closest_to_numpy(hops.intersects_closest(r.as_wrapper, oc, dc, 12_345, 20_000))
    for k in fullc:
        assert_bits_equal(got[k], fullc[k][12_345:32_345], f"camera window {k}")


def test_allhits_in_bounded_staging_windows_equals_one_launch(cuda_device):
    v, f = synth.triangle_soup(20_000, sigma=0.03, seed=11)
    r = make(v, f)
    o, d = synth.random_rays(40_000, seed=12, device=cuda_device, box=True)
    one = hops.intersects_location(r.as_wrapper, o, d, 8)
    many = hops.intersects_location(r.as_wrapper, o, d, 8, staging_bytes=3000 * 8 * 16)      # 14 windows
    assert one[1].shape[0] > 10_000

    few = (r.intersects_count(o, d) <= 8).cpu().numpy()       # with more than 8 hits WHICH 8 are kept is unspecified (as in the reference)

    def canon(res):        # hits of one ray come in traversal order, which depends on what shares its warp: sort within the ray
        loc, ri, ti = (x.cpu().numpy() for x in res)
        keep = few[ri]
        loc, ri, ti = loc[keep], ri[keep], ti[keep]
        order = np.lexsort((ti, ri))
        return ri[order], ti[order], loc[order].view(np.uint32)

    assert torch.equal(one[1], many[1]) and bool((one[1][1:] >= one[1][:-1]).all())     # same rays, ascending
    for a, b in zip(canon(one), canon(many)):
        assert np.array_equal(a, b)
    assert hops.allhits_window_rays(8) * 8 * 16 <= hops.ALLHITS_STAGING_BYTES
    # what a 100 M-ray config-3 call allocates at a time: <= 2 GiB instead of 12.8 GB
    assert hops.allhits_window_rays(8) == (2 << 30) // 128


# ---------------------------------------------------------------- contains_points
def test_contains_default_direction_retry_is_masked_and_matches_the_reference_flow(cuda_device):
    v, f = synth.icosphere(3)
    f_open = f[1:]                                         # open mesh: points under the hole have odd/even counts
    r = make(v, f_open)
    g = torch.Generator().manual_seed(5)
    pts = ((torch.rand((20_000, 3), generator=g) * 2 - 1) * 1.2)
    oi = oracle.OracleIntersector(v, f_open, mode=oracle.MIRROR)
    torch.manual_seed(99)
    want = oi.contains_points(pts.numpy())
    torch.manual_seed(99)
    got = r.contains_points(pts.to(cuda_device))
    assert np.array_equal(got.cpu().numpy(), want)
    # the masked launch itself: only active entries change
    p = pts.to(cuda_device)
    contain, broken, _ = r.contains_parity(p, r.DEFAULT_CHECK_DIRECTION)
    c0, b0 = contain.clone(), broken.clone()
    assert bool(b0.any())
    c1, b1, flags = r.contains_parity(p, [0.1, -0.7, 0.2], active=broken, out=(contain, broken))
    assert torch.equal(c1[~b0], c0[~b0]) and torch.equal(b1[~b0], b0[~b0])
    inside, cp, cm = oi.contains_core(pts.numpy(), [0.1, -0.7, 0.2])
    agree = (cp % 2 == 1) & (cm % 2 == 1)
    m = b0.cpu().numpy()
    assert np.array_equal(c1.cpu().numpy()[m], (inside & agree)[m])
    assert np.array_equal(b1.cpu().numpy()[m], (~agree & ((cp == 0) | (cm == 0)))[m])
    assert flags.tolist() == [int(inside[m].any()), int((~agree & ((cp == 0) | (cm == 0)))[m].any())]


# ---------------------------------------------------------------- host-buffer entry point with compaction
def test_host_compact_entry_point_matches_device_compaction(cuda_device):
    v, f = synth.icosphere(5)
    r = make(v, f)
    o, d = synth.pinhole_rays(1500, 900, device="cpu")          # 1.35 M rays -> several ramped chunks
    d = d.reshape(-1, 3).contiguous().pin_memory()
    o1 = torch.tensor([0.0, 0.0, 3.0]).pin_memory()
    out = hops.host_closest(r.as_wrapper, o1, d, stream_compaction=True)
    hit, front, ray_idx, tri, loc, uv = r.intersects_closest(o1.to(cuda_device).broadcast_to(d.shape), d.to(cuda_device),
                                                             stream_compaction=True)
    assert out["n_hit"] == ray_idx.shape[0] > 100_000
    assert torch.equal(out["hit"], hit.cpu())
    for k, t in (("front_c", front), ("ray_idx_c", ray_idx), ("tri_c", tri), ("loc_c", loc), ("uv_c", uv)):
        assert torch.equal(out[k], t.cpu()), k
    # reuse of the output dict / device work buffer
    out2 = hops.host_closest(r.as_wrapper, o1, d, out=out, stream_compaction=True)
    assert out2["n_hit"] == out["n_hit"] and torch.equal(out2["tri_c"], tri.cpu())


# ---------------------------------------------------------------- blob hygiene
def test_adopt_validates_the_header_and_adopted_blobs_refit(cuda_device):
    v, f = synth.icosphere(4)
    r = make(v, f)
    used = r.as_wrapper._inner.used().clone()
    assert hostsim.check_blob(used.cpu().numpy())[0] == 0
    acc = hops.AccelStructure().adopt(used)                                   # what a non-src rank / load() holds
    v2 = (v * np.array([0.8, 1.3, 1.0], np.float32)).astype(np.float32)
    acc.refit(torch.from_numpy(v2).to(cuda_device), r.mesh_faces)              # needs only the used prefix
    fresh = make(v2, f)
    o, d = synth.random_rays(30_000, seed=4, device=cuda_device, box=True)
    for a, b in zip(hops.intersects_closest(acc, o * 1.5, d), fresh.intersects_closest(o * 1.5, d)):
        assert torch.equal(a, b)
    with pytest.raises(ValueError):
        hops.AccelStructure().adopt(used[: used.numel() // 2].clone())         # truncated
    bad = used.clone()
    bad[16:20] = torch.tensor([61, 0, 0, 0], dtype=torch.uint8, device=cuda_device)   # depth 61 > traversal stack
    with pytest.raises(RuntimeError):
        hops.AccelStructure().adopt(bad)
    bad = used.clone()
    bad[0] = 0
    with pytest.raises(ValueError):
        hops.AccelStructure().adopt(bad)
    if torch.cuda.device_count() > 1:
        o2, d2 = synth.random_rays(10, seed=1, device="cuda:1", box=True)
        with pytest.raises(ValueError):
            r.intersects_any(o2, d2)
        from triro.ray.ray_numpy import RayMeshIntersector as NP

        rn = NP(vertices=v, faces=f, device="cuda:1")                          # second device in the same process
        assert rn.intersects_any(np.array([[0, 0, 3.0]]), np.array([[0, 0, -1.0]])).tolist() == [True]


# ---------------------------------------------------------------- true-size parity (BASELINE configs 3, 4, 5)
def _parity_block(r, om, o, d, what=("closest", "count", "any")):
    on, dn = flat(o), flat(d)
    if "closest" in what:
        check_closest_vs_mirror(closest_to_numpy(r.intersects_closest(o, d)), om, on, dn)
    if "count" in what or "any" in what:
        ref = oracle.query(om, on, dn, oracle.MIRROR, want=("count",))["count"]
        if "count" in what:
            assert np.array_equal(r.intersects_count(o, d).cpu().numpy(), ref), "count vs mirror"
        if "any" in what:
            assert np.array_equal(r.intersects_any(o, d).cpu().numpy(), ref > 0), "any vs mirror"


def test_config3_true_size_heightfield_vs_oracle(cuda_device):
    v, f = synth.heightfield(2048, 1024)                   # 4 194 304 triangles
    r = make(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    o, d = synth.random_rays(1_000_000, seed=1234, device=cuda_device)
    _parity_block(r, om, o, d)


def test_config4_true_size_soup_vs_oracle(cuda_device):
    v, f = synth.triangle_soup(1_000_000)
    r = make(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    o, d = synth.random_rays(1_000_000, seed=9, device=cuda_device, box=True)
    _parity_block(r, om, o, d, what=("closest", "count"))
    # all hits: per-ray sets of (triangle, location) against the oracle's lists (rays with <= 8 hits)
    m = 200_000
    loc, ri, ti = r.intersects_location(o[:m], d[:m])
    ref = oracle.query(om, flat(o[:m]), flat(d[:m]), oracle.MIRROR, list_cap=16, want=("count",))
    cnt = np.minimum(ref["count"], 8)
    assert loc.shape[0] == int(cnt.sum())
    ri_n, ti_n, loc_n = ri.cpu().numpy(), ti.cpu().numpy(), loc.cpu().numpy()
    assert np.array_equal(np.bincount(ri_n, minlength=m), cnt)
    off = np.concatenate([[0], np.cumsum(cnt)])
    ok = np.nonzero((ref["count"] <= 8) & (cnt > 0))[0]
    for i in ok[:: max(1, len(ok) // 20_000)]:
        k = cnt[i]
        order_g = np.argsort(ti_n[off[i]:off[i] + k]); order_r = np.argsort(ref["list_tri"][i, :k])
        assert np.array_equal(ti_n[off[i]:off[i] + k][order_g], ref["list_tri"][i, :k][order_r])
        assert np.array_equal(loc_n[off[i]:off[i] + k][order_g].view(np.uint32), ref["list_loc"][i, :k][order_r].view(np.uint32))
    # contains_points core with the +x direction on 200 k points
    g = torch.Generator(device=cuda_device); g.manual_seed(8)
    pts = torch.rand((200_000, 3), generator=g, device=cuda_device) * 2 - 1
    oi = oracle.OracleIntersector.__new__(oracle.OracleIntersector)
    oi.mesh, oi.mode, oi.mesh_aabb = om, oracle.MIRROR, (v.min(axis=0), v.max(axis=0))
    inside, cp, cm = oi.contains_core(pts.cpu().numpy(), [1.0, 0.0, 0.0])
    agree = (cp % 2 == 1) & (cm % 2 == 1)
    contain, broken, flags = r.contains_parity(pts, [1.0, 0.0, 0.0])
    assert np.array_equal(contain.cpu().numpy(), inside & agree)
    assert np.array_equal(broken.cpu().numpy(), ~agree & ((cp == 0) | (cm == 0)))


def test_config5_true_size_16m_heightfield_vs_oracle(cuda_device):
    v, f = synth.heightfield(4096, 2048)                   # 16 777 216 triangles, blob ~1 GB > L2
    r = make(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    o, d = synth.random_rays(1_000_000, seed=100, device=cuda_device)
    _parity_block(r, om, o, d, what=("closest",))
    hit, front, ray_idx, tri_idx, loc, uv = r.intersects_closest(o, d, stream_compaction=True)
    assert torch.equal(ray_idx.long(), torch.nonzero(hit).reshape(-1))
