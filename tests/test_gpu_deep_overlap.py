"""The trace kernels where one ray crosses tens to hundreds of triangles (deep_overlap_cases.py), against the oracle's
binary32 mirror and the complete hit list: every schedule and every knob of the warp-cooperative kernel (pair-list
threshold, re-fill threshold, lane sharing), all hits at max_hits 1...64 and in staging windows, and contains with
stop_when_broken on concentric shells.

This is where the cooperative kernel's pair list (rt_trace_coop.cuh step 3) fills and overflows, triangles that did not
fit wait in the lane for the next flush, and retirement has to wait for them."""
import numpy as np
import pytest
import torch

import deep_overlap_cases as dc
from helpers import assert_bits_equal, check_closest_vs_mirror, closest_to_numpy
from oracle import oracle
from triro.backend import ops as hops
from triro.ray.ray_optix import RayMeshIntersector

pytestmark = pytest.mark.gpu

MAX_HITS = (1, 3, 8, 13, 64)


class knobs:
    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.old = hops.set_knobs(**self.kw)

    def __exit__(self, *a):
        hops.set_knobs(**self.old)


def schedule_knobs():
    """direct once, and each cooperative schedule under every pair-list threshold, re-fill threshold and lane sharing"""
    out = [("direct", dict(schedule=hops.SCHED_DIRECT))]
    for sname, s in (("coop_coherent", hops.SCHED_COOP_COHERENT), ("coop_incoherent", hops.SCHED_COOP_INCOHERENT)):
        for tri in (0, 1, 7, 96):
            for refill in (0, 1, 32):
                for share in (1, 0):
                    out.append((f"{sname}/tri{tri}/refill{refill}/share{share}",
                                dict(schedule=s, tri_threshold=tri, refill_threshold=refill, no_lane_sharing=1 - share)))
    return out


ALLHITS_SCHEDULES = (("direct", hops.SCHED_DIRECT), ("coop_coherent", hops.SCHED_COOP_COHERENT),
                     ("coop_incoherent", hops.SCHED_COOP_INCOHERENT), ("auto", hops.SCHED_AUTO))


def make(v, f, **kw):
    return RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f), **kw)


def device_rays(name, kind, dev):
    """the scene's rays on the device: broadcast and image sets as a stride-0 origin (the coherent path)"""
    o, d = dc.rays(name, kind)
    dt = torch.from_numpy(d).to(dev)
    if kind in ("broadcast", "image"):
        ot = torch.from_numpy(o.reshape(-1, 3)[0].copy()).to(dev).broadcast_to(dt.shape)
    else:
        ot = torch.from_numpy(o).to(dev)
    return o.reshape(-1, 3), d.reshape(-1, 3), ot, dt


_ref_cache: dict = {}


def reference(name, kind):
    key = (name, kind)
    if key not in _ref_cache:
        v, f = dc.scene(name)
        o, d = dc.rays(name, kind)
        _ref_cache.clear()
        _ref_cache[key] = (dc.mirror(v, f, o, d), dc.complete_hits(v, f, o, d))
    return _ref_cache[key]


def check_allhits(res, ch, max_hits, what):
    """rays ascending, group size min(count, max_hits), distinct triangles, every hit in the complete set with its
    location bits (hence exactly the complete set where count <= max_hits)"""
    loc, ri, ti = (x.cpu().numpy() for x in res)
    cnt = ch["count"]
    assert np.all(np.diff(ri.astype(np.int64)) >= 0), f"{what}: rays not ascending"
    assert np.array_equal(np.bincount(ri, minlength=len(cnt)), np.minimum(cnt, max_hits)), f"{what}: group sizes"
    dc.check_hits_subset(ch, ri, ti, loc, what)


@pytest.mark.parametrize("kind", dc.RAY_SETS)
@pytest.mark.parametrize("name", list(dc.SCENES))
def test_every_schedule_and_knob_equals_the_mirror(cuda_device, name, kind):
    v, f = dc.scene(name)
    on, dn, o, d = device_rays(name, kind, cuda_device)
    ref, ch = reference(name, kind)
    assert np.array_equal(ref["count"], ch["count"])
    r = make(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=False)
    for label, kw in schedule_knobs():
        with knobs(**kw):
            got = closest_to_numpy(r.intersects_closest(o, d))
            first = r.intersects_first(o, d).cpu().numpy().reshape(-1)
            cnt = r.intersects_count(o, d).cpu().numpy().reshape(-1)
            anyh = r.intersects_any(o, d).cpu().numpy().reshape(-1)
        for k in ("hit", "front", "tri", "loc", "uv"):
            assert_bits_equal(got[k], ref[k], f"{label} closest.{k}")
        assert np.array_equal(first, ref["tri"]), f"{label} first"
        assert np.array_equal(cnt, ref["count"]), f"{label} count: {int((cnt != ref['count']).sum())} rays differ"
        assert np.array_equal(anyh, ref["count"] > 0), f"{label} any"
    check_closest_vs_mirror(got, om, on, dn)


@pytest.mark.parametrize("kind", dc.RAY_SETS)
@pytest.mark.parametrize("name", list(dc.SCENES))
def test_all_hits_at_every_max_hits_are_hits_of_the_mirror(cuda_device, name, kind):
    v, f = dc.scene(name)
    _, _, o, d = device_rays(name, kind, cuda_device)
    _, ch = reference(name, kind)
    for mh in MAX_HITS:
        r = make(v, f, max_hits=mh)
        for label, s in ALLHITS_SCHEDULES:
            with knobs(schedule=s):
                ti, ri, loc = r.intersects_id(o, d, return_locations=True)
            check_allhits((loc, ri, ti), ch, mh, f"{label} max_hits={mh}")


@pytest.mark.parametrize("name,max_hits", [("coplanar200", 13), ("coplanar200", 64), ("mixed", 13), ("mixed", 64),
                                           ("shells32", 64)])
def test_all_hits_in_staging_windows_equal_one_launch(cuda_device, name, max_hits):
    """windows of 3000 and 5111 rays (not multiples of the 2048-ray scan tile) give the same packed result as one launch,
    up to the order within a ray; rays with count <= max_hits have the same hit set whatever the order of tests"""
    v, f = dc.scene(name)
    r = make(v, f)
    o1, d1 = dc.rays(name, "pooled", seed=1)
    o2, d2 = dc.rays(name, "pooled", seed=2)
    o = torch.from_numpy(np.concatenate([o1, o2, o1[:1500]])).to(cuda_device)
    d = torch.from_numpy(np.concatenate([d1, d2, d1[:1500]])).to(cuda_device)
    n = o.shape[0]
    cnt = r.intersects_count(o, d).cpu().numpy()
    few = cnt <= max_hits
    assert (few & (cnt > 0)).mean() > 0.05

    def canon(res):
        loc, ri, ti = (x.cpu().numpy() for x in res)
        keep = few[ri]
        loc, ri, ti = loc[keep], ri[keep], ti[keep]
        order = np.lexsort((ti, ri))
        return ri[order], ti[order], loc[order].view(np.uint32)

    one = hops.intersects_location(r.as_wrapper, o, d, max_hits)
    assert np.array_equal(np.bincount(one[1].cpu().numpy(), minlength=n), np.minimum(cnt, max_hits))
    for window in (3000, 5111):
        many = hops.intersects_location(r.as_wrapper, o, d, max_hits, staging_bytes=window * max_hits * 16)
        assert hops.allhits_window_rays(max_hits, window * max_hits * 16) == window
        assert torch.equal(one[1], many[1]), f"window {window}: ray indices"
        for a, b in zip(canon(one), canon(many)):
            assert np.array_equal(a, b), f"window {window}"


def _shell_points(dev, n, lo, hi, seed):
    rng = np.random.default_rng(seed)
    p = rng.normal(size=(n, 3))
    p = (p / np.linalg.norm(p, axis=1, keepdims=True) * rng.uniform(lo, hi, (n, 1))).astype(np.float32)
    return p, torch.from_numpy(p).to(dev)


@pytest.mark.parametrize("sched", ["direct", "coop_incoherent", "auto"])
def test_contains_on_shells_equals_the_mirror_and_the_analytic_parity(cuda_device, sched):
    v, f = dc.scene("shells32")
    r = make(v, f)
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR, use_bvh=False)
    p, pt = _shell_points(cuda_device, 20_000, 0.0, 1.2, 5)
    odd, clear = dc.shell_parity(p, 32)
    s = {"direct": hops.SCHED_DIRECT, "coop_incoherent": hops.SCHED_COOP_INCOHERENT, "auto": hops.SCHED_AUTO}[sched]
    for direction in ([1.0, 0.0, 0.0], [0.3, 0.5, 0.8], list(r.DEFAULT_CHECK_DIRECTION)):
        with knobs(schedule=s):
            contain, broken, flags = r.contains_parity(pt, direction)
        inside, cp, cm = oi.contains_core(p, direction)
        agree = (cp % 2 == 1) & (cm % 2 == 1)
        want_broken = ~agree & ((cp == 0) | (cm == 0))
        assert np.array_equal(contain.cpu().numpy(), inside & agree), f"{direction} contain"
        assert np.array_equal(broken.cpu().numpy(), want_broken), f"{direction} broken"
        assert flags.tolist() == [int(inside.any()), int(want_broken.any())]
        assert np.array_equal(contain.cpu().numpy()[clear], odd[clear]), f"{direction} analytic parity"


def test_stop_when_broken_on_shells(cuda_device):
    v, f = dc.scene("shells32")
    r = make(v, f)
    direction = [0.3, 0.5, 0.8]
    # inside the outermost shell, away from every shell: no point is broken, the flag must change nothing
    p, pt = _shell_points(cuda_device, 30_000, 0.0, 0.95 * dc.shell_inradius_factor(), 7)
    clear = dc.shell_parity(p, 32)[1]
    pt = pt[torch.from_numpy(clear).to(cuda_device)].contiguous()
    c0, b0, f0 = r.contains_parity(pt, direction)
    c1, b1, f1 = r.contains_parity(pt, direction, stop_when_broken=True)
    assert f0.tolist() == [1, 0] and not bool(b0.any())
    assert torch.equal(c0, c1) and torch.equal(b0, b1) and torch.equal(f0, f1)
    # points outside every shell are broken (the line through them meets the shells on one side at most)
    q, qt = _shell_points(cuda_device, 30_000, 0.0, 1.6, 8)
    _, _, f2 = r.contains_parity(qt, direction, stop_when_broken=True)
    assert f2.tolist()[1] == 1
    # masked retry: `active` aliases `broken`; only the active entries may change, and they get the mirror's answer
    contain, broken, _ = r.contains_parity(qt, direction)
    c_before, b_before = contain.clone(), broken.clone()
    assert bool(b_before.any()) and not bool(b_before.all())
    retry = [0.1, -0.7, 0.2]
    c3, b3, f3 = r.contains_parity(qt, retry, active=broken, out=(contain, broken))
    keep = ~b_before
    assert torch.equal(c3[keep], c_before[keep]) and torch.equal(b3[keep], b_before[keep])
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR, use_bvh=False)
    inside, cp, cm = oi.contains_core(q, retry)
    agree = (cp % 2 == 1) & (cm % 2 == 1)
    m = b_before.cpu().numpy()
    assert np.array_equal(c3.cpu().numpy()[m], (inside & agree)[m])
    assert np.array_equal(b3.cpu().numpy()[m], (~agree & ((cp == 0) | (cm == 0)))[m])
    assert f3.tolist() == [int(inside[m].any()), int((~agree & ((cp == 0) | (cm == 0)))[m].any())]
