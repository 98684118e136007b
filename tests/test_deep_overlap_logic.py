"""CPU tier of the deep-overlap scenes (deep_overlap_cases.py): the host build of every scene is a valid blob, the host
simulation of the per-lane traversal agrees with the oracle's binary32 mirror bit for bit where a ray crosses hundreds of
triangles, and the complete-hit-list reference the GPU tests rely on agrees with the mirror itself."""
import numpy as np
import pytest

import deep_overlap_cases as dc
import hostsim
from helpers import assert_bits_equal
from oracle import oracle

CPU_RAY_SETS = ("pooled", "broadcast", "tiny33")


@pytest.mark.parametrize("name", list(dc.SCENES))
def test_host_build_of_every_scene_passes_the_full_check(name):
    v, f = dc.scene(name)
    rc, info = hostsim.check_blob(hostsim.build_blob(v, f), v, f)
    assert rc == 0, f"hs_check_blob code {rc}"
    assert info["tris"] == len(f)


@pytest.mark.parametrize("kind", CPU_RAY_SETS)
@pytest.mark.parametrize("name", list(dc.SCENES))
def test_host_simulation_equals_the_mirror_under_deep_overlap(name, kind):
    v, f = dc.scene(name)
    o, d = dc.rays(name, kind)
    blob = hostsim.build_blob(v, f)
    ref = dc.mirror(v, f, o, d)
    sim = hostsim.trace(blob, "closest", o, d)
    for k in ("hit", "front", "tri", "loc", "uv"):
        assert_bits_equal(sim[k], ref[k], f"closest.{k}")
    assert np.array_equal(hostsim.trace(blob, "count", o, d)["count"], ref["count"]), "count"
    assert np.array_equal(hostsim.trace(blob, "any", o, d)["hit"], (ref["count"] > 0).astype(np.uint8)), "any"
    if name == "dup600":                   # every hit ties in t: the smallest face index wins
        hit = ref["count"] > 0
        assert hit.any() and (ref["tri"][hit] == 0).all()


@pytest.mark.parametrize("kind", CPU_RAY_SETS)
@pytest.mark.parametrize("name", list(dc.SCENES))
def test_complete_hits_agrees_with_the_mirror(name, kind):
    """the block union has exactly count hits per ray, and the mirror's own nearest-64 list is a subset of it with the
    same location bits (complete when count <= 64)"""
    v, f = dc.scene(name)
    o, d = dc.rays(name, kind)
    ch = dc.complete_hits(v, f, o, d)
    ref = dc.mirror(v, f, o, d, want=("count",), list_cap=oracle.MAX_LIST)
    assert np.array_equal(ch["count"], ref["count"])
    assert ch["count"].max() > 0
    j = np.arange(oracle.MAX_LIST)[None, :] < ref["list_n"][:, None]
    ray = np.nonzero(j)[0]
    dc.check_hits_subset(ch, ray, ref["list_tri"][j], ref["list_loc"][j], "mirror list")
    assert np.array_equal(ref["list_n"], np.minimum(ref["count"], oracle.MAX_LIST))


def test_complete_hits_reaches_hundreds_of_hits_per_ray():
    """the scenes do what they are for: rays with far more hits than a warp's pair list holds (128) and than max_hits"""
    for name, least in (("dup600", 600), ("stack300", 300), ("mixed", 514), ("shells32", 64)):
        v, f = dc.scene(name)
        o, d = dc.rays(name, "pooled")
        assert dc.complete_hits(v, f, o, d)["count"].max() == least, name


def test_mirror_contains_matches_the_analytic_shell_parity():
    v, f = dc.scene("shells32")
    rng = np.random.default_rng(17)
    p = rng.normal(size=(3000, 3))
    p = (p / np.linalg.norm(p, axis=1, keepdims=True) * rng.uniform(0.0, 1.2, (3000, 1))).astype(np.float32)
    odd, clear = dc.shell_parity(p, 32)
    assert clear.mean() > 0.5 and odd[clear].any() and (~odd[clear]).any()
    oi = oracle.OracleIntersector(v, f, mode=oracle.MIRROR, use_bvh=False)
    for direction in ([1.0, 0.0, 0.0], [0.3, 0.5, 0.8], list(oi.DEFAULT_DIRECTION)):
        inside, cp, cm = oi.contains_core(p, direction)
        assert np.array_equal(cp[clear] % 2 == 1, odd[clear]) and np.array_equal(cm[clear] % 2 == 1, odd[clear])
        assert np.array_equal((inside & (cp % 2 == 1) & (cm % 2 == 1))[clear], odd[clear])
