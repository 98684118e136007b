"""CPU-only coverage of the product's builder / traversal LOGIC: the __host__ __device__ functions of
trimesh-ray-optix_b200/csrc (Morton codes, Karras hierarchy, BVH8 collapse + quantisation, node
test, watertight triangle test, traversal state machine) are stepped on the CPU by tests/hostsim
and compared with the oracle.  (The CUDA kernels themselves are covered by the -m gpu tests.)"""
import os

import numpy as np
import pytest

import hostsim
from oracle import oracle
from triro import synth


def mesh(name):
    if name.startswith("tri"):
        n = int(name[3:])
        rng = np.random.default_rng(n)
        return rng.uniform(-1, 1, size=(3 * n, 3)).astype(np.float32), np.arange(3 * n, dtype=np.int32).reshape(n, 3)
    if name.startswith("ico"):
        return synth.icosphere(int(name[3:]))
    if name == "soup":
        return synth.triangle_soup(5000, sigma=0.03, seed=3)
    if name == "hf":
        return synth.heightfield(48, 24)
    if name == "cube":
        return synth.cube()
    if name == "dup":       # many identical Morton codes: 64 copies of the same triangle + a degenerate one
        v = np.tile(np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0]], np.float32), (65, 1))
        v[-3:] = 1.0
        return v, np.arange(195, dtype=np.int32).reshape(65, 3)
    raise KeyError(name)


MESHES = ["tri1", "tri2", "tri3", "tri4", "tri9", "ico0", "ico2", "ico4", "soup", "hf", "cube", "dup"]


@pytest.mark.parametrize("name", MESHES)
def test_blob_structure_and_conservative_quantisation(name):
    v, f = mesh(name)
    blob = hostsim.build_blob(v, f)
    code, info = hostsim.check_blob(blob, v, f)
    assert code == 0, f"hs_check_blob -> {code}"
    assert info["tris"] == len(f)
    assert np.array_equal(np.sort(hostsim.blob_prims(blob, len(f))), np.arange(len(f)))
    assert info["depth"] <= 60
    if len(f) > 64:
        # node pool bound used by rt_bvh_sizes (wide_node_cap, rt_core.cuh) for the builder's leaf size
        leaf = min(3, max(1, int(os.environ.get("TRIRO_LEAF_TRIS", "2"))))
        n = len(f)
        assert info["nodes"] <= {3: n // 3 + 2, 2: (2 * n) // 5 + 2, 1: (5 * n) // 8 + 2}[leaf]


@pytest.mark.parametrize("name", MESHES)
def test_traversal_matches_oracle_mirror_bit_for_bit(name):
    v, f = mesh(name)
    blob = hostsim.build_blob(v, f)
    o, d = synth.random_rays(4000, seed=len(f), box=True)
    o, d = (o * 1.5).numpy(), d.numpy()
    # axis-aligned and zero-component directions exercise the slab test's +-tiny substitution
    d[:200] = np.eye(3, dtype=np.float32)[np.arange(200) % 3] * np.where(np.arange(200) % 2, 1, -1)[:, None]
    om = oracle.OracleMesh(v, f, use_bvh=False)
    ref = oracle.query(om, o, d, oracle.MIRROR)
    got = hostsim.trace(blob, "closest", o, d)
    for k in ("hit", "front", "tri"):
        assert np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["loc"].view(np.uint32), ref["loc"].view(np.uint32))
    assert np.array_equal(got["uv"].view(np.uint32), ref["uv"].view(np.uint32))
    assert np.array_equal(hostsim.trace(blob, "count", o, d)["count"], ref["count"])
    assert np.array_equal(hostsim.trace(blob, "any", o, d)["hit"], (ref["count"] > 0).astype(np.uint8))
    assert got["max_stack"] <= hostsim.check_blob(blob)[1]["depth"]


def test_traversal_matches_truth_outside_grazing_set():
    v, f = synth.icosphere(4)
    blob = hostsim.build_blob(v, f)
    o, d = synth.pinhole_rays(160, 90)
    o, d = o.numpy().reshape(-1, 3), d.numpy().reshape(-1, 3)
    ref = oracle.query(oracle.OracleMesh(v, f), o, d, oracle.TRUTH)
    got = hostsim.trace(blob, "closest", o, d)
    clean = ref["flags"] == 0
    assert clean.mean() > 0.98
    for k in ("hit", "front", "tri"):
        assert np.array_equal(got[k][clean], ref[k][clean]), k
    both = clean & (ref["hit"] == 1)
    assert np.abs(got["loc"][both] - ref["loc"][both]).max() < 1e-5


def test_closest_hit_tie_break_is_by_primitive_index():
    """Two coincident triangles: the smaller face index wins regardless of BVH order."""
    tri = np.array([[0.5, -0.5, 0], [0, 0.5, 0], [-0.5, -0.5, 0]], np.float32)
    v = np.concatenate([tri, tri + [3, 0, 0], tri, tri + [0, 3, 0], tri + [0, 0, -1]]).astype(np.float32)
    f = np.arange(15, dtype=np.int32).reshape(5, 3)
    blob = hostsim.build_blob(v, f)
    o = np.array([[0, 0, 4]], np.float32); d = np.array([[0, 0, -1]], np.float32)
    assert hostsim.trace(blob, "closest", o, d)["tri"].tolist() == [0]
    assert hostsim.trace(blob, "count", o, d)["count"].tolist() == [3]
    assert hostsim.trace(blob, "closest", o, -d)["hit"].tolist() == [0]


def test_empty_mesh_and_nan_rays():
    blob = hostsim.build_blob(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    assert hostsim.check_blob(blob)[0] == 0
    o = np.array([[0, 0, 3], [np.nan, 0, 3]], np.float32); d = np.array([[0, 0, -1], [0, 0, -1]], np.float32)
    assert hostsim.trace(blob, "any", o, d)["hit"].tolist() == [0, 0]
    v, f = synth.icosphere(1)
    blob = hostsim.build_blob(v, f)
    d2 = np.array([[0, 0, 0], [0, 0, -1]], np.float32)
    assert hostsim.trace(blob, "count", o, d2)["count"].tolist() == [0, 0]


@pytest.mark.parametrize("name", ["tri2", "tri9", "ico3", "soup", "hf"])
def test_refit_keeps_the_blob_conservative_and_results_exact(name):
    """Refit path (SURVEY 8f): deform the vertices, re-fit in place, compare with the oracle on the new mesh."""
    v, f = mesh(name)
    blob = hostsim.build_blob(v, f)
    rng = np.random.default_rng(1)
    v2 = (v * np.array([1.3, 0.8, 1.1], np.float32) + rng.normal(0, 0.02, size=v.shape).astype(np.float32) + np.float32(0.1)).astype(np.float32)
    blob2 = hostsim.refit_blob(blob, v2, f)
    code, info = hostsim.check_blob(blob2)
    assert code == 0, f"hs_check_blob after refit -> {code}"
    o, d = synth.random_rays(3000, seed=5, box=True)
    o, d = (o * 1.6).numpy(), d.numpy()
    ref = oracle.query(oracle.OracleMesh(v2, f, use_bvh=False), o, d, oracle.MIRROR)
    got = hostsim.trace(blob2, "closest", o, d)
    for k in ("hit", "front", "tri"):
        assert np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["loc"].view(np.uint32), ref["loc"].view(np.uint32))
    assert np.array_equal(hostsim.trace(blob2, "count", o, d)["count"], ref["count"])
    # refit with the original vertices reproduces the original boxes' answers
    blob3 = hostsim.refit_blob(blob2, v, f)
    assert hostsim.check_blob(blob3)[0] == 0
    ref0 = oracle.query(oracle.OracleMesh(v, f, use_bvh=False), o, d, oracle.MIRROR)
    assert np.array_equal(hostsim.trace(blob3, "closest", o, d)["tri"], ref0["tri"])


@pytest.mark.parametrize("scale,offset", [(1e6, 0.0), (1e-6, 0.0), (1.0, 1e4), (1e-3, -5e2), (1e4, 3e7)])
def test_extreme_scales_and_offsets_stay_conservative(scale, offset):
    """Quantised boxes and the padded slab test must stay conservative far from the unit cube: huge / tiny meshes and
    meshes far from the origin (few mantissa bits left for the geometry).  Bit-exact against the brute-force mirror."""
    v, f = synth.icosphere(3)
    v = (v.astype(np.float64) * scale + offset).astype(np.float32)
    blob = hostsim.build_blob(v, f)
    assert hostsim.check_blob(blob)[0] == 0
    o, d = synth.random_rays(3000, seed=11, box=True)
    o = ((o.numpy().astype(np.float64) * 2.0) * scale + offset).astype(np.float32)
    d = d.numpy()
    ref = oracle.query(oracle.OracleMesh(v, f, use_bvh=False), o, d, oracle.MIRROR)
    got = hostsim.trace(blob, "closest", o, d)
    for k in ("hit", "front", "tri"):
        assert np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["loc"].view(np.uint32), ref["loc"].view(np.uint32))
    assert np.array_equal(hostsim.trace(blob, "count", o, d)["count"], ref["count"])


def _grid_and_lattice_rays(n=16, tilt=0.0):
    """Flat n x n grid in z = 0 over [-1,1]^2 and rays aimed exactly at its vertices, edge midpoints (axis-aligned and
    diagonal edges) and cell centres — the classic crack test for a ray/triangle routine."""
    v, f = synth.heightfield(n, n, amplitude=0.0)
    xs = np.linspace(-1, 1, 2 * n + 1, dtype=np.float64)[1:-1]             # half-cell lattice, interior only
    gx, gy = np.meshgrid(xs, xs, indexing="xy")
    targets = np.stack([gx.ravel(), gy.ravel(), np.zeros(gx.size)], axis=1)
    origins = targets + np.array([tilt, -0.5 * tilt, 1.0]) * 2.0
    d = (targets - origins)
    return v, f, origins.astype(np.float32), d.astype(np.float32)


@pytest.mark.parametrize("tilt", [0.0, 0.25, 1.0])
def test_watertight_no_ray_leaks_through_shared_edges_or_vertices(tilt):
    v, f, o, d = _grid_and_lattice_rays(16, tilt)
    blob = hostsim.build_blob(v, f)
    got = hostsim.trace(blob, "closest", o, d)
    assert got["hit"].all(), f"{int((got['hit'] == 0).sum())} rays leaked through the mesh"
    assert np.abs(got["loc"][:, 2]).max() < 1e-6
    ref = oracle.query(oracle.OracleMesh(v, f, use_bvh=False), o, d, oracle.MIRROR)
    for k in ("hit", "front", "tri"):
        assert np.array_equal(got[k], ref[k]), k
    cnt = hostsim.trace(blob, "count", o, d)["count"]
    assert np.array_equal(cnt, ref["count"]) and cnt.min() >= 1
    # the binary64 truth also reports a hit everywhere (it may count shared edges differently: those rays are flagged)
    tru = oracle.query(oracle.OracleMesh(v, f, use_bvh=False), o, d, oracle.TRUTH)
    assert tru["hit"].all()
    clean = tru["flags"] == 0
    assert np.array_equal(cnt[clean], tru["count"][clean])


@pytest.mark.parametrize("name", ["ico3", "soup", "hf", "tri9"])
def test_results_do_not_depend_on_the_bvh_topology(name):
    """The same collapse / quantisation / traversal code over a DIFFERENT binary topology (top-down binned SAH instead
    of Morton + Karras, hs_build_sah) must give a valid conservative blob and bit-identical answers: closest hits are
    tie-broken by primitive index, counts are exhaustive - nothing may depend on the tree."""
    v, f = mesh(name)
    a, b = hostsim.build_blob(v, f), hostsim.build_blob_sah(v, f)
    assert hostsim.check_blob(a)[0] == 0 and hostsim.check_blob(b)[0] == 0
    assert sorted(hostsim.blob_prims(b, len(f)).tolist()) == list(range(len(f)))
    rng = np.random.default_rng(5)
    o = rng.uniform(-1.5, 1.5, size=(4000, 3)).astype(np.float32)
    d = rng.normal(size=(4000, 3)).astype(np.float32)
    ra, rb = hostsim.trace(a, "closest", o, d), hostsim.trace(b, "closest", o, d)
    for k in ("hit", "front", "tri"):
        assert np.array_equal(ra[k], rb[k]), k
    assert np.array_equal(ra["loc"].view(np.uint32), rb["loc"].view(np.uint32))
    assert np.array_equal(ra["uv"].view(np.uint32), rb["uv"].view(np.uint32))
    assert np.array_equal(hostsim.trace(a, "count", o, d)["count"], hostsim.trace(b, "count", o, d)["count"])
    assert np.array_equal(hostsim.trace(a, "any", o, d)["hit"], hostsim.trace(b, "any", o, d)["hit"])


@pytest.mark.parametrize("name", ["ico3", "cube", "flat", "hf", "soup", "far"])
def test_root_frame_test_never_rejects_a_ray_the_root_node_test_enters(name):
    """The pooled kernels drop a ray at pool fill when it misses the box around the root's child slots (rt_core.cuh
    frame_missed).  That is only sound if such a ray fails EVERY slot of the root in node_test - checked here with the
    very code the device runs (hostsim hs_frame_check), on random rays and on rays that graze the frame: along its faces,
    through its edges and corners, starting on it, one ulp either side.  Also: the 1/d of the fill is the set-up's 1/d."""
    g = np.random.default_rng(5)
    if name == "ico3":
        v, f = synth.icosphere(3)
    elif name == "cube":
        v = np.array([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]], np.float32)
        f = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5], [0, 4, 7], [0, 7, 3]], np.int32)
    elif name == "flat":
        v, f = synth.heightfield(8, 8, amplitude=0.0)
    elif name == "hf":
        v, f = synth.heightfield(64, 32)
    elif name == "soup":
        v, f = synth.triangle_soup(5000, sigma=0.05, seed=3)
    else:
        v, f = synth.icosphere(2)
        v = (v.astype(np.float64) * 3.0 + np.array([1000.25, -2000.5, 3000.125])).astype(np.float32)
    blob = hostsim.build_blob(v, f)
    lo, hi = v.min(0).astype(np.float64), v.max(0).astype(np.float64)
    n = 60_000
    ext = hi - lo + 1e-3
    grid = np.stack([lo, (lo + hi) / 2, hi, lo - ext * 0.5, hi + ext * 0.5])
    o = grid[g.integers(0, 5, (n, 3)), np.arange(3)].astype(np.float32)
    kind = g.integers(0, 4, n)
    axes = np.eye(3)[g.integers(0, 3, n)] * g.choice([-1.0, 1.0], (n, 1))
    diag = g.choice([-1.0, 0.0, 1.0], (n, 3)); diag[(diag == 0).all(1)] = [1, 0, 0]
    corner = grid[g.integers(0, 3, (n, 3)), np.arange(3)] - o; corner[(corner == 0).all(1)] = [0, 0, 1]
    rnd = g.normal(size=(n, 3))
    d = np.where((kind == 0)[:, None], axes, np.where((kind == 1)[:, None], diag, np.where((kind == 2)[:, None], corner, rnd))).astype(np.float32)
    jit = g.integers(0, 3, n)
    o = np.where((jit == 1)[:, None], np.nextafter(o, np.float32(np.inf)), np.where((jit == 2)[:, None], np.nextafter(o, np.float32(-np.inf)), o)).astype(np.float32)
    rejected, unsound, root_rejects = hostsim.frame_check(blob, o, d)
    assert unsound == 0
    assert rejected <= root_rejects
    assert rejected > n // 50                                  # the test does reject a good part of these rays
    # plain random rays as well
    ro, rd = synth.random_rays(20_000, seed=8, box=True)
    ro = (ro.numpy().astype(np.float64) * (hi - lo).max() * 1.5 + (lo + hi) / 2).astype(np.float32)
    r2, u2, _ = hostsim.frame_check(blob, ro, rd.numpy())
    assert u2 == 0


@pytest.mark.parametrize("h,w,w_log2", [(4, 8, 3), (360, 640, 3), (2160, 3840, 3), (8, 4, 2), (40, 36, 2), (2, 16, 4), (64, 96, 3)])
def test_tile_work_order_is_a_bijection_made_of_tiles(h, w, w_log2):
    """rt_core.cuh tile_map (the work order of coherent image batches): every pixel exactly once, and 32 consecutive
    work items cover one tile of 2^w_log2 x (32 >> w_log2) pixels."""
    m = hostsim.tile_map(h, w, w_log2).astype(np.int64)
    assert np.array_equal(np.sort(m), np.arange(h * w))
    tw, th = 1 << w_log2, 32 >> w_log2
    y, x = m // w, m % w
    for t in sorted({0, min(1, len(m) // 32 - 1), len(m) // 32 - 1}):
        ys, xs = y[32 * t:32 * t + 32], x[32 * t:32 * t + 32]
        assert ys.max() - ys.min() == th - 1 and xs.max() - xs.min() == tw - 1
        assert ys.min() % th == 0 and xs.min() % tw == 0
