"""GPU builder and refit against the host simulation, node for node.

rt_bvh_build (k_scene_bounds, k_morton, the onesweep sort, k_karras, k_refit, k_collapse, k_fill_tris,
k_place_parents, k_finalize) is compared with hs_build - the same pipeline one element at a time - after both blobs
are renumbered canonically (hs_canonical: k_collapse's bump allocators number nodes and records in launch order).
The sizes sit on every boundary of the GPU code: the refit tile (1024 leaves), the sort tile (4096 keys) and the four
key-width regimes of morton_axis_bits (10, 13, 16 and 21 bits per axis; 4, 5, 6 and 8 sort passes).  rt_bvh_refit is
compared with hs_refit byte for byte on the same input blob, and rt_sort_pairs_u64 with numpy's stable argsort.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import hostsim  # noqa: E402
from builder_cases import DISTRIBUTIONS, mesh  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402

pytestmark = pytest.mark.gpu

BIG = {"hf_4097x4096": 2 * 4097 * 4096}


def gpu_build(v, f, dev) -> np.ndarray:
    """rt_bvh_build called directly (AccelStructure.build refuses out-of-range faces); the blob starts as 0xa5 bytes, so
    any byte of the used prefix the builder leaves undefined shows up in the comparison.  Returns the whole blob."""
    lib = hops.get_module()
    vt = torch.from_numpy(np.ascontiguousarray(v)).to(dev)
    ft = torch.from_numpy(np.ascontiguousarray(f)).to(dev)
    ws_b, blob_b = C.c_size_t(), C.c_size_t()
    hops._check(lib.rt_bvh_sizes(len(v), len(f), C.byref(ws_b), C.byref(blob_b)), "rt_bvh_sizes")
    ws = torch.empty(max(ws_b.value, 256), dtype=torch.uint8, device=dev)
    blob = torch.full((blob_b.value,), 0xA5, dtype=torch.uint8, device=dev)
    hops._check(lib.rt_bvh_build(hops._ptr(vt), len(v), hops._ptr(ft), len(f), hops._ptr(ws), ws.numel(), hops._ptr(blob),
                                 blob.numel(), hops._stream(dev)), "rt_bvh_build")
    out = blob.cpu().numpy()
    del ws, blob, vt, ft
    return out


def used_of(blob) -> int:
    return int(blob[40:48].view(np.uint64)[0])


def first_difference(a, b, blob) -> str:
    d = np.flatnonzero(a != b)
    if len(d) == 0:
        return "equal"
    o = int(d[0])
    h = hops.parse_header(blob[:256].tobytes())
    if o < 256:
        where = "header"
    elif o < h["nodes_offset"]:
        where = f"record {(o - 256) // 48} byte {(o - 256) % 48}"
    elif o < h["parents_offset"]:
        where = f"node {(o - h['nodes_offset']) // 80} byte {(o - h['nodes_offset']) % 80}"
    else:
        where = f"parent link {(o - h['parents_offset']) // 4}"
    return f"{len(d)} bytes differ, first at offset {o} ({where})"


def assert_same_prefix(got, want, what):
    ug, uw = used_of(got), used_of(want)
    assert ug == uw, f"{what}: used_bytes {ug} != {uw}"
    a, b = got[:ug], want[:uw]
    assert np.array_equal(a, b), f"{what}: {first_difference(a, b, want)}"


def check(blob, v, f, what):
    code, info = hostsim.check_blob(blob, v, f)
    assert code == 0, f"{what}: hs_check_blob -> {code}"
    return info


# ------------------------------------------------------------------ builds, GPU against host
SMALL = [9, 1025, 5000]
BOUNDARIES = [1, 2, 3, 8, 9, 1023, 1024, 1025, 2049, 4095, 4096, 4097, 8193, 16384, 16385]
CASES = ([(d, n) for d in sorted(DISTRIBUTIONS) for n in SMALL]
         + [(d, n) for n in BOUNDARIES for d in ("soup", "identical") if n not in SMALL or d not in ("soup", "identical")]
         + [("soup", 1 << 24), ("soup", (1 << 24) + 1), ("identical", (1 << 24) + 1),
            ("hf_4097x4096", BIG["hf_4097x4096"]), ("identical", BIG["hf_4097x4096"])])
CASES = sorted(set(CASES), key=lambda c: (c[1], c[0]))

_cache: dict = {}


def built(dist, n, dev):
    """(vertices, faces, GPU blob) of one case, kept for the refit tests of the two largest regimes"""
    key = (dist, n)
    if key in _cache:
        return _cache[key]
    v, f = mesh(dist, n)
    g = gpu_build(v, f, dev)
    if key in (("soup", (1 << 24) + 1), ("hf_4097x4096", BIG["hf_4097x4096"])):
        _cache[key] = (v, f, g)
    return v, f, g


@pytest.mark.parametrize("dist,n", CASES, ids=[f"{d}-{n}" for d, n in CASES])
def test_gpu_build_equals_host_build(cuda_device, dist, n):
    v, f, g = built(dist, n, cuda_device)
    info = check(g, v, f, "GPU blob")
    assert info["tris"] == n
    h = hostsim.build_blob(v, f)
    check(h, v, f, "host blob")
    hdr_g, hdr_h = hops.parse_header(g[:256].tobytes()), hops.parse_header(h[:256].tobytes())
    for k in ("n_tris", "n_nodes", "depth", "n_nodes_cap", "tris_offset", "nodes_offset", "parents_offset", "used_bytes",
              "bad_index_faces", "node_overflow"):
        assert hdr_g[k] == hdr_h[k], f"header {k}: GPU {hdr_g[k]} host {hdr_h[k]}"
    assert g[48:72].tobytes() == h[48:72].tobytes(), f"header aabb: GPU {hdr_g['aabb_lo']}{hdr_g['aabb_hi']} " \
                                                     f"host {hdr_h['aabb_lo']}{hdr_h['aabb_hi']}"
    if dist == "bad_index":
        assert hdr_g["bad_index_faces"] == int(((f < 0) | (f >= len(v))).any(1).sum()) > 0
    cg, ch = hostsim.canonical(g), hostsim.canonical(h)
    del h
    assert_same_prefix(cg, ch, f"canonical GPU vs host ({dist}, {n})")
    del ch
    # a second GPU build of the same mesh: the same blob up to numbering
    g2 = gpu_build(v, f, cuda_device)
    assert_same_prefix(hostsim.canonical(g2), cg, f"two GPU builds ({dist}, {n})")


# ------------------------------------------------------------------ refit, GPU against hs_refit
def deformations(v):
    rng = np.random.default_rng(len(v))
    finite = np.isfinite(v)
    yield "jitter", (v + rng.normal(0, 1e-3, v.shape).astype(np.float32) * finite).astype(np.float32)
    yield "anisotropic", (v * np.array([3.0, 0.25, 1.5], np.float32)).astype(np.float32)
    yield "one_point", np.broadcast_to(np.array([0.25, -0.5, 0.125], np.float32), v.shape).copy()
    nan = v.copy()
    nan[rng.random(len(v)) < 0.03] = np.nan
    yield "some_nan", nan
    yield "offset_3e7", (v.astype(np.float64) + 3e7).astype(np.float32)


def gpu_refit(blob_np, v, f, dev, prefix_only=False) -> np.ndarray:
    """rt_bvh_refit on a copy of blob_np (the whole blob, or an adopted used prefix as save/load and broadcast carry)"""
    data = blob_np[:used_of(blob_np)] if prefix_only else blob_np
    acc = hops.AccelStructure().adopt(torch.from_numpy(np.ascontiguousarray(data)).to(dev))
    acc.refit(torch.from_numpy(np.ascontiguousarray(v)).to(dev), torch.from_numpy(np.ascontiguousarray(f)).to(dev))
    out = acc.blob.cpu().numpy()
    acc.free()
    return out


def run_refits(blob, v, f, dev, which, prefix_only=False):
    cur = blob
    for name, v2 in deformations(v):
        if name not in which:
            continue
        got = gpu_refit(cur, v2, f, dev, prefix_only)
        want = hostsim.refit_blob(cur[:len(got)], v2, f)
        assert_same_prefix(got, want, f"refit {name}: GPU vs hs_refit")
        check(got, v2, f, f"refit {name}")
        cur = got
    back = gpu_refit(cur, v, f, dev, prefix_only)
    assert_same_prefix(back, blob, "refit back to the original vertices vs the build")


def test_refit_16_bit_regime(cuda_device):
    v, f, g = built("soup", (1 << 24) + 1, cuda_device)
    run_refits(g, v, f, cuda_device, ("anisotropic", "one_point", "offset_3e7"))


def test_refit_21_bit_regime(cuda_device):
    v, f, g = built("hf_4097x4096", BIG["hf_4097x4096"], cuda_device)
    run_refits(g, v, f, cuda_device, ("jitter", "some_nan"))
    _cache.clear()


@pytest.mark.parametrize("dist,n", [("soup", 5000), ("heightfield", 4097), ("nan_some", 1025)])
def test_refit_of_an_adopted_used_prefix(cuda_device, dist, n):
    v, f = mesh(dist, n)
    g = gpu_build(v, f, cuda_device)
    run_refits(g, v, f, cuda_device, ("jitter", "anisotropic", "one_point", "some_nan", "offset_3e7"), prefix_only=True)


# ------------------------------------------------------------------ sort
@pytest.mark.parametrize("kind,n", [("bit63", 100_003), ("equal", 300_000), ("random", 4095), ("random", 4096),
                                    ("random", 4097), ("random", (1 << 25) + 3)])
def test_sort_matches_numpy_stable_argsort(cuda_device, kind, n):
    rng = np.random.default_rng(n)
    if kind == "bit63":        # half the keys have bit 63 set: the top digit must sort as unsigned
        keys = rng.integers(0, 1 << 62, size=n, dtype=np.uint64) | (rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63))
        keys[:5] = [0xFFFFFFFFFFFFFFFF, 0x8000000000000000, 0x7FFFFFFFFFFFFFFF, 0, 0x8000000000000000]
    elif kind == "equal":      # one key over ~73 sort tiles: only stability orders the values
        keys = np.full(n, 0x8000000000000001, np.uint64)
    else:
        keys = rng.integers(0, np.iinfo(np.uint64).max, size=n, dtype=np.uint64, endpoint=True)
    vals = rng.permutation(n).astype(np.int32)
    k = torch.from_numpy(keys.view(np.int64)).to(cuda_device)
    vv = torch.from_numpy(vals).to(cuda_device)
    hops.sort_pairs_u64(k, vv)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k.cpu().numpy().view(np.uint64), keys[order]), "sorted keys"
    assert np.array_equal(vv.cpu().numpy(), vals[order]), "values (stability)"


# ------------------------------------------------------------------ layout: a host-built blob is a product blob
@pytest.mark.parametrize("dist,n", [("icosphere", 5120), ("soup", 20_000), ("nan_some", 4097)])
def test_host_built_blob_adopted_on_the_gpu_answers_like_the_gpu_blob(cuda_device, dist, n):
    v, f = mesh(dist, n)
    host = hops.AccelStructure().adopt(torch.from_numpy(hostsim.build_blob(v, f)).to(cuda_device))
    prefix = hops.AccelStructure().adopt(host.used().clone())
    gpu = hops.AccelStructure().build(torch.from_numpy(v).to(cuda_device), torch.from_numpy(f).to(cuda_device))
    o, d = synth.random_rays(200_000, seed=n, device=cuda_device, box=True)
    o = o * 1.5
    p = torch.rand((100_000, 3), generator=torch.Generator(device=cuda_device).manual_seed(n), device=cuda_device) * 3 - 1.5
    ref = (hops.intersects_closest(gpu, o, d), hops.intersects_count(gpu, o, d), hops.closest_point(gpu, p))
    for acc, what in ((host, "host blob"), (prefix, "used prefix of the host blob")):
        got = (hops.intersects_closest(acc, o, d), hops.intersects_count(acc, o, d), hops.closest_point(acc, p))
        for qa, qb in zip(got, ref):
            for x, y in zip(qa if isinstance(qa, tuple) else (qa,), qb if isinstance(qb, tuple) else (qb,)):
                assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes(), what
