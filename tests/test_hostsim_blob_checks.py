"""CPU tier: the host builder (hs_build, the product's pipeline one element at a time) on every mesh distribution of
builder_cases, the blob checker (hs_check_blob) against single corruptions, and the canonical renumbering
(hs_canonical) that lets a GPU blob be compared with a host blob byte for byte."""
from __future__ import annotations

import os
import struct
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "pointquery"))
import hostsim  # noqa: E402
import pointquery as pq  # noqa: E402
from builder_cases import DISTRIBUTIONS, mesh  # noqa: E402
from triro import synth  # noqa: E402

HDR = 256


def header(blob):
    magic, abi, n_tris, n_nodes, depth, cap = struct.unpack_from("<6I", blob, 0)
    tris_off, nodes_off, used = struct.unpack_from("<3Q", blob, 24)
    aabb = struct.unpack_from("<6f", blob, 48)
    bad, overflow = struct.unpack_from("<2I", blob, 72)
    (parents_off,) = struct.unpack_from("<Q", blob, 80)
    return dict(n_tris=n_tris, n_nodes=n_nodes, depth=depth, cap=cap, tris_offset=tris_off, nodes_offset=nodes_off,
                used_bytes=used, aabb=aabb, bad=bad, parents_offset=parents_off)


@pytest.mark.parametrize("n", [1, 2, 9, 1025, 16385])
@pytest.mark.parametrize("dist", sorted(DISTRIBUTIONS))
def test_host_build_passes_the_full_check(dist, n):
    v, f = mesh(dist, n)
    blob = hostsim.build_blob(v, f)
    code, info = hostsim.check_blob(blob, v, f)
    assert code == 0, f"hs_check_blob -> {code}"
    assert info["tris"] == n
    h = header(blob)
    if dist == "bad_index":
        assert h["bad"] == int(((f < 0) | (f >= len(v))).any(1).sum()) > 0
        assert hostsim.check_blob(blob)[0] == 103                  # without the faces a bad index is an error
    else:
        assert h["bad"] == 0
    if dist == "nan_all":
        assert h["aabb"] == (np.inf,) * 3 + (-np.inf,) * 3        # the empty box, not NaN bit patterns


def test_empty_mesh_blob():
    blob = hostsim.build_blob(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))
    assert hostsim.check_blob(blob, np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32))[0] == 0
    h = header(blob)
    assert h["n_nodes"] == 1 and h["aabb"] == (0.0,) * 6
    assert struct.unpack_from("<I", blob, h["parents_offset"])[0] == 0xFFFFFFFF
    assert h["used_bytes"] == h["parents_offset"] + 16


@pytest.mark.parametrize("dist,n", [("soup", 5000), ("heightfield", 4096), ("identical", 1025), ("nan_some", 777),
                                    ("icosphere", 1280)])
def test_canonical_form(dist, n):
    v, f = mesh(dist, n)
    blob = hostsim.build_blob(v, f)
    can = hostsim.canonical(blob)
    assert np.array_equal(hostsim.canonical(can), can), "hs_canonical is not idempotent"
    assert hostsim.check_blob(can, v, f)[0] == 0
    assert np.array_equal(can[:HDR], blob[:HDR])
    # same traversal answers, bit for bit
    o, d = synth.random_rays(3000, seed=n, box=True)
    o, d = (o * 1.5).numpy(), d.numpy()
    for mode in ("closest", "count", "any"):
        a, b = hostsim.trace(blob, mode, o, d), hostsim.trace(can, mode, o, d)
        for k in ("hit", "front", "tri", "count"):
            assert np.array_equal(a[k], b[k]), (mode, k)
        for k in ("loc", "uv"):
            assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), (mode, k)
    p = np.random.default_rng(n).uniform(-1.5, 1.5, (3000, 3)).astype(np.float32)
    a, b = pq.sim_closest_point(blob, p), pq.sim_closest_point(can, p)
    for k in ("closest", "distance", "tri", "uv"):
        assert np.ascontiguousarray(a[k]).tobytes() == np.ascontiguousarray(b[k]).tobytes(), k


def _mutated(blob, fn):
    b = blob.copy()
    fn(b, header(b))
    return b


def _u32(b, off, fn):
    x = struct.unpack_from("<I", b, off)[0]
    struct.pack_into("<I", b, off, fn(x) & 0xFFFFFFFF)


def _f32(b, off, val):
    struct.pack_into("<f", b, off, val)


def _first_inner_node(b, h):
    for w in range(h["n_nodes"]):
        if b[h["nodes_offset"] + 80 * w + 15] != 0:
            return w
    raise AssertionError("no inner node")


def _plane_inward(b, h):
    # node 0, slot holding something: raise its quantised x lower plane by one step (the box no longer contains it)
    nd = h["nodes_offset"]
    imask, trimask = b[nd + 15], struct.unpack_from("<I", b, nd + 24)[0]
    s = next(s for s in range(8) if (imask >> s) & 1 or (trimask >> (3 * s)) & 7)
    qlo = nd + 32 + s
    hi = b[nd + 56 + s]
    assert b[qlo] < hi
    b[qlo] += 1


MUTATIONS = {
    # v0 of record 7 moved onto its v1: still inside every box, but no longer the face's vertex
    "record_vertex": (lambda b, h: b.__setitem__(slice(h["tris_offset"] + 48 * 7, h["tris_offset"] + 48 * 7 + 12),
                                                 b[h["tris_offset"] + 48 * 7 + 16:h["tris_offset"] + 48 * 7 + 28]), 21),
    "prim_id": (lambda b, h: _u32(b, h["tris_offset"] + 48 * 3 + 12, lambda x: (x + 1) % h["n_tris"]), 22),
    "parent_link": (lambda b, h: _u32(b, h["parents_offset"] + 4 * 5, lambda x: x ^ 1), 20),
    "root_parent_link": (lambda b, h: _u32(b, h["parents_offset"], lambda x: 0), 20),
    "plane_inward": (_plane_inward, 10),
    "child_base_plus_one": (lambda b, h: _u32(b, h["nodes_offset"] + 80 * _first_inner_node(b, h) + 16, lambda x: x + 1), None),
    "used_bytes": (lambda b, h: struct.pack_into("<Q", b, 40, h["used_bytes"] - 16), 32),
    "record_pad": (lambda b, h: _u32(b, h["tris_offset"] + 48 * 2 + 28, lambda x: 1), 25),
    "node_reserved": (lambda b, h: _u32(b, h["nodes_offset"] + 80 * 1 + 28, lambda x: 1), 25),
    "header_gap_byte": (lambda b, h: b.__setitem__(250, 1), 25),
    "aabb": (lambda b, h: _f32(b, 48, np.nextafter(np.float32(h["aabb"][0]), np.float32(-np.inf))), 33),
    "n_nodes_cap": (lambda b, h: _u32(b, 20, lambda x: x + 1), 30),
    "parents_offset": (lambda b, h: struct.pack_into("<Q", b, 80, h["parents_offset"] + 256), 31),
    "bad_index_faces": (lambda b, h: _u32(b, 72, lambda x: x + 1), 34),
}


@pytest.mark.parametrize("name", sorted(MUTATIONS))
def test_check_blob_names_each_corruption(name):
    v, f = synth.icosphere(3)
    blob = hostsim.build_blob(v, f)
    assert hostsim.check_blob(blob, v, f)[0] == 0
    fn, code = MUTATIONS[name]
    bad = _mutated(blob, fn)
    got = hostsim.check_blob(bad, v, f)[0]
    if name == "child_base_plus_one":
        # the walk reaches the wrong subtrees: a slot box that does not contain them, a node outside the pool, a node
        # twice or a node never reached
        assert got in (1, 2, 10, 11), got
    else:
        assert got == code, f"{name}: expected {code}, got {got}"


def test_refit_to_the_original_vertices_reproduces_the_build():
    for dist, n in (("soup", 3000), ("heightfield", 2048), ("nan_some", 999), ("identical", 1500)):
        v, f = mesh(dist, n)
        blob = hostsim.build_blob(v, f)
        used = header(blob)["used_bytes"]
        rng = np.random.default_rng(n)
        v2 = (v * np.float32(1.7) + rng.normal(0, 0.05, v.shape).astype(np.float32)).astype(np.float32)
        moved = hostsim.refit_blob(blob, v2, f)
        assert hostsim.check_blob(moved, v2, f)[0] == 0
        back = hostsim.refit_blob(moved, v, f)
        assert np.array_equal(back[:used], blob[:used]), dist
