"""Scenes where one ray crosses many triangles, their ray sets, and a complete-hit-list reference; shared by the CPU
tests (test_deep_overlap_logic.py) and the GPU tests of the trace kernels (test_gpu_deep_overlap.py).

Deep overlap is where the warp-cooperative kernel's pair list (rt_trace_coop.cuh) fills, overflows and flushes with
triangles still waiting, where all-hits records go past max_hits, and where ties in t decide closest and first.  Every
scene is deterministic and small enough for the oracle's brute-force mirror:

  dup(K)       K exact copies of one triangle, face order shuffled: every hit ties in t (the smallest index wins)
  coplanar(K)  K different overlapping triangles in one plane: t ties across triangles whose barycentrics differ
  stack(L)     L parallel quads (2L triangles), slightly larger layer by layer
  shells(K)    K concentric closed icospheres: at most 2K hits per ray; contains parity known analytically
  book(K)      K triangles fanned around one shared edge, rays aimed at the spine (edges, grazing hits)
  mixed        an icosphere with a dup(512) cluster inside: lanes with 1-2 hits next to lanes with hundreds

scene(name) -> (vertices float32 [m, 3], faces int32 [n, 3]);  rays(name, kind) -> (origins, directions) as float32
numpy arrays: kind "pooled" and "tinyN" are [n, 3] with one origin per ray, "broadcast" is [n, 3] and "image" [H, W, 3]
(H % 4 == 0, W % 8 == 0), both with one origin for all rays (broadcast_origin() says which)."""
from __future__ import annotations

import numpy as np

from oracle import oracle
from triro import synth

ONE_TRI = np.array([[0.5, -0.5, 0.25], [0.0, 0.5, 0.25], [-0.5, -0.5, 0.25]], np.float32)
SHELL_SUBDIV = 2
BLOCK = oracle.MAX_LIST      # faces per oracle call of complete_hits: one block cannot give a ray more hits than its list


def dup(k: int, seed: int = 1, tri=ONE_TRI):
    """k copies of `tri` (each with its own three vertices), faces in shuffled order"""
    v = np.tile(tri, (k, 1)).astype(np.float32)
    f = np.arange(3 * k, dtype=np.int32).reshape(k, 3)
    return v, np.ascontiguousarray(f[np.random.default_rng(seed).permutation(k)])


def coplanar(k: int, seed: int = 2):
    """k random triangles in the plane z = 0.25 around the origin, all overlapping the unit square's middle"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-0.2, 0.2, size=(k, 1, 2))
    p = c + rng.uniform(-1.0, 1.0, size=(k, 3, 2))
    v = np.concatenate([p, np.full((k, 3, 1), 0.25)], axis=2).reshape(-1, 3).astype(np.float32)
    return v, np.arange(3 * k, dtype=np.int32).reshape(k, 3)


def stack(layers: int):
    """layers quads at z = -0.01 k, half-size 1 + 0.001 k"""
    q = []
    for k in range(layers):
        h, z = 1.0 + 0.001 * k, -0.01 * k
        q += [[-h, -h, z], [h, -h, z], [h, h, z], [-h, h, z]]
    v = np.array(q, np.float32)
    b = 4 * np.arange(layers, dtype=np.int32)[:, None]
    f = np.concatenate([b + np.array([0, 1, 2], np.int32), b + np.array([0, 2, 3], np.int32)], axis=1).reshape(-1, 3)
    return v, np.ascontiguousarray(f)


def shell_radii(k: int) -> np.ndarray:
    return (0.25 + 0.75 * np.arange(1, k + 1) / k).astype(np.float64)


def shells(k: int):
    """k concentric icospheres (subdivision SHELL_SUBDIV) of radii shell_radii(k), each closed and outward-facing"""
    v1, f1 = synth.icosphere(SHELL_SUBDIV)
    vs, fs = [], []
    for i, r in enumerate(shell_radii(k)):
        vs.append((v1.astype(np.float64) * r).astype(np.float32))
        fs.append(f1 + i * len(v1))
    return np.concatenate(vs), np.concatenate(fs).astype(np.int32)


def shell_inradius_factor() -> float:
    """smallest distance from the centre to a face plane of the unit icosphere: a point closer than r * this to the
    centre is inside the shell of radius r, a point farther than r is outside"""
    v, f = synth.icosphere(SHELL_SUBDIV)
    a, b, c = (v[f[:, i]].astype(np.float64) for i in range(3))
    n = np.cross(b - a, c - a)
    return float((np.abs((n * a).sum(1)) / np.linalg.norm(n, axis=1)).min())


def shell_parity(points, k: int, margin: float = 1e-3):
    """(number of shells that enclose each point is odd, the point is well away from every shell)"""
    rho = np.linalg.norm(np.asarray(points, np.float64), axis=1)
    radii = shell_radii(k)
    inr = radii * shell_inradius_factor()
    enclosing = (rho[:, None] < inr[None, :] * (1 - margin)).sum(1)
    clear = ~((rho[:, None] >= inr[None, :] * (1 - margin)) & (rho[:, None] <= radii[None, :] * (1 + margin))).any(1)
    return enclosing % 2 == 1, clear


def book(k: int):
    """k triangles sharing the edge (0,0,-1)-(0,0,1), third vertices on the unit circle of z = 0"""
    th = np.linspace(0.0, 2.0 * np.pi, k, endpoint=False)
    v = [[0.0, 0.0, -1.0], [0.0, 0.0, 1.0]] + [[np.cos(a), np.sin(a), 0.0] for a in th]
    f = np.stack([np.zeros(k), np.ones(k), 2 + np.arange(k)], axis=1)
    return np.array(v, np.float32), f.astype(np.int32)


def mixed():
    """icosphere(4) of radius 1 around a dup(512) cluster of a small triangle at the centre"""
    vs, fs = synth.icosphere(4)
    vd, fd = dup(512, seed=3, tri=(ONE_TRI * np.float32(0.4)).astype(np.float32))
    return np.concatenate([vs, vd]), np.concatenate([fs, fd + len(vs)]).astype(np.int32)


SCENES = {
    "dup600": lambda: dup(600),
    "coplanar200": lambda: coplanar(200),
    "stack300": lambda: stack(300),
    "shells32": lambda: shells(32),
    "book96": lambda: book(96),
    "mixed": mixed,
}

RAY_SETS = ("pooled", "broadcast", "image", "tiny1", "tiny31", "tiny33")
N_POOLED = 4096
IMAGE_HW = (32, 64)
_cache: dict = {}


def scene(name: str):
    if name not in _cache:
        v, f = SCENES[name]()
        _cache[name] = (np.ascontiguousarray(v, np.float32), np.ascontiguousarray(f, np.int32))
    return _cache[name]


def _targets(name: str, rng, n: int) -> np.ndarray:
    """points the rays of a scene aim at: where the overlap is deepest, with some spill-over so that rays also miss"""
    if name in ("dup600", "coplanar200"):
        return np.stack([rng.uniform(-0.7, 0.7, n), rng.uniform(-0.7, 0.7, n), np.full(n, 0.25)], 1)
    if name == "stack300":
        return np.stack([rng.uniform(-1.2, 1.2, n), rng.uniform(-1.2, 1.2, n), np.full(n, -3.5)], 1)
    if name == "shells32":
        return rng.uniform(-0.3, 0.3, (n, 3))
    if name == "book96":
        return np.stack([rng.normal(0, 1e-3, n) * (rng.random(n) < 0.5), np.zeros(n), rng.uniform(-1.1, 1.1, n)], 1)
    assert name == "mixed"
    t = rng.uniform(-0.9, 0.9, (n, 3))
    near = rng.random(n) < 0.5                      # half the rays go through the cluster
    t[near] = np.stack([rng.uniform(-0.15, 0.15, near.sum()), rng.uniform(-0.15, 0.15, near.sum()),
                        np.full(near.sum(), 0.1)], 1)
    return t


def _origins(name: str, rng, n: int) -> np.ndarray:
    if name in ("dup600", "coplanar200"):            # above and below the plane
        s = np.where(rng.random(n) < 0.5, 1.0, -1.0)
        return np.stack([rng.uniform(-1.5, 1.5, n), rng.uniform(-1.5, 1.5, n), 0.25 + s * rng.uniform(0.5, 2.0, n)], 1)
    if name == "stack300":
        return np.stack([rng.uniform(-1.2, 1.2, n), rng.uniform(-1.2, 1.2, n), rng.uniform(0.5, 3.0, n)], 1)
    if name == "shells32":                          # inside, between and outside the shells
        d = rng.normal(size=(n, 3))
        return d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(0.0, 1.6, (n, 1))
    if name == "book96":
        a = rng.uniform(0, 2 * np.pi, n)
        return np.stack([2.0 * np.cos(a), 2.0 * np.sin(a), rng.uniform(-0.5, 0.5, n)], 1)
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1, keepdims=True) * 2.5


def broadcast_origin(name: str) -> np.ndarray:
    return {"dup600": [0.05, 0.02, 2.0], "coplanar200": [0.05, -0.03, 2.0], "stack300": [0.02, 0.01, 3.0],
            "shells32": [0.011, -0.007, 0.013], "book96": [1.5, 0.5, 0.1], "mixed": [0.0, 0.0, 2.5]}[name]


def rays(name: str, kind: str, seed: int = 0):
    """(origins, directions) float32 numpy arrays; see the module docstring"""
    rng = np.random.default_rng([seed, list(SCENES).index(name), RAY_SETS.index(kind)])
    if kind in ("broadcast", "image"):
        n = N_POOLED if kind == "broadcast" else IMAGE_HW[0] * IMAGE_HW[1]
        o = np.tile(np.array(broadcast_origin(name), np.float64), (n, 1))
    else:
        n = N_POOLED if kind == "pooled" else int(kind[4:])
        o = _origins(name, rng, n)
    d = _targets(name, rng, n) - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o, d = o.astype(np.float32), d.astype(np.float32)
    if kind == "image":
        return o.reshape(*IMAGE_HW, 3), d.reshape(*IMAGE_HW, 3)
    return o, d


def mirror(v, f, o, d, want=("hit", "front", "tri", "loc", "uv", "count"), **kw):
    """the oracle's binary32 mirror over every triangle (brute force)"""
    return oracle.query(oracle.OracleMesh(v, f, use_bvh=False), np.reshape(o, (-1, 3)), np.reshape(d, (-1, 3)),
                        oracle.MIRROR, want=want, brute=True, **kw)


def complete_hits(v, f, o, d):
    """Every hit of every ray, with the mirror's location bits: dict of ray int64[m], tri int32[m], loc float32[m, 3]
    sorted by (ray, tri), and count int32[n] (hits per ray).

    The mirror lists only the list_cap nearest hits of a ray, so the faces are queried in blocks of BLOCK = list_cap
    triangles: each block's list is complete, a hit's location depends only on the ray and its triangle, and the union
    of the blocks (triangle indices shifted back by the block offset) is the exact hit set."""
    o = np.ascontiguousarray(np.reshape(o, (-1, 3)), np.float32)
    d = np.ascontiguousarray(np.reshape(d, (-1, 3)), np.float32)
    n = len(o)
    rays_, tris, locs = [], [], []
    for b in range(0, len(f), BLOCK):
        q = oracle.query(oracle.OracleMesh(v, f[b:b + BLOCK], use_bvh=False), o, d, oracle.MIRROR, list_cap=BLOCK,
                         want=("count",), brute=True)
        assert np.array_equal(q["list_n"], q["count"])
        j = np.arange(BLOCK)[None, :] < q["list_n"][:, None]
        rays_.append(np.nonzero(j)[0].astype(np.int64))
        tris.append(q["list_tri"][j] + np.int32(b))
        locs.append(q["list_loc"][j])
    ray = np.concatenate(rays_) if rays_ else np.zeros(0, np.int64)
    tri = np.concatenate(tris) if tris else np.zeros(0, np.int32)
    loc = np.concatenate(locs) if locs else np.zeros((0, 3), np.float32)
    order = np.lexsort((tri, ray))
    return dict(ray=ray[order], tri=tri[order].astype(np.int32), loc=np.ascontiguousarray(loc[order]),
                count=np.bincount(ray, minlength=n).astype(np.int32))


def hit_keys(ray, tri) -> np.ndarray:
    """one int64 per (ray, triangle) pair, ordered like lexsort((tri, ray))"""
    return np.asarray(ray, np.int64) * (1 << 32) + np.asarray(tri, np.int64)


def check_hits_subset(ch: dict, ray, tri, loc, what=""):
    """every (ray, tri, loc bits) of a result is in the complete hit set, and no ray lists a triangle twice"""
    ray = np.asarray(ray, np.int64); tri = np.asarray(tri, np.int32); loc = np.asarray(loc, np.float32).reshape(-1, 3)
    keys = hit_keys(ray, tri)
    ref = hit_keys(ch["ray"], ch["tri"])
    order = np.argsort(keys, kind="stable")
    sk = keys[order]
    assert not (sk[1:] == sk[:-1]).any(), f"{what}: a ray lists the same triangle twice"
    pos = np.searchsorted(ref, keys)
    found = pos < len(ref)
    found[found] = ref[pos[found]] == keys[found]
    assert found.all(), f"{what}: {int((~found).sum())} hits are not hits of the mirror (first ray {ray[~found][0]}, tri {tri[~found][0]})"
    bad = (ch["loc"][pos].view(np.uint32) != loc.view(np.uint32)).any(1)
    assert not bad.any(), f"{what}: {int(bad.sum())} hit locations differ from the mirror's bits (first ray {ray[bad][0]})"
