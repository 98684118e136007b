"""The decoupled look-back scan and the order-preserving scatters of rt_compact.cu against numpy, on crafted masks
(rt_compact_scan / rt_compact_scatter / rt_compact_scatter_at through the C ABI), and the all-hits scatter with 64-bit
ray indices at large bases (hops.intersects_location).

Sizes cross every tile boundary (2048 rays per tile) and reach batches whose look-back has to walk past its first
32-tile window; payloads are random bit patterns, NaNs included, compared bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

import deep_overlap_cases as dc
from triro.backend import ops as hops
from triro.ray.ray_optix import RayMeshIntersector

pytestmark = pytest.mark.gpu

TILE = 2048
SIZES = [1, 7, 8, 9, 2047, 2048, 2049, 32 * TILE - 1, 32 * TILE, 33 * TILE + 1, 65 * TILE + 3, 2 ** 22 + 5, 2 ** 24 + 1]
PATTERNS = ["zeros", "ones", "first", "last", "alternating", "density1e-4", "density0.5", "density0.9999", "bytes2", "bytes255"]


def mask_bytes(pattern: str, n: int, seed: int) -> np.ndarray:
    """uint8 mask; every nonzero byte is a hit"""
    rng = np.random.default_rng([seed, n])
    m = np.zeros(n, np.uint8)
    if pattern == "ones":
        m[:] = 1
    elif pattern == "first":
        m[0] = 1
    elif pattern == "last":
        m[-1] = 1
    elif pattern == "alternating":
        m[1::2] = 1
    elif pattern.startswith("density"):
        m[rng.random(n) < float(pattern[7:])] = 1
    elif pattern == "bytes2":            # 2 and 255 count as hits, mixed with 1
        m[rng.random(n) < 0.5] = 2
        m[rng.random(n) < 0.1] = 1
    elif pattern == "bytes255":
        m[rng.random(n) < 0.7] = 255
    return m


def payload(n: int, dev, seed: int):
    """front u8, tri i32, loc f32[3], uv f32[2] of random bits (NaN patterns included), generated on the device"""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    front = torch.randint(0, 256, (n,), dtype=torch.uint8, device=dev, generator=g)
    tri = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), dtype=torch.int32, device=dev, generator=g)
    loc = torch.randint(-2 ** 31, 2 ** 31 - 1, (n, 3), dtype=torch.int32, device=dev, generator=g)
    uv = torch.randint(-2 ** 31, 2 ** 31 - 1, (n, 2), dtype=torch.int32, device=dev, generator=g)
    loc[::5, 0] = 0x7FC00001          # quiet NaN with a payload
    uv[::7, 1] = -0x00400001          # 0xFFBFFFFF: negative signalling-NaN pattern
    return front, tri, loc.view(torch.float32), uv.view(torch.float32)


def make(v, f, **kw):
    return RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f), **kw)


def ptr(t, byte_offset=0):
    return C.c_void_p(t.data_ptr() + byte_offset)


def scan(lib, hit, dev):
    n = hit.numel()
    ws_b = C.c_size_t()
    assert lib.rt_compact_sizes(n, C.byref(ws_b)) == 0
    ws = torch.empty(max(ws_b.value, 256), dtype=torch.uint8, device=dev)
    total = torch.full((1,), -1, dtype=torch.int64, device=dev)
    assert lib.rt_compact_scan(ptr(hit), n, ptr(ws), ws.numel(), ptr(total), hops._stream(dev)) == 0
    return ws, int(total.item())


@pytest.mark.parametrize("n", SIZES)
def test_scan_and_scatter_equal_numpy_boolean_gathers(cuda_device, n):
    lib = hops.get_module()
    dev = cuda_device
    front, tri, loc, uv = payload(n, dev, seed=n)
    ref_payload = [x.cpu().numpy() for x in (front, tri, loc, uv)]
    for pattern in PATTERNS:
        m = mask_bytes(pattern, n, seed=PATTERNS.index(pattern))
        sel = m != 0
        hit = torch.from_numpy(m).to(dev)
        ws, h = scan(lib, hit, dev)
        assert h == int(sel.sum()), f"{pattern}: total {h} != {int(sel.sum())}"
        outs = (torch.empty(h, dtype=torch.uint8, device=dev), torch.empty(h, dtype=torch.int32, device=dev),
                torch.empty(h, dtype=torch.int32, device=dev), torch.empty((h, 3), dtype=torch.float32, device=dev),
                torch.empty((h, 2), dtype=torch.float32, device=dev))
        if h > 0:
            assert lib.rt_compact_scatter(ptr(hit), n, ptr(ws), ptr(front), ptr(tri), ptr(loc), ptr(uv), ptr(outs[0]),
                                          ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), ptr(outs[4]), hops._stream(dev)) == 0
        got = [x.cpu().numpy() for x in outs]
        assert np.array_equal(got[1], np.nonzero(sel)[0].astype(np.int32)), f"{pattern}: ray indices"
        for name, g_, r_ in zip(("front", "tri", "loc", "uv"), (got[0], got[2], got[3], got[4]), ref_payload):
            a = g_.view(np.uint32) if g_.dtype == np.float32 else g_
            b = r_[sel].view(np.uint32) if r_.dtype == np.float32 else r_[sel]
            assert np.array_equal(a, b), f"{pattern}: {name} differs from the boolean gather"


@pytest.mark.parametrize("ray_idx_bytes,ray_base", [(4, 0), (8, 0), (8, 3 * 2 ** 31 + 5)])
@pytest.mark.parametrize("n", [9, 2049, 65 * TILE + 3])
def test_compact_scatter_at_writes_only_its_rows(cuda_device, n, ray_idx_bytes, ray_base):
    """rt_compact_scatter_at at a row offset inside larger tensors filled with a sentinel: rows [row0, row0 + h) get the
    packed hits with ray index ray_base + i (4 or 8 bytes), every other row keeps the sentinel"""
    lib = hops.get_module()
    dev = cuda_device
    front, tri, loc, uv = payload(n, dev, seed=7 + n)
    m = mask_bytes("density0.5", n, seed=3)
    m[-1] = 255
    sel = m != 0
    hit = torch.from_numpy(m).to(dev)
    ws, h = scan(lib, hit, dev)
    assert h == int(sel.sum())
    row0, guard = 37, 53
    rows = row0 + h + guard
    idt = torch.int64 if ray_idx_bytes == 8 else torch.int32
    out_front = torch.full((rows,), 0xA5, dtype=torch.uint8, device=dev)
    out_ray = torch.full((rows,), -3, dtype=idt, device=dev)
    out_tri = torch.full((rows,), -5, dtype=torch.int32, device=dev)
    out_loc = torch.full((rows, 3), -7.5, dtype=torch.float32, device=dev)
    out_uv = torch.full((rows, 2), -9.25, dtype=torch.float32, device=dev)
    assert lib.rt_compact_scatter_at(ptr(hit), n, ptr(ws), ptr(front), ptr(tri), ptr(loc), ptr(uv), ray_base, ray_idx_bytes,
                                     ptr(out_front, row0), ptr(out_ray, row0 * ray_idx_bytes), ptr(out_tri, row0 * 4),
                                     ptr(out_loc, row0 * 12), ptr(out_uv, row0 * 8), hops._stream(dev)) == 0
    idx = np.nonzero(sel)[0]
    ref = dict(front=front.cpu().numpy()[sel], ray=idx.astype(np.int64) + ray_base, tri=tri.cpu().numpy()[sel],
               loc=loc.cpu().numpy()[sel].view(np.uint32), uv=uv.cpu().numpy()[sel].view(np.uint32))
    got = dict(front=out_front.cpu().numpy(), ray=out_ray.cpu().numpy().astype(np.int64), tri=out_tri.cpu().numpy(),
               loc=out_loc.cpu().numpy().view(np.uint32), uv=out_uv.cpu().numpy().view(np.uint32))
    sentinel = dict(front=0xA5, ray=-3, tri=-5, loc=np.float32(-7.5).view(np.uint32), uv=np.float32(-9.25).view(np.uint32))
    for k in got:
        assert np.array_equal(got[k][row0:row0 + h], ref[k]), f"{k}: packed rows"
        assert (got[k][:row0] == sentinel[k]).all() and (got[k][row0 + h:] == sentinel[k]).all(), f"{k}: rows outside"


@pytest.mark.parametrize("max_hits", [8, 13])
def test_all_hits_with_int64_ray_indices_at_a_large_base(cuda_device, max_hits):
    """intersects_location with ray_idx_base = 2^33 + 7 and int64 indices, over several staging windows, equals the
    int32 result (one launch) plus the base: k_allhits_scatter<int64_t> keeps all 64 bits"""
    v, f = dc.scene("stack300")
    r = make(v, f)
    o1, d1 = dc.rays("stack300", "pooled", seed=3)
    o2, d2 = dc.rays("mixed", "pooled", seed=3)
    o = torch.from_numpy(np.concatenate([o1, o2 * np.float32(0.3)])).to(cuda_device)
    d = torch.from_numpy(np.concatenate([d1, d2])).to(cuda_device)
    base = 2 ** 33 + 7
    l32, r32, t32 = hops.intersects_location(r.as_wrapper, o, d, max_hits)
    assert r32.dtype == torch.int32 and r32.numel() > 10_000
    l64, r64, t64 = hops.intersects_location(r.as_wrapper, o, d, max_hits, ray_idx_base=base, ray_idx_dtype=torch.int64,
                                             staging_bytes=1500 * max_hits * 16)
    assert r64.dtype == torch.int64
    assert torch.equal(r64, r32.long() + base)
    cnt = r.intersects_count(o, d).cpu().numpy()
    few = torch.from_numpy(cnt <= max_hits).to(cuda_device)[r32.long()]
    k32 = np.lexsort((t32[few].cpu().numpy(), r32[few].cpu().numpy()))
    k64 = np.lexsort((t64[few].cpu().numpy(), (r64[few] - base).cpu().numpy()))
    assert np.array_equal(t32[few].cpu().numpy()[k32], t64[few].cpu().numpy()[k64])
    assert np.array_equal(l32[few].cpu().numpy()[k32].view(np.uint32), l64[few].cpu().numpy()[k64].view(np.uint32))


def test_four_million_rays_at_max_hits_64_on_shells(cuda_device):
    """4 M rays on 32 concentric shells (up to 64 hits each) at max_hits 64: two staging windows of ~2 M rays, whose count
    scans cross ~1000 tiles each.  Every ray's group is complete (count <= 64); a seeded sample is checked hit for hit
    against the complete mirror hit list, the rest against the device count."""
    v, f = dc.scene("shells32")
    r = make(v, f, max_hits=64)
    n = 4_000_000
    g = torch.Generator(device=cuda_device)
    g.manual_seed(41)
    o = (torch.rand((n, 3), generator=g, device=cuda_device) * 2 - 1) * 1.2
    d = torch.randn((n, 3), generator=g, device=cuda_device)
    d = d / torch.norm(d, dim=-1, keepdim=True)
    assert hops.allhits_window_rays(64) < n <= 2 * hops.allhits_window_rays(64)
    ti, ri, loc = r.intersects_id(o, d, return_locations=True)
    cnt = r.intersects_count(o, d)
    assert int(cnt.max()) <= 64 and int(cnt.max()) > 32
    ri_l = ri.long()
    assert bool((ri_l[1:] >= ri_l[:-1]).all())
    assert torch.equal(torch.bincount(ri_l, minlength=n), cnt.long())
    rng = np.random.default_rng(5)
    sample = np.sort(rng.choice(n, 20_000, replace=False))
    on, dn = o.cpu().numpy()[sample], d.cpu().numpy()[sample]
    ch = dc.complete_hits(v, f, on, dn)
    assert np.array_equal(cnt.cpu().numpy()[sample], ch["count"])
    start = torch.cat([torch.zeros(1, dtype=torch.long, device=cuda_device), torch.cumsum(cnt.long(), 0)]).cpu().numpy()
    rows = np.concatenate([np.arange(start[s], start[s + 1]) for s in sample])
    local = np.repeat(np.arange(len(sample)), ch["count"])
    rows_t = torch.from_numpy(rows).to(cuda_device)
    assert np.array_equal(ri_l[rows_t].cpu().numpy(), sample[local])
    dc.check_hits_subset(ch, local, ti[rows_t].cpu().numpy(), loc[rows_t].cpu().numpy(), "4 M rays sample")
