"""Shared helpers of the parity tests (test infrastructure)."""
from __future__ import annotations

import numpy as np

from oracle import oracle


def assert_bits_equal(a, b, what=""):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.dtype.kind == "f":
        bad = a.view(np.uint32) != b.view(np.uint32)
    else:
        bad = a != b
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} elements differ (first at {np.argwhere(bad)[0]})"


def window_of(n, sizes_fn, workspace_bytes):
    """The window a gradient entry point picks for n rows: the largest number of rows, at most n, whose workspace
    sizes_fn(rows) fits workspace_bytes."""
    lo, hi = 0, n + 1
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if sizes_fn(mid) <= workspace_bytes else (lo, mid)
    return lo


def closest_to_numpy(res):
    hit, front, tri, loc, uv = res
    return dict(hit=hit.cpu().numpy().reshape(-1).astype(np.uint8), front=front.cpu().numpy().reshape(-1).astype(np.uint8),
                tri=tri.cpu().numpy().reshape(-1), loc=loc.cpu().numpy().reshape(-1, 3), uv=uv.cpu().numpy().reshape(-1, 2))


def check_closest_vs_mirror(got: dict, mesh: oracle.OracleMesh, o, d):
    """Bit-exact comparison against the oracle's binary32 mirror (every ray, no exclusions)."""
    ref = oracle.query(mesh, o, d, oracle.MIRROR, closest_only=True, want=("hit", "front", "tri", "loc", "uv"))
    for k in ("hit", "front", "tri", "loc", "uv"):
        assert_bits_equal(got[k], ref[k], f"closest.{k} vs mirror")
    return ref


def check_closest_vs_truth(got: dict, mesh: oracle.OracleMesh, o, d, max_graze_fraction=0.02, rel_tol=1e-5):
    """Comparison against the binary64 truth: masks and indices exact outside the documented
    grazing set, locations / uv within rel_tol (relative to the scene scale, as north_star says
    1e-5 relative)."""
    ref = oracle.query(mesh, o, d, oracle.TRUTH, want=("hit", "front", "tri", "loc", "uv", "flags", "t"))
    graze = ref["flags"] != 0
    assert graze.mean() <= max_graze_fraction, f"grazing set too large: {graze.mean():.4f}"
    clean = ~graze
    for k in ("hit", "front", "tri"):
        bad = (got[k] != ref[k]) & clean
        assert not bad.any(), f"closest.{k}: {int(bad.sum())} non-grazing rays differ from the binary64 truth"
    both = clean & (ref["hit"] == 1) & (got["hit"] == 1)
    if both.any():
        scale = max(1.0, float(np.abs(mesh.vertices).max()))
        err_loc = np.abs(got["loc"][both] - ref["loc"][both]).max() / scale
        err_uv = np.abs(got["uv"][both] - ref["uv"][both]).max()
        assert err_loc <= rel_tol, f"location error {err_loc:.3e} > {rel_tol}"
        # uv are O(1) weights; tolerance scales with ray length / triangle size (binary32 conditioning)
        assert err_uv <= 2e-3, f"uv error {err_uv:.3e}"
    return ref, graze


def compare_with_readme_figure(locs_800: np.ndarray):
    """Compares an [800,800,3] hit-location image (zeros where nothing was hit) with the plot area of the reference's
    published README figure (tests/golden/readme_location_png.npz, made by tests/golden/make_location_fixture.py).
    matplotlib's imshow clips RGB to [0,1] and resamples 800 px to ~370 px, hence the tolerances.
    Returns (mask IoU, mean abs colour difference on the disc)."""
    import os

    import torch
    import torch.nn.functional as F

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "readme_location_png.npz"))
    ref = g["plot_area"].astype(np.float32) / 255.0                       # [370, 369, 3]
    img = torch.from_numpy(np.clip(locs_800, 0.0, 1.0).astype(np.float32)).permute(2, 0, 1)[None]
    small = F.interpolate(img, size=ref.shape[:2], mode="area")[0].permute(1, 2, 0).numpy()
    m_ref = ref.sum(axis=2) > 0.16
    m_got = small.sum(axis=2) > 0.16
    iou = float((m_ref & m_got).sum() / max((m_ref | m_got).sum(), 1))
    both = m_ref & m_got
    diff = float(np.abs(ref[both] - small[both]).mean())
    return iou, diff
