"""Generalized winding number on one GPU (rt_winding_moments, rt_winding_number): moment-pass time, throughput with
traversal counters, bit-for-bit parity with the host simulator, accuracy against the binary64 oracle, exact mode, and
signed_distance with the winding sign against the contains sign.

Meshes: the config-2 icosphere (327 680 triangles), the config-4 soup (1 M), the config-3 heightfield (4.19 M) and,
for the moment pass only, the config-5 heightfield (16.8 M).  Point sets (a)-(c) of BASELINE §6: (a) 10 M points
jittered around the surface (sigma = 1 % of the bbox diagonal), (b) 10 M points uniform in the 1.2x bbox, (c) a 256^3
grid over the 1.2x bbox in row-major order.  Every call is timed with CUDA events after a warm-up, with L2 overwritten
before every timed pass.  A separate instrumented call gives nodes, exact triangles and far-field terms per point;
bytes per point = 80 per node + 64 per inner child's moment record + 48 per triangle + 12 in + 4 out, an upper bound of
what traversal touches.  A sample of every set is compared bit for bit with the host simulator (tests/winding/), a
smaller one with the binary64 brute-force oracle (max and p99 |dw|).

    python tools/winding_number_probe.py [--out profiles/winding_number_probe.json] [--points 10000000] [--grid 256]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT, os.path.join(ROOT, "tests", "winding"),
          os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import winding as W  # noqa: E402
from closest_point_probe import card, point_sets, time_call  # noqa: E402
from triro import synth  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402

MAKERS = {"config2_icosphere": lambda: synth.icosphere(7), "config4_soup": lambda: synth.triangle_soup(1_000_000),
          "config3_heightfield": lambda: synth.heightfield(2048, 1024),
          "config5_heightfield": lambda: synth.heightfield(4096, 2048)}


def moments_ms(acc, reps, flush):
    inner = acc._inner

    def run():
        inner.winding_moments = None
        hops.winding_moments(acc)
    return time_call(run, reps, flush)


def bits_equal(a, b):
    return bool(np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "winding_number_probe.json"))
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=20_000, help="points per set compared with the host simulator")
    ap.add_argument("--accuracy", type=int, default=1_000, help="points per set compared with the binary64 oracle")
    ap.add_argument("--meshes", default="config2_icosphere,config4_soup,config3_heightfield")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("winding_number_probe needs a CUDA device: nothing is measured without one")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "torch": torch.__version__, "host_threads": os.cpu_count(), "points": a.points, "grid": a.grid,
           "reps": a.reps, "beta": 2.0, "timing": "CUDA events per call, median of reps, L2 overwritten before each",
           "moments": [], "rows": [], "exact": [], "signed_distance": []}
    for mname in a.meshes.split(",") + ["config5_heightfield"]:
        v, f = MAKERS[mname]()
        rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
        acc = rmi.as_wrapper
        ms = moments_ms(acc, a.reps, flush)
        out["moments"].append(dict(mesh=mname, tris=int(len(f)), nodes=acc.header["n_nodes"], ms_median=float(np.median(ms)),
                                   ms_all=ms))
        print(json.dumps(out["moments"][-1]), flush=True)
        if mname == "config5_heightfield":
            del rmi, acc
            torch.cuda.empty_cache()
            continue
        blob = acc.blob.cpu().numpy()
        host_m = W.sim_moments(blob)
        moments_equal = bits_equal(hops.winding_moments(acc)[: len(host_m)].cpu().numpy(), host_m)
        diag, sets = point_sets(v, a.points, a.grid, dev)
        for sname in ("a_surface", "b_uniform", "c_grid"):
            pts = sets[sname][0]
            n = pts.shape[0]
            ms = time_call(lambda: hops.winding_number(acc, pts, 2.0), a.reps, flush)
            cnt = torch.zeros(4, dtype=torch.int64, device=dev)
            w = hops.winding_number(acc, pts, 2.0, counters=cnt)
            nodes, tris, npts, far = cnt.tolist()
            med = float(np.median(ms))
            step = max(1, n // a.parity) if sname == "c_grid" else 1
            sl = slice(0, a.parity * step, step)
            sample = pts[sl].cpu().numpy()
            sim = W.sim_winding(blob, sample, 2.0, host_m)
            t0 = time.time()
            # brute force costs points x triangles: the 4.19 M-triangle heightfield gets a tenth of the sample
            acc_n = a.accuracy if len(f) <= 2_000_000 else a.accuracy // 10
            acc_sl = slice(0, acc_n * max(1, n // acc_n), max(1, n // acc_n)) if sname == "c_grid" else slice(0, acc_n)
            truth = W.truth(v, f, pts[acc_sl].cpu().numpy())
            truth_s = time.time() - t0
            dw = np.abs(w[acc_sl].cpu().numpy().astype(np.float64) - truth)
            row = dict(mesh=mname, tris=int(len(f)), points=sname, n=n, ms_median=med, ms_all=ms, mpts_s=n / med / 1e3,
                       nodes_per_pt=nodes / npts, exact_tris_per_pt=tris / npts, far_terms_per_pt=far / npts,
                       bytes_per_pt_bound=(80 * nodes + 64 * (nodes - npts + far) + 48 * tris) / npts + 12 + 4,
                       parity_points=len(sample), parity_hostsim_bit_exact=bits_equal(w[sl].cpu().numpy(), sim["w"]),
                       moments_bit_exact=moments_equal, accuracy_points=len(truth), max_abs_dw=float(dw.max()),
                       p99_abs_dw=float(np.percentile(dw, 99)), truth_oracle_s=truth_s)
            out["rows"].append(row)
            print(json.dumps({k: (round(x, 6) if isinstance(x, float) else x) for k, x in row.items() if k != "ms_all"}), flush=True)
            del w
        # signed distance: the winding sign against the contains sign, on the uniform points
        pts = sets["b_uniform"][0]
        ms_w = time_call(lambda: rmi.signed_distance(pts, sign="winding"), a.reps, flush)
        ms_c = time_call(lambda: rmi.signed_distance(pts, sign="contains"), a.reps, flush)
        sw, sc = rmi.signed_distance(pts, sign="winding"), rmi.signed_distance(pts, sign="contains")
        out["signed_distance"].append(dict(mesh=mname, points="b_uniform", n=pts.shape[0], ms_winding=float(np.median(ms_w)),
                                           ms_contains=float(np.median(ms_c)),
                                           sign_agreement=float(((sw > 0) == (sc > 0)).float().mean()),
                                           magnitudes_equal=bool(torch.equal(sw.abs(), sc.abs()))))
        print(json.dumps(out["signed_distance"][-1]), flush=True)
        del rmi, acc, sets, sw, sc
        torch.cuda.empty_cache()
    # exact mode (beta = inf) on a small mesh
    v, f = synth.icosphere(5)
    rmi = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    acc = rmi.as_wrapper
    _, sets = point_sets(v, 1_000_000, 2, dev)
    pts = sets["b_uniform"][0]
    ms = time_call(lambda: hops.winding_number(acc, pts, float("inf")), a.reps, flush)
    w = hops.winding_number(acc, pts, float("inf"))
    sample = pts[: a.accuracy].cpu().numpy()
    sim = W.sim_winding(acc.blob.cpu().numpy(), sample, float("inf"))
    dw = np.abs(w[: a.accuracy].cpu().numpy().astype(np.float64) - W.truth(v, f, sample))
    out["exact"].append(dict(mesh="icosphere5", tris=int(len(f)), points="b_uniform", n=pts.shape[0],
                             ms_median=float(np.median(ms)), mpts_s=pts.shape[0] / float(np.median(ms)) / 1e3,
                             parity_hostsim_bit_exact=bits_equal(w[: a.accuracy].cpu().numpy(), sim["w"]),
                             max_abs_dw=float(dw.max()), p99_abs_dw=float(np.percentile(dw, 99))))
    print(json.dumps(out["exact"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
