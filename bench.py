#!/usr/bin/env python
"""bench.py — Mrays/s closest-hit (+ BVH build ms) on the BASELINE.json configurations, vs a CPU baseline.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: trimesh if importable, else the oracle port
    python bench.py --gpus 1 ... --dump-outputs DIR          # also write the last timed step's results to DIR/*.npy

N = 1  (config.workload = "config2"): icosphere subdivision 7 (327 680 triangles), 3840x2160 pinhole camera rays
       (8 294 400 rays, origin a stride-0 broadcast as in the reference's test/performance_test.py:36-41),
       `intersects_closest` incl. location + uv.  One step = one pass of the hot path over that ray batch.
       The line also carries a `configs` block: every other BASELINE configuration (README grid, the 1.31 M-triangle
       icosphere = north_star's 1 M-triangle target, config 3 any / count, config 4 closest / all hits /
       contains_points, the per-GPU slice of config 5, the reference's own 640x360 benchmark loop), each with its
       roofline fraction and a `parity` verdict from comparing a >= 1 M-ray subsample with the oracle's binary32
       mirror on the TRUE-SIZE mesh (outside every timed region).
N > 1  (config.workload = "config5"): north_star's multi-GPU job — 16.8 M-triangle heightfield built on rank 0 and
       NCCL-broadcast, 125 M random rays per rank (seed 100 + rank).  `value` = sharded
       `intersects_closest(stream_compaction=True)` (results stay on their rank: weak scaling, no data-path
       collective); `gathered` = the same call with the complete 6-tuple assembled on rank 0 (peer copies over
       NVLink, and the NCCL all-gather route beside it); `strong` = ONE 66 M-ray batch split N ways with the dense
       5-tuple landing on rank 0.

Timing: W >= 3 warm-up steps; every timed step is bracketed by CUDA events on the launch stream with an L2 flush
(512 MiB memset) between steps at N = 1 (at N > 1 a step's working set is 6 GB >> L2); the job time is the max over
ranks of the summed step times.  Clocks are sampled through NVML during the timed region.

--dump-outputs DIR (N = 1): after the timed steps, the closest-hit 5-tuple of the last step is written for a fixed,
seeded sample of DUMP_RAYS of the frame's rays as DIR/{ray_index,hit,front,tri_idx,location,uv}.npy (float64 ray
indices into the flattened frame, everything else float32; 40 MiB in all).  The workload is deterministic, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

sys.dont_write_bytecode = True      # the checkout may be read-only: nothing is written into it, not even __pycache__
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "trimesh-ray-optix_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

METRIC = "Mrays/s closest-hit"
UNIT = "Mrays/s"
WIDTH, HEIGHT = 3840, 2160
SUBDIV = 7
CFG5_GRID = (4096, 2048)            # 16 777 216 triangles
CFG5_RAYS_PER_GPU = 125_000_000
STRONG_RAYS = 8 * WIDTH * HEIGHT    # 66 355 200: one batch split N ways
E2E_RAYS_PER_GPU = 25_000_000       # N > 1: rays per rank and step of the host-buffer end-to-end leg
PARITY_RAYS = 1_000_000
DUMP_RAYS = 1 << 20
WORKLOAD2 = "config2: icosphere subdiv 7 (327680 tris), 3840x2160 pinhole rays, intersects_closest (hit, front, tri, loc, uv)"
WORKLOAD5 = ("config5: 4096x2048 heightfield (16777216 tris) built on rank 0 + NCCL broadcast, 125M random rays per GPU "
             "(seed 100+rank), intersects_closest(stream_compaction=True)")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def make_workload(device, rank: int):
    from triro import synth

    v, f = synth.icosphere(SUBDIV)
    # rank-dependent camera so that ranks do not trace identical rays
    o, d = synth.pinhole_rays(WIDTH, HEIGHT, device=device, origin=(0.02 * rank, -0.01 * rank, 3.0))
    return v, f, o, d


def config5_rays(n: int, seed: int, device):
    """Config-5 ray recipe: random_rays in 25 M-ray pieces (seeds seed*16 + piece) into one [n, 3] pair."""
    from triro import synth

    o = torch.empty((n, 3), device=device); d = torch.empty((n, 3), device=device)
    chunk = 25_000_000
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        oc, dc = synth.random_rays(m, seed=seed * 16 + i // chunk, device=device)
        o[i:i + m] = oc; d[i:i + m] = dc
        del oc, dc
    return o, d


def bytes_per_ray(stats: dict, b_in: float, b_out: float) -> float:
    return b_in + b_out + 80.0 * stats["nodes_per_ray"] + 48.0 * stats["tris_per_ray"]


# ------------------------------------------------------------------------------------- CPU side (oracle = the checker)
def oracle_all_cores():
    """The oracle on every host core, whatever OMP_NUM_THREADS a launcher (torch.distributed.run sets 1) exported."""
    from oracle import oracle

    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    return oracle, oracle.set_num_threads(max(cores, os.cpu_count() or 1))


def try_trimesh_closest(v, f, o_np, d_np):
    """The reference's own CPU comparison call (test/performance_test.py:75): trimesh's ray engine, if trimesh is
    importable on this box (it is not in the offline image).  Returns (seconds, n_hit) or None."""
    try:
        import trimesh  # noqa: F401
    except Exception:
        return None
    mesh = trimesh.Trimesh(vertices=v, faces=f, process=False)
    t0 = time.perf_counter()
    loc, ray_idx, tri_idx = mesh.ray.intersects_location(o_np, d_np, multiple_hits=False)
    return time.perf_counter() - t0, len(ray_idx)


def cpu_closest(v, f, o_np, d_np, sample: int, reps: int = 1):
    """Times the oracle port (binary32 mirror behind its binned-SAH BVH2, OpenMP over rays) on a bounded sample of
    the workload's rays.  Returns (Mrays/s, cores, sample description, seconds)."""
    oracle, cores = oracle_all_cores()
    n = len(d_np)
    stride = max(1, n // sample)
    d_s = np.ascontiguousarray(d_np[::stride])
    o_s = np.ascontiguousarray(np.broadcast_to(o_np, d_np.shape)[::stride])
    mesh = oracle.OracleMesh(v, f, use_bvh=True)           # BVH build is not timed (neither is the GPU's)
    oracle.query(mesh, o_s[:1000], d_s[:1000], oracle.MIRROR, closest_only=True, want=("hit", "tri", "loc", "uv", "front"))
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        oracle.query(mesh, o_s, d_s, oracle.MIRROR, closest_only=True, want=("hit", "front", "tri", "loc", "uv"))
        best = min(best, time.perf_counter() - t0)
    what = "the full frame" if stride == 1 else f"every {stride}th ray of the {WIDTH}x{HEIGHT} frame"
    return len(d_s) / best / 1e6, cores, f"{what} ({len(d_s)} rays)", best


def parity_closest(om, res, o, d, idx=None) -> dict:
    """Compares a closest-hit 5-tuple (optionally the rows `idx` of it) with the oracle's binary32 mirror on the same
    rays: every field, every ray, bit for bit."""
    from oracle import oracle

    on = (o if idx is None else o[idx]).detach().cpu().numpy().reshape(-1, 3)
    dn = (d if idx is None else d[idx]).detach().cpu().numpy().reshape(-1, 3)
    ref = oracle.query(om, on, dn, oracle.MIRROR, closest_only=True, want=("hit", "front", "tri", "loc", "uv"))
    names = ("hit", "front", "tri", "loc", "uv")
    bad = {}
    for k, t in zip(names, res):
        g = (t if idx is None else t[idx]).detach().cpu().numpy()
        r = ref[k]
        g = g.reshape(r.shape)
        if r.dtype.kind == "f":
            nb = int((g.view(np.uint32) != r.view(np.uint32)).sum())
        else:
            nb = int((g.astype(r.dtype) != r).sum())
        if nb:
            bad[k] = nb
    return {"parity": "bit-exact" if not bad else "MISMATCH", "rays_checked": len(on), "mismatches": bad or None,
            "against": "oracle MIRROR (binary32) on the true-size mesh"}


def dump_closest(out_dir: str, res, n: int) -> None:
    """Writes the rows of a dense closest-hit 5-tuple over n rays picked by a fixed seed as out_dir/<name>.npy."""
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_RAYS, n), replace=False))
    sel = torch.from_numpy(idx).to(res[0].device)
    np.save(os.path.join(out_dir, "ray_index.npy"), idx.astype(np.float64))
    for name, t in zip(("hit", "front", "tri_idx", "location", "uv"), res):
        rows = t.reshape(n, *t.shape[res[0].dim():])[sel]
        np.save(os.path.join(out_dir, f"{name}.npy"), rows.cpu().numpy().astype(np.float32))   # tri_idx < 2^24: exact


def parity_ints(name, got, ref) -> dict:
    nb = int((np.asarray(got).reshape(-1) != np.asarray(ref).reshape(-1)).sum())
    return {"parity": "bit-exact" if nb == 0 else "MISMATCH", "rays_checked": int(np.asarray(ref).size),
            "mismatches": {name: nb} if nb else None, "against": "oracle MIRROR (binary32) on the true-size mesh"}


def run_reference(args):
    """--impl reference: the reference's own CPU path is trimesh (+embree), absent offline, and its GPU path needs the
    OptiX SDK (absent); this arm therefore times trimesh when it imports and otherwise the oracle port of the path,
    on ALL host cores, on the same workload as this repo's arm at that N.  Rank 0 alone runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from triro import synth

    oracle, cores = oracle_all_cores()
    world = args.gpus
    want = ("hit", "front", "tri", "loc", "uv")
    if world == 1:
        v, f = synth.icosphere(SUBDIV)
        o, d = synth.pinhole_rays(WIDTH, HEIGHT, device="cpu")
        d_s = np.ascontiguousarray(d.reshape(-1, 3).numpy())
        o_s = np.ascontiguousarray(np.broadcast_to(np.array([[0.0, 0.0, 3.0]], np.float32), d_s.shape))
        workload, sample, same = WORKLOAD2, f"the full {WIDTH}x{HEIGHT} frame ({len(d_s)} rays) per step", True
    else:
        v, f = synth.heightfield(*CFG5_GRID)
        n = 8_000_000
        o, d = synth.random_rays(n, seed=100 * 16, device="cpu")     # = the first 8 M rays of rank 0's config-5 slice
        o_s, d_s = np.ascontiguousarray(o.numpy()), np.ascontiguousarray(d.numpy())
        workload = WORKLOAD5
        sample, same = f"bounded sample: the first {n} rays of rank 0's 125M-ray slice per step (dense closest hit, no compaction)", False
    tm = try_trimesh_closest(v, f, o_s[: 200_000], d_s[: 200_000]) if world == 1 else None
    mesh = oracle.OracleMesh(v, f, use_bvh=True)
    for _ in range(max(min(args.warmup, 2), 1)):
        oracle.query(mesh, o_s, d_s, oracle.MIRROR, closest_only=True, want=want)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.query(mesh, o_s, d_s, oracle.MIRROR, closest_only=True, want=want)
    dt = (time.perf_counter() - t0) / steps
    val = len(d_s) / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "step": sample, "same_config": same},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample + "; oracle binary32 mirror behind its own binned-SAH BVH2 (scalar, double-precision boxes), OpenMP over rays"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "trimesh": ({"available": True, "mrays_s": 200_000 / tm[0] / 1e6, "sample": "200000 rays, mesh.ray.intersects_location(multiple_hits=False)"}
                    if tm else {"available": False, "why": "import trimesh fails in the offline image (reference test/performance_test.py:75 is the call that would be timed)"}),
        "note": "reference OptiX path not buildable offline (no OptiX SDK); CPU arm = oracle port, a stated baseline and not an Embree-class tracer",
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------- GPU arm helpers
class Timer:
    def __init__(self, dev, flush=None):
        self.dev, self.flush = dev, flush

    def __call__(self, fn, reps=3, warm=1):
        ts, out = [], None
        for i in range(warm + reps):
            out = None
            if self.flush is not None:
                self.flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out = fn(); e1.record(); torch.cuda.synchronize(self.dev)
            if i >= warm:
                ts.append(e0.elapsed_time(e1))
        return min(ts), out


def build_timed(vt, ft, dev):
    from triro.backend import ops as hops

    accel = hops.AccelStructure()
    vd, fd = vt.to(dev), ft.to(dev)
    ms = []
    for _ in range(4):
        accel.build(vd, fd, timing=True)
        ms.append(accel.build_ms)
    accel.free()
    return min(ms[1:])


def config_row(rmi, name, query, n, ms, stats, b_in, b_out, peak, build_ms, parity, note=None):
    bpr = bytes_per_ray(stats, b_in, b_out) if stats else None
    h = rmi.as_wrapper.header
    row = {"config": name, "query": query, "tris": h["n_tris"], "rays": n, "ms": ms, "mrays_s": n / ms / 1e3,
           "nodes_per_ray": stats["nodes_per_ray"] if stats else None, "tris_per_ray": stats["tris_per_ray"] if stats else None,
           "bytes_per_ray": bpr, "frac": (bpr * n / (ms * 1e-3) / (peak * 1e9)) if bpr else None,
           "build_ms": build_ms, "blob_mb": h["used_bytes"] / 1e6}
    row.update(parity or {"parity": None})
    if note:
        row["note"] = note
    return row


def run_configs(dev, peak, timer) -> list:
    """Every BASELINE configuration other than the headline one, on this GPU; parity against the oracle on >= 1 M-ray
    subsamples of the true-size meshes, outside the timed regions."""
    from triro import synth
    from triro.backend import ops as hops
    from triro.ray.ray_optix import RayMeshIntersector

    oracle, _ = oracle_all_cores()
    rows = []

    def mk(v, f):
        vt, ft = torch.from_numpy(v), torch.from_numpy(f)
        return RayMeshIntersector(vertices=vt, faces=ft), build_timed(vt, ft, dev)

    # ---- config 1: README quick-start (README.md:24-51), 800x800 grid, stream compaction, trimesh's default icosphere too
    for sub in (2, 3):
        v, f = synth.icosphere(sub)
        r, bms = mk(v, f)
        o, d = synth.readme_rays(800, device=dev)
        ms, out = timer(lambda: r.intersects_closest(o, d, stream_compaction=True), reps=5, warm=2)
        dense = r.intersects_closest(o, d)
        om = oracle.OracleMesh(v, f, use_bvh=False)
        par = parity_closest(om, dense, o, d)
        hitfrac = float(out[0].float().mean())
        ok = bool(torch.equal(out[2].long(), torch.nonzero(out[0].reshape(-1)).reshape(-1)))
        if not ok:
            par["parity"] = "MISMATCH"; par["mismatches"] = {"ray_idx": "not the positions of the hit mask"}
        st = hops.trace_stats(r.as_wrapper, o, d, "closest")
        rows.append(config_row(r, f"1 (README grid, icosphere subdiv {sub})", "intersects_closest(stream_compaction=True)", 640_000, ms,
                               st, 12, 1 + 29 * hitfrac, peak, bms, par, "dense trace + scan + host sync + scatter; all 640000 rays checked"))
        del r, o, d, out, dense
    # ---- north_star's target: closest hit on a 1 M-triangle MESH (icosphere subdiv 8 = 1 310 720 triangles), 4K camera
    v, f = synth.icosphere(8)
    r, bms = mk(v, f)
    o, d = synth.pinhole_rays(WIDTH, HEIGHT, device=dev)
    n = WIDTH * HEIGHT
    ms, out = timer(lambda: r.intersects_closest(o, d), reps=5, warm=2)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    idx = torch.arange(0, n, 8, device=dev)                      # every 8th ray of the frame: 1 036 800 rays
    flat = tuple(x.reshape(n, *x.shape[2:]) for x in out)
    par = parity_closest(om, flat, o.reshape(n, 3), d.reshape(n, 3), idx)
    st = hops.trace_stats(r.as_wrapper, o, d, "closest")
    rows.append(config_row(r, "1M-triangle mesh (icosphere subdiv 8, 1310720 tris), 3840x2160 pinhole", "intersects_closest", n, ms, st, 12, 26,
                           peak, bms, par, "north_star target: >= 70 % of the memory roofline for closest-hit on a 1M-triangle mesh"))
    del r, o, d, out, flat, om
    # ---- config 3: 4.19 M-triangle heightfield, 100 M random rays, any + count
    v, f = synth.heightfield(2048, 1024)
    r, bms = mk(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    n = 100_000_000
    o = torch.empty((n, 3), device=dev); d = torch.empty((n, 3), device=dev)
    for i in range(10):
        oc, dc = synth.random_rays(10_000_000, seed=1234 + i, device=dev)
        o[i * 10_000_000:(i + 1) * 10_000_000] = oc; d[i * 10_000_000:(i + 1) * 10_000_000] = dc
        del oc, dc
    sub = slice(0, PARITY_RAYS)
    on, dn = o[sub].cpu().numpy(), d[sub].cpu().numpy()
    ref_cnt = oracle.query(om, on, dn, oracle.MIRROR, want=("count",))["count"]
    ms, anyh = timer(lambda: r.intersects_any(o, d), reps=3, warm=1)
    st = hops.trace_stats(r.as_wrapper, o, d, "any")
    rows.append(config_row(r, "3 (heightfield 2048x1024, 100M random rays)", "intersects_any", n, ms, st, 24, 1, peak, bms,
                           parity_ints("any", anyh[sub].cpu().numpy(), ref_cnt > 0)))
    del anyh
    ms, cnt = timer(lambda: r.intersects_count(o, d), reps=3, warm=1)
    st = hops.trace_stats(r.as_wrapper, o, d, "count")
    rows.append(config_row(r, "3 (heightfield 2048x1024, 100M random rays)", "intersects_count", n, ms, st, 24, 4, peak, bms,
                           parity_ints("count", cnt[sub].cpu().numpy(), ref_cnt)))
    del cnt
    closest_sub = r.intersects_closest(o[sub], d[sub])
    par_c3 = parity_closest(om, closest_sub, o[sub], d[sub])
    rows[-1]["closest_parity_same_rays"] = par_c3["parity"]
    del r, o, d, om, closest_sub
    torch.cuda.empty_cache()
    # ---- config 4: 1 M-triangle soup; 10 M points contains_points (default direction and +x), 10 M rays all hits + closest
    v, f = synth.triangle_soup(1_000_000)
    r, bms = mk(v, f)
    om = oracle.OracleMesh(v, f, use_bvh=True)
    n = 10_000_000
    g = torch.Generator(device=dev); g.manual_seed(8)
    pts = torch.rand((n, 3), generator=g, device=dev) * 2 - 1
    torch.manual_seed(0)
    ms, inside = timer(lambda: r.contains_points(pts), reps=3, warm=1)
    oi = oracle.OracleIntersector.__new__(oracle.OracleIntersector)
    oi.mesh, oi.mode, oi.mesh_aabb = om, oracle.MIRROR, (v.min(axis=0), v.max(axis=0))
    m = 250_000
    ins, cp, cm = oi.contains_core(pts[:m].cpu().numpy(), r.DEFAULT_CHECK_DIRECTION)
    agree = (cp % 2 == 1) & (cm % 2 == 1)
    contain, broken, _ = r.contains_parity(pts[:m], r.DEFAULT_CHECK_DIRECTION)
    nb = int((contain.cpu().numpy() != (ins & agree)).sum() + (broken.cpu().numpy() != (~agree & ((cp == 0) | (cm == 0)))).sum())
    par = {"parity": "bit-exact" if nb == 0 else "MISMATCH", "rays_checked": 2 * m, "mismatches": {"contain/broken": nb} if nb else None,
           "against": "oracle MIRROR counts along +-dir for the first 250000 points (parity core; the retry direction is random)"}
    row = config_row(r, "4 (1M-triangle soup, 10M points)", "contains_points (default direction)", n, ms, None, 0, 0, peak, bms, par,
                     f"fused +-dir parity launch + masked in-place retry of the broken points; inside fraction {float(inside.float().mean()):.3e}")
    row["mpoints_s"] = row.pop("mrays_s")
    rows.append(row)
    xdir = torch.tensor([1.0, 0.0, 0.0], device=dev)
    ms, inside_x = timer(lambda: r.contains_points(pts, xdir), reps=3, warm=1)
    ins, cp, cm = oi.contains_core(pts[:m].cpu().numpy(), [1.0, 0.0, 0.0])
    agree = (cp % 2 == 1) & (cm % 2 == 1)
    contain, broken, _ = r.contains_parity(pts[:m], [1.0, 0.0, 0.0])
    nb = int((contain.cpu().numpy() != (ins & agree)).sum() + (broken.cpu().numpy() != (~agree & ((cp == 0) | (cm == 0)))).sum())
    par = {"parity": "bit-exact" if nb == 0 else "MISMATCH", "rays_checked": 2 * m, "mismatches": {"contain/broken": nb} if nb else None,
           "against": "oracle MIRROR counts along +-x for the first 250000 points"}
    row = config_row(r, "4 (1M-triangle soup, 10M points)", "contains_points (+x)", n, ms, None, 0, 0, peak, bms, par,
                     "explicit direction: the reference returns all False when any point is 'broken' (ray_optix.py:279) - kept")
    row["mpoints_s"] = row.pop("mrays_s")
    rows.append(row)
    del pts, inside, inside_x
    o, d = synth.random_rays(n, seed=9, device=dev, box=True)
    sub = slice(0, PARITY_RAYS)
    ms, out = timer(lambda: r.intersects_location(o, d), reps=3, warm=1)
    loc, ri, ti = out
    ref = oracle.query(om, o[sub].cpu().numpy(), d[sub].cpu().numpy(), oracle.MIRROR, list_cap=16, want=("count",))
    cnt_g = r.intersects_count(o, d)
    st = hops.trace_stats(r.as_wrapper, o, d, "count")
    hits_sub = int(np.minimum(ref["count"], 8).sum())
    lim = int((ri < PARITY_RAYS).sum())
    ok_counts = bool(np.array_equal(np.bincount(ri[:lim].cpu().numpy(), minlength=PARITY_RAYS), np.minimum(ref["count"], 8)))
    # per-ray triangle sets (rays with <= 8 hits): sort (ray, tri) on both sides
    got_pairs = np.stack([ri[:lim].cpu().numpy(), ti[:lim].cpu().numpy()], 1)
    k = np.minimum(ref["count"], 8)
    full_rays = ref["count"] <= 8
    ref_pairs = np.array([(i, t) for i in np.nonzero(full_rays & (k > 0))[0][:200_000] for t in ref["list_tri"][i, :k[i]]], dtype=np.int64).reshape(-1, 2)
    sel = np.isin(got_pairs[:, 0], np.unique(ref_pairs[:, 0]))
    gp = got_pairs[sel]; gp = gp[np.lexsort((gp[:, 1], gp[:, 0]))]; rp = ref_pairs[np.lexsort((ref_pairs[:, 1], ref_pairs[:, 0]))]
    ok_sets = gp.shape == rp.shape and bool((gp == rp).all())
    par = {"parity": "bit-exact" if (ok_counts and ok_sets and lim == hits_sub) else "MISMATCH", "rays_checked": PARITY_RAYS,
           "mismatches": None if (ok_counts and ok_sets) else {"counts_ok": ok_counts, "sets_ok": ok_sets},
           "against": "oracle MIRROR hit lists: clamped counts of 1M rays, per-ray triangle sets of the first 200000 rays with hits"}
    rows.append(config_row(r, "4 (1M-triangle soup, 10M random rays)", "intersects_location (all hits)", n, ms, st, 24,
                           4 + 20 * float(cnt_g.clamp(max=8).float().mean()), peak, bms, par,
                           f"one traversal in bounded staging windows + scan + host sync + scatter; mean hits/ray {float(cnt_g.float().mean()):.2f}, rays with > 8 hits {float((cnt_g > 8).float().mean()):.2e}"))
    del out, loc, ri, ti, cnt_g
    ms, out = timer(lambda: r.intersects_closest(o, d), reps=3, warm=1)
    st = hops.trace_stats(r.as_wrapper, o, d, "closest")
    rows.append(config_row(r, "4 (1M-triangle soup, 10M random rays)", "intersects_closest", n, ms, st, 24, 26, peak, bms,
                           parity_closest(om, tuple(x[sub] for x in out), o[sub], d[sub])))
    del r, o, d, om, out
    torch.cuda.empty_cache()
    # ---- the per-GPU slice of config 5 (the N = 1 counterpart of the N > 1 `value`): 16.8 M triangles, 125 M rays
    v, f = synth.heightfield(*CFG5_GRID)
    r, bms = mk(v, f)
    n = CFG5_RAYS_PER_GPU
    o, d = config5_rays(n, 100, dev)
    ms, out = timer(lambda: r.intersects_closest(o, d, stream_compaction=True), reps=3, warm=1)
    del out
    ms_dense, out = timer(lambda: r.intersects_closest(o, d), reps=3, warm=1)
    st = hops.trace_stats(r.as_wrapper, o, d, "closest")
    om = oracle.OracleMesh(v, f, use_bvh=True)
    sub = slice(0, PARITY_RAYS)
    par = parity_closest(om, tuple(x[sub] for x in out), o[sub], d[sub])
    hf = float(out[0].float().mean())
    rows.append(config_row(r, "5 slice (heightfield 4096x2048 = 16777216 tris, 125M random rays = one rank of the 8-GPU job)",
                           "intersects_closest(stream_compaction=True)", n, ms, st, 24, 26 + 1 + 29 * hf, peak, bms, par,
                           f"blob 1 GB > L2; dense trace alone {ms_dense:.3f} ms = {n / ms_dense / 1e3:.0f} Mrays/s (frac {bytes_per_ray(st, 24, 26) * n / (ms_dense * 1e-3) / (peak * 1e9):.3f})"))
    del r, o, d, om, out
    torch.cuda.empty_cache()
    return rows


def perf_test_like(dev) -> dict:
    """The reference's own benchmark loop (test/performance_test.py:29-60): 640x360 pinhole rays, N back-to-back
    intersects_closest calls, wall clock, one synchronisation at the end.  Published: 83.6 us per call on an RTX 3090
    with RT cores on the reference's own scene (README.md:63-68); here the 327 680-triangle icosphere."""
    from triro import synth
    from triro.ray.ray_optix import RayMeshIntersector

    cam_mat = torch.tensor([[5.6272650e-01, 2.7091104e-01, 7.8099048e-01], [8.2602328e-01, -1.4769979e-01, -5.4393965e-01],
                            [3.2007132e-02, -9.5120555e-01, 3.0689341e-01]], device=dev)
    rw = 640; rh = int(rw * 9 / 16); rf = int(rw * 25 / 36)
    v, f = synth.icosphere(7)
    dirs = synth.gen_rays(cam_mat, rw, rh, rf, device=dev)
    origins = (cam_mat[:, 2] * 3.0).broadcast_to(dirs.shape)
    r = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    for _ in range(200):
        res = r.intersects_closest(origins, dirs)
    torch.cuda.synchronize(dev)
    iters = 5000
    t0 = time.perf_counter()
    for _ in range(iters):
        res = r.intersects_closest(origins, dirs)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); res = r.intersects_closest(origins, dirs); e1.record(); torch.cuda.synchronize(dev)
    # host floor: the same call on a mesh of 20 triangles (traversal ~ nothing)
    v0, f0 = synth.icosphere(0)
    r0 = RayMeshIntersector(vertices=torch.from_numpy(v0), faces=torch.from_numpy(f0))
    for _ in range(200):
        r0.intersects_closest(origins, dirs)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(iters):
        r0.intersects_closest(origins, dirs)
    torch.cuda.synchronize(dev)
    dt0 = time.perf_counter() - t0
    return {"us_per_call": dt / iters * 1e6, "device_us_one_call": e0.elapsed_time(e1) * 1e3, "rays_per_call": rw * rh,
            "mrays_s": rw * rh * iters / dt / 1e6, "hit_fraction": float(res[0].float().mean()),
            "us_per_call_20_triangle_mesh": dt0 / iters * 1e6,
            "reference_published_us_per_call": 83.6,
            "note": "reference loop test/performance_test.py:29-60 (640x360, no sync inside the loop); its published 83.6 us is an RTX 3090 with RT cores on its own scene file (README.md:63-68), which is not available offline"}


def ncu_side_data():
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)
    return {}


# ------------------------------------------------------------------------------------- GPU arm, N = 1
def run_b200_single(args, dev):
    from triro.backend import ops as hops
    from triro.ray.ray_optix import RayMeshIntersector

    all_cpus = os.sched_getaffinity(0)
    v, f, o, d = make_workload(dev, 0)
    vt, ft = torch.from_numpy(v), torch.from_numpy(f)
    rmi = RayMeshIntersector(vertices=vt, faces=ft)
    build_ms = build_timed(vt, ft, dev)
    n = d.numel() // 3
    stats = hops.trace_stats(rmi.as_wrapper, o, d, "closest")
    bpr = bytes_per_ray(stats, 12.0, 26.0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    steps, warm = args.steps, max(args.warmup, 3)

    def one_step():
        return rmi.intersects_closest(o, d)

    for _ in range(warm):
        res = one_step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ClockSampler(dev.index) as clk:
        for a, b in ev:
            flush.zero_()                       # evict the previous step's working set from L2 (untimed)
            a.record()
            res = one_step()
            b.record()
        torch.cuda.synchronize()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    if args.dump_outputs:
        assert len(f) < 1 << 24, "tri_idx would not be exact in float32"
        dump_closest(args.dump_outputs, res, n)

    # end-to-end through the host-buffer entry points: pinned host rays in, pinned host results out
    o_host = torch.tensor([0.0, 0.0, 3.0]).pin_memory()
    d_host = d.reshape(-1, 3).cpu().pin_memory()
    out = hops.host_closest(rmi.as_wrapper, o_host, d_host)
    for _ in range(2):
        out = hops.host_closest(rmi.as_wrapper, o_host, d_host, out=out)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = hops.host_closest(rmi.as_wrapper, o_host, d_host, out=out)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    assert int(out["hit"].sum()) == int(res[0].sum()), "host path and device path disagree"
    outc = hops.host_closest(rmi.as_wrapper, o_host, d_host, stream_compaction=True)
    for _ in range(2):
        outc = hops.host_closest(rmi.as_wrapper, o_host, d_host, out=outc, stream_compaction=True)
    t0 = time.perf_counter()
    for _ in range(steps):
        outc = hops.host_closest(rmi.as_wrapper, o_host, d_host, out=outc, stream_compaction=True)
    e2e_c_ms = (time.perf_counter() - t0) * 1e3
    nh = outc["n_hit"]
    assert nh == int(res[0].sum()) and torch.equal(outc["tri_c"], res[2].reshape(-1)[res[0].reshape(-1)].cpu()), "compacting host path disagrees"
    del out, outc, d_host

    peak, peak_src = measured_peaks()
    ms_per_step = total_ms / steps
    value = n * steps / (total_ms * 1e-3) / 1e6
    kernel_ms = statistics.mean(step_ms)
    achieved = bpr * n / (kernel_ms * 1e-3) / 1e9
    side = ncu_side_data()
    traffic = side.get("k_trace_closest_config2_dram_bytes_per_launch")
    inst = side.get("k_trace_closest_config2_warp_instructions_per_launch")
    clocks = clk.summary()
    sm_count = hops.get_module().rt_device_sm_count()
    issue_frac = None
    if inst and clocks.get("sm_mhz"):
        issue_frac = inst / (sm_count * 4 * clocks["sm_mhz"] * 1e6 * kernel_ms * 1e-3)
    # headline parity: every 8th ray of the timed frame against the oracle on the same mesh
    oracle, _ = oracle_all_cores()
    om = oracle.OracleMesh(v, f, use_bvh=True)
    idx = torch.arange(0, n, 8, device=dev)
    flat = tuple(x.reshape(n, *x.shape[2:]) for x in res)
    parity = parity_closest(om, flat, o.reshape(n, 3), d.reshape(n, 3), idx)
    del om, flat
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD2, "rays_per_gpu": n,
                   "l2": "flushed between steps (512 MiB memset); step working set 315 MB > 126 MB L2", "parallelism": "single GPU"},
        "parity": parity,
        "bvh_build_ms": build_ms, "bvh_nodes": rmi.as_wrapper.header["n_nodes"], "bvh_depth": rmi.as_wrapper.header["depth"],
        "bvh_blob_mb": rmi.as_wrapper.header["used_bytes"] / 1e6,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": "k_trace_coop<closest> (or k_trace, see schedule)",
                     "bytes_per_ray": bpr, "nodes_per_ray": stats["nodes_per_ray"], "tris_per_ray": stats["tris_per_ray"],
                     "hit_fraction": stats["hit_fraction"], "kernel_ms": kernel_ms,
                     "roofline_mrays_per_s": peak * 1e9 / bpr / 1e6,
                     "compulsory_bytes_per_ray": 12.0 + 26.0 + rmi.as_wrapper.header["used_bytes"] / n,
                     "traffic_over_algorithmic": (traffic / (bpr * n)) if traffic else None,
                     "issue_frac": issue_frac,
                     "issue_frac_note": "second, honest bound: warp instructions per launch (ncu smsp__inst_executed.sum, profiles/traffic.json) / (SMs x 4 schedulers x median SM clock x kernel time); the blob is L2-resident, so this - not HBM - is what binds config 2",
                     "ncu_commit": side.get("commit")},
        "e2e": {"value": n * steps / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": 12 * n + 12,
                "d2h_bytes_per_step": 26 * n, "api": "rt_host_trace_closest (pinned host buffers, ramped chunks up to 2 Mi rays on 3 streams)"},
        "e2e_compact": {"value": n * steps / (e2e_c_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": 12 * n + 12,
                        "d2h_bytes_per_step": n + 29 * nh, "api": "rt_host_trace_closest_compact: stream_compaction=True on the device, only the hit mask + packed rows cross PCIe"},
        "gpu_launches": steps, "clocks": clocks,
    }
    del res
    torch.cuda.empty_cache()
    timer = Timer(dev, flush)
    if not args.no_configs:
        t0 = time.perf_counter()
        line["perf_test_like"] = perf_test_like(dev)
        line["configs"] = run_configs(dev, peak, timer)
        line["configs_seconds"] = time.perf_counter() - t0
        line["configs_parity_all_bit_exact"] = all(r.get("parity") == "bit-exact" for r in line["configs"]) and parity["parity"] == "bit-exact"
    os.sched_setaffinity(0, all_cpus)          # the CPU baseline uses every host core
    val, cores, sample, secs = cpu_closest(v, f, np.array([[0.0, 0.0, 3.0]], np.float32), d.reshape(-1, 3).cpu().numpy(), sample=8_294_400, reps=2)
    line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "seconds": secs,
                            "what": "oracle port: binary32 mirror behind a scalar binned-SAH BVH2 with double-precision boxes, OpenMP over rays - a stated baseline, not an Embree-class tracer"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------- GPU arm, N > 1 (config 5)
def run_b200_multi(args, dev, world, rank, local_rank):
    import torch.distributed as dist

    from triro import synth
    from triro.backend import ops as hops
    from triro.distributed import PeerOutputs, PeerPacked, ShardedRayMeshIntersector, all_counts, bind_to_device_cpus, gather_fixed

    all_cpus = os.sched_getaffinity(0)
    if not os.environ.get("TRIRO_BENCH_NO_BIND"):
        bind_to_device_cpus(local_rank)
    dist.init_process_group("nccl", device_id=dev)
    v, f = synth.heightfield(*CFG5_GRID)               # every rank holds the mesh description; only rank 0 builds
    vt, ft = torch.from_numpy(v), torch.from_numpy(f)
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    sh = ShardedRayMeshIntersector.build(vt, ft, src=0)
    torch.cuda.synchronize(); dist.barrier()
    build_bcast_ms = (time.perf_counter() - t0) * 1e3      # includes the H2D upload of the mesh on rank 0
    build_ms = build_timed(vt, ft, dev) if rank == 0 else None
    blob = sh.local.as_wrapper._inner.used()
    bts = []
    for _ in range(3):
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); dist.broadcast(blob, src=0); e1.record(); torch.cuda.synchronize()
        bts.append(e0.elapsed_time(e1))
    bcast_ms = min(bts[1:])
    r = sh.local
    n = CFG5_RAYS_PER_GPU if not args.rays_per_gpu else args.rays_per_gpu
    o, d = config5_rays(n, 100 + rank, dev)
    stats = hops.trace_stats(r.as_wrapper, o, d, "closest")
    steps, warm = args.steps, max(args.warmup, 3)

    def one_step():
        return r.intersects_closest(o, d, stream_compaction=True)

    # solo: this rank alone, no cross-rank synchronisation (what N = 1 gives on the same per-GPU workload)
    solo = []
    for i in range(warm + 3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); res = one_step(); e1.record(); torch.cuda.synchronize()
        if i >= warm:
            solo.append(e0.elapsed_time(e1))
        del res
    torch.cuda.synchronize(); dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ClockSampler(local_rank) as clk:
        for a, b in ev:
            a.record()
            res = one_step()
            b.record()
            if a is not ev[-1][0]:
                del res
        torch.cuda.synchronize()
    dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    hit, front, ray_idx, tri_idx, loc, uv = res
    n_hit_local = int(ray_idx.shape[0])

    def whole(fn, reps=3):
        ts, out = [], None
        for _ in range(reps):
            out = None
            torch.cuda.synchronize(); dist.barrier()
            t0 = time.perf_counter(); out = fn(); torch.cuda.synchronize(); dist.barrier()
            ts.append((time.perf_counter() - t0) * 1e3)
        t = torch.tensor([min(ts[1:])], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), out

    # (a) gathered, peer route: every rank traces + packs its slice, then copies its packed rows into rank 0's
    #     symmetric-memory tensors at its global row offset over NVLink (no NCCL on the data path)
    counts = all_counts(n_hit_local, dev)
    hits_total = sum(counts)
    base = rank * n
    rb = 8 if world * n > 2**31 - 1 else 4
    packed = PeerPacked(1 << max(hits_total - 1, 1).bit_length(), world * n, dev)

    def gathered_peer():
        h_, f_, t_, l_, u_ = hops.intersects_closest(r.as_wrapper, o, d)
        ws, total = hops.compact_scan(h_)
        mine = dict(front=torch.empty(total, dtype=torch.uint8, device=dev), ray=torch.empty(total, dtype=torch.int64 if rb == 8 else torch.int32, device=dev),
                    tri=torch.empty(total, dtype=torch.int32, device=dev), loc=torch.empty(3 * total, dtype=torch.float32, device=dev),
                    uv=torch.empty(2 * total, dtype=torch.float32, device=dev))
        hops.compact_scatter_at(h_, ws, f_, t_, l_, u_, base, rb, mine["front"].data_ptr(), mine["ray"].data_ptr(),
                                mine["tri"].data_ptr(), mine["loc"].data_ptr(), mine["uv"].data_ptr())
        cs = all_counts(total, dev)
        row0 = sum(cs[:rank])
        for name, t in mine.items():
            packed.peer_rows(0, name, row0, total, rb).copy_(t)
        packed.peer_hit_mask(0, base, base + n).copy_(h_.view(torch.uint8))
        return sum(cs)

    del res, hit, front, tri_idx, loc, uv
    t_peer, h_peer = whole(gathered_peer)
    ok_peer = True
    if rank == 0:
        vws = packed.local_views(h_peer, rb, (world * n,))
        ok_peer = h_peer == hits_total and bool((vws["ray"][1:] > vws["ray"][:-1]).all()) and int(vws["hit"].sum()) == h_peer
        ok_peer = ok_peer and bool(torch.equal(vws["ray"][:n_hit_local].to(torch.int64), ray_idx.to(torch.int64)))
        del vws

    # (b) gathered, NCCL route: padded all_gather of every array to every rank
    def gathered_nccl():
        r6 = r.intersects_closest(o, d, stream_compaction=True)
        cs = all_counts(r6[2].shape[0], dev)
        outs = [gather_fixed(r6[0], [n] * world)]
        for i, x in enumerate(r6[1:]):
            outs.append(gather_fixed(x.long() + base if i == 1 else x, cs))
        return int(outs[2].shape[0])

    t_nccl, h_nccl = whole(gathered_nccl)
    del packed
    torch.cuda.empty_cache()

    # (c) strong scaling: ONE 66 M-ray batch (replicated description), each rank traces its window, the dense 5-tuple
    #     lands on rank 0 (kernel peer stores for 2 ranks, bulk peer copies beyond)
    os_, ds_ = config5_rays(STRONG_RAYS, 7, dev)
    outs = PeerOutputs(STRONG_RAYS, dev)
    t_strong, _ = whole(lambda: sh.intersects_closest_to_root(os_, ds_, root=0, outputs=outs))
    strong_local = None
    if rank == 0:
        ms1, _ = Timer(dev)(lambda: r.intersects_closest(os_, ds_), reps=2, warm=1)
        strong_local = ms1
    del outs, os_, ds_
    torch.cuda.empty_cache()

    # (d) end to end with HOST buffers: every rank feeds a bounded sample of its slice (the first 25 M rays) from pinned host
    #     memory through rt_host_trace_closest_compact (H2D of 24 B/ray, trace, compaction on the device, D2H of the hit
    #     mask + packed rows); the ranks share the box's PCIe / host-memory bandwidth
    m_e2e = min(n, E2E_RAYS_PER_GPU)
    o_h = o[:m_e2e].cpu().pin_memory(); d_h = d[:m_e2e].cpu().pin_memory()
    outc = hops.host_closest(r.as_wrapper, o_h, d_h, stream_compaction=True)
    e2e_steps = 3
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        outc = hops.host_closest(r.as_wrapper, o_h, d_h, out=outc, stream_compaction=True)
    e2e_ms_local = (time.perf_counter() - t0) * 1e3
    e2e_hits = outc["n_hit"]
    del outc, o_h, d_h

    t = torch.tensor([total_ms, statistics.mean(solo), e2e_ms_local], dtype=torch.float64, device=dev)
    tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms, solo_ms_max, e2e_ms = float(tmax[0]), float(tmax[1]), float(tmax[2])
    if rank == 0:
        peak, peak_src = measured_peaks()
        hf = n_hit_local / n
        bpr = bytes_per_ray(stats, 24.0, 26.0 + 1.0 + 29.0 * hf)
        ms_per_step = total_ms / steps
        value = world * n * steps / (total_ms * 1e-3) / 1e6
        kernel_ms = statistics.mean(step_ms)
        # parity of rank 0's slice: 1 M rays against the oracle on the true-size mesh
        os.sched_setaffinity(0, all_cpus)
        oracle, cores = oracle_all_cores()
        parity = None
        if not args.no_configs:
            om = oracle.OracleMesh(v, f, use_bvh=True)
            sub = slice(0, PARITY_RAYS)
            dense = r.intersects_closest(o[sub], d[sub])
            parity = parity_closest(om, dense, o[sub], d[sub])
            k = int((ray_idx < PARITY_RAYS).sum())
            parity["compacted_ray_idx_ok"] = bool(torch.equal(ray_idx[:k].long(), torch.nonzero(dense[0]).reshape(-1)))
            del om, dense
        gathered_bytes = hits_total * (29 + (rb - 4)) + world * n
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD5, "rays_per_gpu": n, "rays_total": world * n,
                       "l2": "no flush: a step reads 3 GB of rays and a 1 GB blob, far beyond the 126 MB L2",
                       "parallelism": f"ray-sharded x{world}: BVH built on rank 0 and NCCL-broadcast, contiguous ray slices, results stay sharded in `value`, gathered on rank 0 in `gathered`",
                       "note": "N > 1 runs north_star's multi-GPU job (config 5); the N = 1 line's headline is config 2 - its counterpart of this `value` is configs['5 slice'] there and `weak_scaling.per_gpu_solo_mrays_s` here"},
            "parity": parity,
            "bvh_build_ms": build_ms, "bvh_broadcast_ms": bcast_ms, "bvh_broadcast_gb_s": blob.numel() / bcast_ms / 1e6,
            "bvh_blob_mb": blob.numel() / 1e6, "bvh_upload_build_broadcast_wall_ms": build_bcast_ms,
            "weak_scaling": {"per_gpu_solo_mrays_s": n / solo_ms_max / 1e3, "efficiency_vs_solo": value / (world * n / solo_ms_max / 1e3),
                             "what": "solo = the slowest rank's own time for the same step with no cross-rank barrier"},
            "gathered": {"what": "whole call intersects_closest(stream_compaction=True) of all ranks' rays with the complete 6-tuple assembled on rank 0",
                         "hits_total": hits_total, "bytes_into_root": gathered_bytes,
                         "peer_copies": {"ms": t_peer, "mrays_s": world * n / t_peer / 1e3, "verified": ok_peer,
                                         "route": "trace + scan + pack locally, exchange totals (one int64 each), bulk peer-to-peer copies into rank 0's symmetric-memory tensors at the global row offset"},
                         "nccl_all_gather": {"ms": t_nccl, "mrays_s": world * n / t_nccl / 1e3, "hits": h_nccl,
                                             "route": "padded all_gather_into_tensor of every array to every rank (gather_fixed)"},
                         "transfer_ms_estimate": max(t_peer - kernel_ms, 0.0),
                         "root_nvlink_ingress_gb_s": (gathered_bytes * (world - 1) / world / 1e9) / max((t_peer - kernel_ms) * 1e-3, 1e-9),
                         "limiter": "root NVLink ingress: all packed rows of the other ranks enter one GPU (900 GB/s per direction)"},
            "strong": {"what": f"ONE {STRONG_RAYS}-ray batch on the same mesh split {world} ways, dense 5-tuple assembled on rank 0 (intersects_closest_to_root)",
                       "ms": t_strong, "mrays_s": STRONG_RAYS / t_strong / 1e3, "one_gpu_ms": strong_local,
                       "speedup_vs_one_gpu": strong_local / t_strong if strong_local else None,
                       "bytes_into_root": 26 * STRONG_RAYS * (world - 1) // world},
            "roofline": {"bound": "hbm", "achieved": bpr * n / (kernel_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bpr * n / (kernel_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "kernel": "k_trace_coop<closest> + scan + scatter (one step)", "bytes_per_ray": bpr,
                         "nodes_per_ray": stats["nodes_per_ray"], "tris_per_ray": stats["tris_per_ray"], "hit_fraction": hf, "kernel_ms": kernel_ms},
            "e2e": {"value": world * m_e2e * e2e_steps / (e2e_ms * 1e-3) / 1e6, "unit": UNIT,
                    "h2d_bytes_per_step": 24 * m_e2e * world, "d2h_bytes_per_step": (m_e2e + 29 * e2e_hits) * world,
                    "sample": f"the first {m_e2e} rays of every rank's 125M-ray slice per step (pinned host buffers, bounded so that {world} ranks pin < 12 GB of host memory)",
                    "api": "rt_host_trace_closest_compact on every rank (pinned host rays in; hit mask + packed rows out); max over ranks of the wall time"},
            "gpu_launches": steps * world * 3, "clocks": clk.summary(),
            "nccl": {"version": ".".join(str(x) for x in torch.cuda.nccl.version()), "debug_env": os.environ.get("NCCL_DEBUG")},
        }
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        run_b200_multi(args, dev, world, rank, local_rank)
    else:
        run_b200_single(args, dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block and the oracle parity checks (quick runs, ncu)")
    ap.add_argument("--rays-per-gpu", type=int, default=0, help="N > 1 only: override config 5's 125 M rays per GPU (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1 only: write the last timed step's results (seeded sample) "
                                                          "to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "b200" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1:
            ap.error("--dump-outputs is implemented for the CUDA path with --gpus 1")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
