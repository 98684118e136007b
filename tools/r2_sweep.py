"""Round-2 schedule sweep on ONE GPU: every traversal schedule (direct = round 1, coop_coherent /
coop_incoherent = warp-cooperative triangle tests) x pair-list threshold on the BASELINE scenes, with a
bit-equality check between schedules, the nodes / triangles fetched per ray and the roofline fraction.

usage: python tools/r2_sweep.py [tag] [scenes, comma separated] [quick]
writes gpurun_out/<tag>_sweep.json
"""
import json, os, statistics, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "trimesh-ray-optix_b200")); sys.path.insert(0, ROOT)
import torch
from triro import synth
from triro.ray.ray_optix import RayMeshIntersector
from triro.backend import ops as hops

tag = sys.argv[1] if len(sys.argv) > 1 else "r2"
scenes = sys.argv[2].split(",") if len(sys.argv) > 2 else ["config2", "ico8", "hf4m", "soup1m", "hf16m", "small"]
dev = torch.device("cuda:0")
PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
rows = []
NAMES = {0: "auto", 1: "direct", 3: "coop_coherent", 4: "coop_incoherent"}


def timed(fn, reps=5, warm=2):
    ts = []
    for i in range(warm + reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        if i >= warm:
            ts.append(e0.elapsed_time(e1))
    return min(ts), statistics.median(ts), out


def scene(name):
    if name == "config2":
        v, f = synth.icosphere(7); o, d = synth.pinhole_rays(3840, 2160, device=dev); coherent = True
    elif name == "ico8":
        v, f = synth.icosphere(8); o, d = synth.pinhole_rays(3840, 2160, device=dev); coherent = True
    elif name == "hf4m":
        v, f = synth.heightfield(2048, 1024); o, d = synth.random_rays(20_000_000, seed=1234, device=dev); coherent = False
    elif name == "soup1m":
        v, f = synth.triangle_soup(1_000_000); o, d = synth.random_rays(10_000_000, seed=9, device=dev, box=True); coherent = False
    elif name == "hf16m":
        v, f = synth.heightfield(4096, 2048); o, d = synth.random_rays(30_000_000, seed=100, device=dev); coherent = False
    elif name == "small":      # the reference's own benchmark shape (test/performance_test.py:29-60): 640x360 rays per call
        v, f = synth.icosphere(7); o, d = synth.pinhole_rays(640, 360, device=dev); coherent = True
    else:
        raise SystemExit(name)
    return v, f, o, d, coherent


for name in scenes:
    v, f, o, d, coherent = scene(name)
    r = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    h = r.as_wrapper.header
    n = d.numel() // 3
    b_in = 12 if coherent else 24
    queries = [("closest", r.intersects_closest, 26, "closest")]
    if name in ("hf4m", "soup1m"):
        queries += [("any", r.intersects_any, 1, "any"), ("count", r.intersects_count, 4, "count")]
    base = {}
    for qname, fn, b_out, smode in queries:
        for sched in [int(x) for x in os.environ.get("SWEEP_SCHEDS", "1,3,4").split(",")]:
            thrs = [0] if sched == 1 else ([8, 16, 24, 32, 64] if sched == 3 else [16, 32, 64, 96])
            if os.environ.get("SWEEP_THRS"):
                thrs = [int(x) for x in os.environ["SWEEP_THRS"].split(",")] if sched != 1 else [0]
            if sched in (1, 3) and not coherent and name != "soup1m":
                thrs = thrs[:1]          # late re-fill on incoherent batches: one point is enough
            if sched == 4 and coherent and name == "small":
                thrs = thrs[:1]
            refills = [int(x) for x in os.environ.get("SWEEP_REFILL", "0").split(",")] if sched >= 3 else [0]
            for thr, refill in [(t, rf) for t in thrs for rf in refills]:
                old = hops.set_knobs(schedule=sched, tri_threshold=thr, refill_threshold=refill)
                try:
                    st = hops.trace_stats(r.as_wrapper, o, d, smode)
                    ms, med, out = timed(lambda: fn(o, d))
                finally:
                    hops.set_knobs(**old)
                res = out if isinstance(out, tuple) else (out,)
                if qname not in base:
                    base[qname] = tuple(x.clone() for x in res)
                    same = True
                else:
                    same = all(torch.equal(a, b) for a, b in zip(res, base[qname]))
                bpr = b_in + b_out + 80 * st["nodes_per_ray"] + 48 * st["tris_per_ray"]
                row = dict(scene=name, query=qname, schedule=NAMES[sched], tri_threshold=thr, refill_threshold=refill, tris=h["n_tris"], rays=n, ms=ms, ms_median=med,
                           mrays_s=n / ms / 1e3, nodes_per_ray=st["nodes_per_ray"], tris_per_ray=st["tris_per_ray"], bytes_per_ray=bpr,
                           frac=bpr * n / (ms * 1e-3) / (PEAK * 1e9), identical_to_first=same)
                rows.append(row)
                print(json.dumps(row), flush=True)
                assert same, "schedules disagree"
    if name == "small":
        # wall-clock per call of the reference's loop (no sync inside), default schedule
        for sched in (1, 0):
            old = hops.set_knobs(schedule=sched)
            for _ in range(200):
                r.intersects_closest(o, d)
            torch.cuda.synchronize(); t0 = time.time()
            for _ in range(5000):
                r.intersects_closest(o, d)
            torch.cuda.synchronize(); dt = time.time() - t0
            hops.set_knobs(**old)
            row = dict(scene=name, query="perf_test_like loop", schedule=NAMES.get(sched, "auto"), us_per_call=dt / 5000 * 1e6)
            rows.append(row); print(json.dumps(row), flush=True)
    del r, o, d
    torch.cuda.empty_cache()

os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(dict(peak_hbm_gbs=PEAK, lib=os.environ.get("TRIRO_B200_LIB", "default"), rows=rows),
          open(os.path.join(ROOT, "gpurun_out", f"{tag}_sweep.json"), "w"), indent=1)
