"""Small end-to-end run for compute-sanitizer (memcheck / racecheck): every kernel of the library on tiny inputs."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "trimesh-ray-optix_b200")); sys.path.insert(0, ROOT)
import torch
from triro import synth
from triro.ray.ray_optix import RayMeshIntersector
from triro.backend import ops as hops
dev = torch.device("cuda:0")
for sub, soup in ((3, False), (0, True)):
    v, f = synth.triangle_soup(3000, sigma=0.05, seed=1) if soup else synth.icosphere(sub)
    r = RayMeshIntersector(vertices=torch.from_numpy(v), faces=torch.from_numpy(f))
    o, d = synth.random_rays(5000, seed=3, device=dev, box=True)
    o = o * 1.5
    oc, dc = synth.readme_rays(64, device=dev)
    for sched in (0, 1, 3, 4):                  # AUTO + every explicit schedule (per-lane, cooperative)
        old = hops.set_knobs(schedule=sched)
        for (oo, dd) in ((o, d), (oc, dc)):
            r.intersects_closest(oo, dd, stream_compaction=True); r.intersects_any(oo, dd); r.intersects_first(oo, dd)
            r.intersects_count(oo, dd); r.intersects_location(oo, dd); r.intersects_id(oo, dd, multiple_hits=False)
            hops.trace_stats(r.as_wrapper, oo, dd, "closest")
        r.contains_points(o)
        hops.set_knobs(**old)
    hops.intersects_closest(r.as_wrapper, o, d, 100, 1000)           # ray window
    old = hops.set_knobs(no_lane_sharing=1)
    r.intersects_closest(o, d); r.intersects_count(o, d)
    hops.set_knobs(**old)
    hops.intersects_location(r.as_wrapper, o, d, 8, staging_bytes=1000 * 8 * 16)
    r.contains_points(o)
    r.refit(torch.from_numpy(v * 1.1))
    r.intersects_closest(o, d)
    out = hops.host_closest(r.as_wrapper, torch.tensor([0.0, 0.0, 3.0]).pin_memory(), dc.reshape(-1, 3).cpu().contiguous().pin_memory())
    out = hops.host_closest(r.as_wrapper, torch.tensor([0.0, 0.0, 3.0]).pin_memory(), dc.reshape(-1, 3).cpu().contiguous().pin_memory(),
                            stream_compaction=True)
k = torch.randint(0, 2**40, (70000,), device=dev); vv = torch.arange(70000, dtype=torch.int32, device=dev)
hops.sort_pairs_u64(k, vv)
torch.cuda.synchronize()
print("sanitize smoke done")
