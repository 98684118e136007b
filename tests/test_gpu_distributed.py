"""GPU tier of the ray-sharding layer: torchrun with 2 ranks over NCCL (SKIPPED with a reason on a 1-GPU box, so that
a pass always means two ranks ran; a single-rank smoke of the same worker is a separate test).  Checks that (a) the gathered
N-rank result of ShardedRayMeshIntersector.intersects_closest and (b) the fused trace + gather
(intersects_closest_to_root: k_trace stores straight into the root's symmetric-memory tensors over NVLink) are
bit-identical to the oracle's MIRROR evaluator on the same rays, and (c) that the fused variable-length routes
(compacted closest hits, all hits: scatter kernels writing into the root's packed tensors) equal the NCCL gather."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
sys.path.insert(0, os.path.join(ROOT, "trimesh-ray-optix_b200")); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, torch.distributed as dist
from triro import synth
from triro.distributed import ShardedRayMeshIntersector, PeerOutputs
rank = int(os.environ["RANK"]); local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local); dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
v, f = synth.icosphere(4)
sh = ShardedRayMeshIntersector.build(torch.from_numpy(v), torch.from_numpy(f), src=0)
o, d = synth.readme_rays(301, device=dev)          # odd size: ragged slices
full = sh.intersects_closest(o, d, gather=True)
outs = PeerOutputs(o.numel() // 3, dev)
peer = sh.intersects_closest_to_root(o, d, root=0, outputs=outs, kernel_stores=True)
peer2 = sh.intersects_closest_to_root(o, d, root=0, outputs=outs)      # buffer reuse
if rank == 0:
    peer2 = tuple(x.clone() for x in peer2)
peer3 = sh.intersects_closest_to_root(o, d, root=0, outputs=outs, kernel_stores=False)     # peer-to-peer copies instead
if rank == 0:
    assert all(torch.equal(a, b) for a, b in zip(peer2, peer3))
peer4 = sh.intersects_closest_to_root(o, d, root=0, outputs=outs, kernel_stores=False, chunks=3)   # windows, copies on a side stream
if rank == 0:
    assert all(torch.equal(a, b) for a, b in zip(peer2, peer4))
assert (peer is None) == (rank != 0)
# variable-length results packed on the root by the ranks' own scatter kernels
comp_nccl = sh.intersects_closest(o, d, stream_compaction=True, gather=True)
comp_peer = sh.intersects_closest_compact_to_root(o, d, root=0)
comp_peer = sh.intersects_closest_compact_to_root(o, d, root=0, packed=sh.last_packed)       # buffer reuse
if rank == 0:
    comp_peer = tuple(x.clone() for x in comp_peer)
comp_peer_k = sh.intersects_closest_compact_to_root(o, d, root=0, packed=sh.last_packed, scatter_to_peer=True)
if rank == 0:
    for a, b in zip(comp_peer, comp_peer_k):
        assert torch.equal(a, b)
o2, d2 = synth.random_rays(50_001, seed=5, device=dev, box=True)
loc_nccl = sh.intersects_location(o2, d2, gather=True)
loc_peer = sh.intersects_location_to_root(o2, d2, root=0)
if rank == 0:
    for a, b in zip(comp_nccl, comp_peer):
        assert a.dtype == b.dtype and torch.equal(a, b), (a.shape, b.shape)
    for a, b in zip(loc_nccl, loc_peer):
        assert a.dtype == b.dtype and torch.equal(a, b), (a.shape, b.shape)
    assert loc_peer[0].shape[0] > 1000 and comp_peer[1].shape[0] == int(comp_peer[0].sum())
else:
    assert comp_peer is None and loc_peer is None
if rank == 0:
    from oracle import oracle
    om = oracle.OracleMesh(v, f)
    ref = oracle.query(om, np.broadcast_to(o.cpu().numpy(), d.shape).reshape(-1, 3), d.cpu().numpy().reshape(-1, 3), mode=oracle.MIRROR)
    for got in (full, peer, peer2):
        hit, front, tri, loc, uv = [x.cpu().numpy() for x in got]
        assert np.array_equal(hit.reshape(-1), ref["hit"].astype(bool)) and np.array_equal(tri.reshape(-1), ref["tri"])
        assert np.array_equal(front.reshape(-1), ref["front"].astype(bool))
        assert np.array_equal(loc.reshape(-1, 3).view(np.uint32), ref["loc"].astype(np.float32).view(np.uint32))
        assert np.array_equal(uv.reshape(-1, 2).view(np.uint32), ref["uv"].astype(np.float32).view(np.uint32))
    print("DIST_OK hits", int(ref["hit"].sum()), "world", dist.get_world_size())
# contains_points: the two whole-batch decisions are OR-reduced and the retry direction comes from rank 0, so the
# sharded answer equals the single-process one also in the retry / quirk branches (open mesh -> broken points)
from triro.ray.ray_optix import RayMeshIntersector
vo, fo = synth.icosphere(3)
sho = ShardedRayMeshIntersector.build(torch.from_numpy(vo), torch.from_numpy(fo[1:]), src=0)
pts = ((torch.rand((30_001, 3), generator=torch.Generator().manual_seed(5)) * 2 - 1) * 1.2).to(dev)
torch.manual_seed(4321 + rank)
if rank == 0:
    torch.manual_seed(99)
got_retry = sho.contains_points(pts)
got_quirk = sho.contains_points(pts, torch.tensor([0.3, 0.5, 0.8], device=dev))
single = RayMeshIntersector(vertices=torch.from_numpy(vo), faces=torch.from_numpy(fo[1:]))
torch.manual_seed(99)
assert torch.equal(got_retry, single.contains_points(pts)), "sharded contains (retry branch) differs from one process"
assert torch.equal(got_quirk, single.contains_points(pts, torch.tensor([0.3, 0.5, 0.8], device=dev)))
# an adopted (broadcast) blob re-fits like the original
if rank != 0:
    sho.local.as_wrapper._inner.refit(torch.from_numpy(vo * 1.1).to(dev), torch.from_numpy(fo[1:]).to(dev))
    assert bool(sho.local.intersects_any(torch.tensor([[0.0, 0.0, 3.0]], device=dev), torch.tensor([[0.0, 0.3, -1.0]], device=dev)))
dist.barrier()
if rank == 0:
    print("DIST_CONTAINS_OK")
dist.destroy_process_group()
'''


def _run(nproc, tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DIST_OK" in r.stdout and "DIST_CONTAINS_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    assert f"world {nproc}" in r.stdout


@pytest.mark.gpu
def test_sharded_closest_and_fused_peer_gather_match_the_oracle(cuda_device, tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs: peer stores / peer copies / NCCL gathers between two ranks; "
                    "the world-size-1 smoke below covers the code path on a one-GPU machine")
    _run(2, tmp_path)


@pytest.mark.gpu
def test_sharded_layer_single_rank_smoke(cuda_device, tmp_path):
    """The same worker with ONE rank: exercises symmetric memory, the to-root routes and the sharded contains flow
    where no second GPU exists.  Says nothing about inter-GPU traffic - the 2-rank test does."""
    _run(1, tmp_path)
