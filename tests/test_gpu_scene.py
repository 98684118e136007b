"""Instanced scenes on the GPU (rt_scene_prepare, rt_scene_trace, RayMeshScene): the prepared table and every query
against the host simulator of rt_scene.cuh bit for bit, dense and compacted, over batch layouts, windows and a user
tmax; one identity instance against RayMeshIntersector; the scene against a RayMeshIntersector of the flattened
geometry; update() after new transforms and after a member's refit, the stale-member error, empty scenes, input
validation and repeatability."""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "scene"))
import scene as sc  # noqa: E402
import scene_cases as cases  # noqa: E402
from helpers import assert_bits_equal  # noqa: E402
from oracle import oracle  # noqa: E402
from triro.backend import ops as hops  # noqa: E402
from triro.ray.ray_optix import RayMeshIntersector  # noqa: E402
from triro.ray.scene import RayMeshScene  # noqa: E402

pytestmark = pytest.mark.gpu


def make(v, f):
    return RayMeshIntersector(vertices=torch.from_numpy(np.ascontiguousarray(v)), faces=torch.from_numpy(np.ascontiguousarray(f)))


def sim_of(scene: RayMeshScene) -> sc.SimScene:
    """the host simulator over the scene's own GPU blobs, copied to the host"""
    return sc.SimScene([m.as_wrapper.blob.cpu().numpy() for m in scene.meshes], scene.instance_mesh.numpy(),
                       scene.transforms.numpy())


def np_closest(res):
    hit, front, inst, tri, loc, uv = res
    return dict(hit=hit.cpu().numpy().reshape(-1).astype(np.uint8), front=front.cpu().numpy().reshape(-1).astype(np.uint8),
                inst=inst.cpu().numpy().reshape(-1), tri=tri.cpu().numpy().reshape(-1), loc=loc.cpu().numpy().reshape(-1, 3),
                uv=uv.cpu().numpy().reshape(-1, 2))


def check_all_modes(scene, sim, o, d, what, tmax=1.0e7):
    """closest (dense and compacted), any and count of the scene against the simulator on the flattened batch"""
    on, dn = o.reshape(-1, 3).cpu().numpy(), d.reshape(-1, 3).cpu().numpy()
    ref = sim.trace("closest", on, dn, tmax=tmax)
    got = np_closest(scene.intersects_closest(o, d))
    for k in ref:
        assert_bits_equal(got[k], ref[k], f"{what}: closest.{k}")
    hit, front_c, ray_idx, inst_c, tri_c, loc_c, uv_c = scene.intersects_closest(o, d, stream_compaction=True)
    rows = np.nonzero(ref["hit"])[0]
    assert_bits_equal(ray_idx.cpu().numpy(), rows.astype(np.int32), f"{what}: ray_idx")
    for k, g in (("front", front_c), ("inst", inst_c), ("tri", tri_c), ("loc", loc_c), ("uv", uv_c)):
        gn = g.cpu().numpy()
        assert_bits_equal(gn.astype(ref[k].dtype) if k == "front" else gn, ref[k][rows], f"{what}: compacted {k}")
    assert_bits_equal(scene.intersects_any(o, d).cpu().numpy().reshape(-1).astype(np.uint8),
                      sim.trace("any", on, dn, tmax=tmax)["hit"], f"{what}: any")
    assert_bits_equal(scene.intersects_count(o, d).cpu().numpy().reshape(-1), sim.trace("count", on, dn, tmax=tmax)["count"],
                      f"{what}: count")
    return ref


@pytest.fixture(scope="module")
def big(cuda_device):
    ms, inst_mesh, t = cases.scene(300, seed=0)
    scene = RayMeshScene([make(v, f) for v, f in ms], torch.from_numpy(inst_mesh), torch.from_numpy(t))
    return scene, sim_of(scene)


def test_prepared_table_matches_sim(big):
    scene, sim = big
    n = scene.instance_mesh.numel()
    table = scene._table.cpu().numpy()
    off = int(table[16:24].view(np.uint64)[0])
    got = table[off:off + 128 * n].view(np.float32).reshape(n, 32)
    assert_bits_equal(got, sim.records(), "instance records")
    tv = scene._tlas.blob  # the top-level records hold (lo, hi, lo) of each instance
    hdr = scene._tlas.header
    recs = tv[hdr["tris_offset"]:hdr["tris_offset"] + 48 * n].cpu().numpy().view(np.float32).reshape(n, 12)
    prim = recs[:, 3].view(np.int32)
    assert sorted(prim.tolist()) == list(range(n))
    assert_bits_equal(recs[:, 0:3], sim.tlas_v[0::2][prim], "top-level lo")
    assert_bits_equal(recs[:, 4:7], sim.tlas_v[1::2][prim], "top-level hi")


@pytest.mark.parametrize("rays", ["random", "camera", "box"])
def test_kernels_match_sim(big, rays):
    scene, sim = big
    if rays == "random":
        o, d = cases.rays(20000, seed=1)
    elif rays == "camera":
        o, d = cases.camera_rays(160, 120)
    else:
        o, d = cases.box_rays(sim.blobs, scene.instance_mesh.numpy(), scene.transforms.numpy(), per_instance=24)
    ref = check_all_modes(scene, sim, torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), rays)
    assert ref["hit"].mean() > 0.05


def test_batch_layouts_windows_and_tmax(big):
    scene, sim = big
    o, d = cases.rays(4 * 6 * 50, seed=3)
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    check_all_modes(scene, sim, ot.reshape(2, 2, 6, 50, 3), dt.reshape(2, 2, 6, 50, 3), "5-d batch")
    big_o = torch.zeros((o.shape[0], 7), device="cuda")
    big_o[:, 2:5] = ot
    check_all_modes(scene, sim, big_o[:, 2:5], dt, "strided origins")
    cam = torch.tensor([0.0, -2.0, 14.0], device="cuda").expand(60, 40, 3)
    cd = torch.from_numpy(cases.camera_rays(40, 60)[1]).cuda().reshape(60, 40, 3)
    check_all_modes(scene, sim, cam, cd, "broadcast origin")
    check_all_modes(RayMeshScene(scene.meshes, scene.instance_mesh, scene.transforms, tmax=6.0), sim, ot, dt, "tmax 6",
                    tmax=6.0)
    ref = sim.trace("closest", o, d)
    for first, count in ((0, 100), (123, 457), (1000, -1)):
        got = np_closest(hops.scene_trace(scene._table, scene._tlas, ot, dt, hops.SCENE_CLOSEST, ray_first=first,
                                          ray_count=count))
        end = len(o) if count < 0 else first + count
        for k in ref:
            assert_bits_equal(got[k], ref[k][first:end], f"window {first}+{count}: {k}")


def test_identity_instance_equals_intersector(cuda_device):
    o, d = cases.rays(30000, seed=7, radius=1.5)
    o[::7] = 0.0
    d[::5, 0] = -0.0
    d[::11, 1] = 0.0
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    for v, f in cases.meshes()[:3]:
        r = make(v, f)
        scene = RayMeshScene([r], [0], torch.eye(4)[None])
        hit, front, inst, tri, loc, uv = scene.intersects_closest(ot, dt)
        rh, rf, rt_, rl, ru = r.intersects_closest(ot, dt)
        for g, e, k in ((hit, rh, "hit"), (front, rf, "front"), (tri, rt_, "tri"), (loc, rl, "loc"), (uv, ru, "uv")):
            assert_bits_equal(g.cpu().numpy(), e.cpu().numpy(), f"identity {k}")
        assert_bits_equal(inst.cpu().numpy(), torch.where(rh, 0, -1).int().cpu().numpy(), "identity inst")
        assert_bits_equal(scene.intersects_any(ot, dt).cpu().numpy(), r.intersects_any(ot, dt).cpu().numpy(), "identity any")
        assert_bits_equal(scene.intersects_count(ot, dt).cpu().numpy(), r.intersects_count(ot, dt).cpu().numpy(),
                          "identity count")


def test_agrees_with_flattened_intersector(cuda_device):
    ms, inst_mesh, t = cases.scene(80, seed=2, coincident=0)
    scene = RayMeshScene(ms, inst_mesh, t)
    fv, ff, fi, fr = sc.flatten(ms, inst_mesh, t)
    flat = make(fv, ff)
    mesh = oracle.OracleMesh(fv, ff)
    for o, d in (cases.rays(20000, seed=4), cases.camera_rays(128, 96)):
        ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
        g = np_closest(scene.intersects_closest(ot, dt))
        fh, _, ftri, floc, _ = (x.cpu().numpy() for x in flat.intersects_closest(ot, dt))
        clean = oracle.query(mesh, o, d, oracle.TRUTH, want=("flags",))["flags"] == 0
        assert (g["hit"].astype(bool)[clean] == fh[clean]).all()
        both = clean & fh
        assert (fi[ftri[both]] == g["inst"][both]).all() and (fr[ftri[both]] == g["tri"][both]).all()
        scale = max(1.0, float(np.abs(fv).max()))
        assert np.abs(g["loc"][both] - floc[both]).max() / scale <= 1e-5
        cnt = scene.intersects_count(ot, dt).cpu().numpy()
        assert (cnt[clean] == flat.intersects_count(ot, dt).cpu().numpy()[clean]).all()


def test_update_refit_and_stale_members(cuda_device):
    ms = cases.meshes()[:3]
    members = [make(v, f) for v, f in ms]
    inst_mesh = np.arange(30) % 3
    t = cases.random_transforms(30, seed=8)
    scene = RayMeshScene(members, inst_mesh, t)
    o, d = cases.rays(8000, seed=5)
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    before = np_closest(scene.intersects_closest(ot, dt))
    t2 = cases.random_transforms(30, seed=9)
    scene.update(torch.from_numpy(t2))
    check_all_modes(scene, sim_of(scene), ot, dt, "new transforms")
    assert not np.array_equal(np_closest(scene.intersects_closest(ot, dt))["inst"], before["inst"])
    v0 = torch.from_numpy(ms[0][0]).cuda() * 1.7
    members[0].refit(v0)
    with pytest.raises(RuntimeError, match="update"):
        scene.intersects_closest(ot, dt)
    with pytest.raises(RuntimeError, match="update"):
        scene.intersects_count(ot, dt)
    scene.update()
    ref = check_all_modes(scene, sim_of(scene), ot, dt, "after refit")
    assert ref["hit"].any()
    members[1].update_raw(torch.from_numpy(ms[1][0]).cuda(), torch.from_numpy(ms[1][1]).cuda())
    with pytest.raises(RuntimeError, match="update"):
        scene.intersects_any(ot, dt)
    scene.update()
    check_all_modes(scene, sim_of(scene), ot, dt, "after rebuild")


def test_empty_scene_and_empty_meshes(cuda_device):
    o, d = cases.rays(1000, seed=6)
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    for scene in (RayMeshScene([cases.meshes()[0]], np.zeros(0, np.int64), np.zeros((0, 3, 4), np.float32)),
                  RayMeshScene([cases.meshes()[3]], [0, 0], np.tile(np.eye(4, dtype=np.float32), (2, 1, 1)))):
        hit, front, inst, tri, loc, uv = scene.intersects_closest(ot, dt)
        assert not hit.any() and not front.any() and (inst == -1).all() and (tri == -1).all()
        assert not loc.any() and not uv.any()
        assert not scene.intersects_any(ot, dt).any() and not scene.intersects_count(ot, dt).any()
        res = scene.intersects_closest(ot, dt, stream_compaction=True)
        assert all(x.numel() == 0 for x in res[1:])
    scene = RayMeshScene([cases.meshes()[0]], [0], torch.eye(4)[None])
    e = torch.zeros((0, 3), device="cuda")
    assert scene.intersects_closest(e, e)[0].shape == (0,) and scene.intersects_count(e, e).shape == (0,)


def test_input_validation(cuda_device):
    v, f = cases.meshes()[0]
    good = np.eye(4, dtype=np.float32)[None, :3]
    inf = good.copy()
    inf[0, 1, 2] = np.inf
    for t in (np.zeros((1, 3, 4), np.float32), np.full((1, 3, 4), np.nan, np.float32), inf):
        with pytest.raises(ValueError):
            RayMeshScene([(v, f)], [0], t)
    bad_last = np.eye(4, dtype=np.float32)[None].copy()
    bad_last[0, 3, 0] = 1.0
    for mesh_idx, t in (([1], good), ([-1], good), ([0], bad_last), ([0, 0], good), ([0], good[:, :2])):
        with pytest.raises(ValueError):
            RayMeshScene([(v, f)], mesh_idx, t)
    scene = RayMeshScene([(v, f)], [0], good)
    o, d = cases.rays(10)
    with pytest.raises(ValueError):
        scene.intersects_closest(torch.from_numpy(o), torch.from_numpy(d))            # host rays
    with pytest.raises(ValueError):
        scene.intersects_any(torch.from_numpy(o).cuda().double(), torch.from_numpy(d).cuda().double())
    # the C entry point refuses what the wrapper would: host memory as a blob, a bad mesh index, a singular transform
    lib = hops.get_module()
    tb = C.c_size_t()
    assert lib.rt_scene_prepare_sizes(1, 1, C.byref(tb)) == 0
    table = torch.zeros(tb.value, dtype=torch.uint8, device="cuda")
    tv = torch.zeros((2, 3), device="cuda"); tf = torch.zeros((1, 3), dtype=torch.int32, device="cuda")
    host_blob = torch.zeros(1024, dtype=torch.uint8)
    dev_blob = scene.meshes[0].as_wrapper.blob
    mesh0 = np.zeros(1, np.int32); mesh1 = np.ones(1, np.int32)
    sing = np.zeros((1, 3, 4), np.float32)
    st = torch.cuda.current_stream().cuda_stream
    for blob, m, t in ((host_blob, mesh0, good), (dev_blob, mesh1, good), (dev_blob, mesh0, sing)):
        addrs = (C.c_void_p * 1)(blob.data_ptr())
        tt = np.ascontiguousarray(t, dtype=np.float32)
        rc = lib.rt_scene_prepare(1, addrs, 1, m.ctypes.data_as(C.c_void_p), tt.ctypes.data_as(C.c_void_p), hops._ptr(table),
                                  table.numel(), hops._ptr(tv), hops._ptr(tf), st)
        assert rc == -1, lib.rt_last_error()
    assert not table.any(), "a refused prepare wrote the table"


def test_mesh_kinds_and_repeatability(cuda_device):
    class Obj:
        def __init__(self, v, f):
            self.vertices, self.faces = v, f

    v, f = cases.meshes()[0]
    v2, f2 = cases.meshes()[2]
    t = cases.random_transforms(50, seed=12)
    inst_mesh = np.arange(50) % 3
    scene = RayMeshScene([make(v, f), (v2, f2), Obj(v, f)], inst_mesh, np.concatenate(
        [t, np.tile(np.array([[[0, 0, 0, 1]]], np.float32), (50, 1, 1))], axis=1))
    o, d = cases.rays(50000, seed=13)
    ot, dt = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    a = np_closest(scene.intersects_closest(ot, dt))
    for _ in range(3):
        b = np_closest(scene.intersects_closest(ot, dt))
        for k in a:
            assert_bits_equal(a[k], b[k], f"repeat {k}")
    check_all_modes(scene, sim_of(scene), ot, dt, "mesh kinds")
    hit = a["hit"].astype(bool)
    # uv interpolate on the instance's mesh gives the object-space hit point; mapped to the world it is loc
    m0 = hit & (inst_mesh[np.maximum(a["inst"], 0)] == 0)
    attr = scene.meshes[0].interpolate(scene.meshes[0].mesh_vertices, torch.from_numpy(a["tri"][m0]).cuda(),
                                       torch.from_numpy(a["uv"][m0]).cuda()).cpu().numpy().astype(np.float64)
    tt = t[a["inst"][m0]].astype(np.float64)
    world = np.einsum("nij,nj->ni", tt[:, :, :3], attr) + tt[:, :, 3]
    assert np.abs(world - a["loc"][m0]).max() <= 1e-4 * max(1.0, np.abs(world).max())
