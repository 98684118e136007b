"""RayMeshScene — closest, any and count ray queries against many instances of meshes, each instance with its own
affine transform, in one launch (the instance acceleration structures of OptiX, which the reference never exposed).

Out of scope: gradients, all-hits (`intersects_location` / `intersects_id`), `contains_points`, point queries
(closest point, signed distance, winding numbers), `triro.distributed` and the numpy adapter.  Query a member
`RayMeshIntersector` for those.
"""
from __future__ import annotations

import torch

import triro.backend.ops as hops
from triro.ray.ray_optix import RayMeshIntersector


class RayMeshScene:
    """A two-level scene: `meshes` are `RayMeshIntersector`s (used through their BVH blob, no rebuild), (vertices,
    faces) pairs or objects with `.vertices` / `.faces` (wrapped in a new intersector); instance i shows mesh
    `instance_mesh[i]` under the object->world transform `transforms[i]` ([I,3,4] or [I,4,4] with last row 0 0 0 1,
    any float dtype, rounded to float32).

    The world ray (o, d) meets instance i as o' = A^-1 (o - b), d' = A^-1 d with the same t, A^-1 computed in float64
    and rounded to float32 once per `update()`.  The closest hit minimises (t, instance, triangle) over every instance
    in (0, tmax), so ties at equal t go to the smaller instance, then the smaller triangle.  `tri_idx` is the row of
    the instance's mesh faces, `uv` are object-space weights of its vertices 0 and 1 (so the mesh's `interpolate`
    works), `loc` is the world point, and `front` is flipped for mirrored instances (det A < 0).  One identity instance
    gives exactly the results of its `RayMeshIntersector`.

    Culling uses padded world boxes; DESIGN.md §4.11 gives the padding and the ray origins (|o|inf at most 32 times
    the instance's reach from the world origin) for which it provably drops no hit.  The member intersectors are
    not watched: after `refit` or `update_raw` of a member, or new transforms, call `update()`; a query raises until
    then.  Not differentiable; no all-hits, containment or point queries (see the module docstring).
    """

    def __init__(self, meshes, instance_mesh, transforms, tmax: float = hops.TMAX_DEFAULT):
        self.tmax = float(tmax)
        if not (self.tmax > 0.0):
            raise ValueError("tmax must be positive")
        self.meshes = [self._wrap(m) for m in meshes]
        devs = {m.as_wrapper.blob.device for m in self.meshes}
        if len(devs) > 1:
            raise ValueError(f"the meshes of a scene must live on one device (got {sorted(str(d) for d in devs)})")
        self.device = devs.pop() if devs else torch.device("cuda", torch.cuda.current_device())
        self.instance_mesh = torch.as_tensor(instance_mesh).reshape(-1).to("cpu", torch.int64)
        self.transforms = None
        self.update(transforms)

    @staticmethod
    def _wrap(m) -> RayMeshIntersector:
        if isinstance(m, RayMeshIntersector):
            return m
        if isinstance(m, (tuple, list)) and len(m) == 2:
            return RayMeshIntersector(vertices=torch.as_tensor(m[0]), faces=torch.as_tensor(m[1]))
        return RayMeshIntersector(mesh=m)

    @staticmethod
    def _transforms(t, n: int) -> torch.Tensor:
        t = torch.as_tensor(t).detach().to("cpu", torch.float64)
        if t.dim() != 3 or t.shape[0] != n or tuple(t.shape[1:]) not in ((3, 4), (4, 4)):
            raise ValueError(f"transforms must be [{n},3,4] or [{n},4,4], got {tuple(t.shape)}")
        if t.shape[1] == 4:
            last = torch.tensor([0.0, 0.0, 0.0, 1.0], dtype=torch.float64)
            if not bool((t[:, 3, :] == last).all()):
                raise ValueError("the last row of a 4x4 transform must be 0 0 0 1")
            t = t[:, :3, :]
        t = t.to(torch.float32).contiguous()
        if not bool(torch.isfinite(t).all()):
            raise ValueError("transforms must be finite")
        return t

    def update(self, transforms=None):
        """Prepare the instances again (inverse transforms, world boxes) and rebuild the top-level tree, with new
        transforms when given.  The meshes' own trees are not touched: refit or rebuild them first."""
        n = self.instance_mesh.numel()
        t = self.transforms if transforms is None else self._transforms(transforms, n)
        if n and (int(self.instance_mesh.min()) < 0 or int(self.instance_mesh.max()) >= len(self.meshes)):
            raise ValueError(f"instance_mesh must index the {len(self.meshes)} meshes")
        blobs = [m.as_wrapper.blob for m in self.meshes]
        self._table, self._tlas = hops.scene_prepare(blobs, self.instance_mesh.to(torch.int32), t, self.device)
        self.transforms = t
        self._members = [(m.as_wrapper._inner.blob, m.as_wrapper._inner.generation) for m in self.meshes]
        return self

    def _check_current(self):
        for k, (m, (blob, gen)) in enumerate(zip(self.meshes, self._members)):
            inner = m.as_wrapper._inner
            if inner.blob is not blob or inner.generation != gen:
                raise RuntimeError(f"mesh {k} of the scene was rebuilt or re-fitted since the last update(): call "
                                   "scene.update() so that the instance boxes follow it")

    def _trace(self, origins, directions, mode):
        self._check_current()
        return hops.scene_trace(self._table, self._tlas, origins, directions, mode, self.tmax)

    def intersects_closest(self, origins: torch.Tensor, directions: torch.Tensor, stream_compaction: bool = False):
        """Closest hit per ray over all instances.

        stream_compaction=False -> (hit[*b], front[*b], inst_idx[*b], tri_idx[*b], loc[*b,3], uv[*b,2])
        stream_compaction=True  -> (hit[*b], front[h], ray_idx[h], inst_idx[h], tri_idx[h], loc[h,3], uv[h,2])
        Misses: inst_idx = tri_idx = -1, loc and uv 0."""
        hit, front, inst, tri, loc, uv = self._trace(origins, directions, hops.SCENE_CLOSEST)
        if stream_compaction:
            front_c, ray_idx, tri_c, loc_c, uv_c = hops.compact_closest(hit, front, tri, loc, uv)
            return hit, front_c, ray_idx, inst.reshape(-1)[ray_idx.long()], tri_c, loc_c, uv_c
        return hit, front, inst, tri, loc, uv

    def intersects_any(self, origins: torch.Tensor, directions: torch.Tensor) -> torch.Tensor:
        """Bool[*b] — does each ray hit any instance in (0, tmax)."""
        return self._trace(origins, directions, hops.SCENE_ANY)

    def intersects_count(self, origins: torch.Tensor, directions: torch.Tensor) -> torch.Tensor:
        """Int32[*b] — the sum over instances of the triangles each ray crosses in (0, tmax)."""
        return self._trace(origins, directions, hops.SCENE_COUNT)
