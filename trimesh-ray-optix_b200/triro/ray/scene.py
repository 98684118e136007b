"""RayMeshScene — closest, any and count ray queries against many instances of meshes, each instance with its own
affine transform, in one launch (the instance acceleration structures of OptiX, which the reference never exposed).

Point queries: `closest_point` and the pseudo-normal `signed_distance` over every instance in one launch, the
distance and the signed value differentiable with respect to the points (DESIGN.md §4.12).

Out of scope: ray gradients, gradients with respect to transforms or member vertices, all-hits
(`intersects_location` / `intersects_id`), `contains_points`, winding numbers and the winding or contains signs,
`triro.distributed` and the numpy adapter.  Query a member `RayMeshIntersector` for those.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

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
    then.  The ray queries are not differentiable; no all-hits or containment queries (see the module docstring).
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
        self._point_side = None        # built on the first point query (_point_state)
        self._normals = None
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

    # ------------------------------------------------------------------ point queries (DESIGN.md §4.12)
    def _point_state(self, signed: bool):
        """The side array of the point queries and, for the sign, the device table of the members' pseudo-normal
        addresses; built on first use, dropped by update().  The scene keeps the normals tensors it points to."""
        if self._point_side is None:
            self._point_side = hops.scene_point_prepare(self._table, self.instance_mesh.numel())
        if signed and self._normals is None:
            rows = [hops.pseudo_normals(m.as_wrapper)[0] for m in self.meshes]
            # a mesh without triangles has no rows: any aligned address will do, the kernel never reads it
            addrs = [r.data_ptr() if r.numel() else m.as_wrapper.blob.data_ptr() for r, m in zip(rows, self.meshes)]
            table = torch.tensor(addrs or [0], dtype=torch.int64).to(self.device)
            self._normals = (table, rows)
        return self._point_side, (self._normals[0] if signed else None)

    def _n_faces(self) -> int:
        return max([int(m.as_wrapper.header["n_tris"]) for m in self.meshes] + [0])

    def closest_point(self, points: torch.Tensor, max_distance=None, return_uv: bool = False):
        """(closest[*b,3], distance[*b], inst_idx[*b], triangle_id[*b][, uv[*b,2]]) — the nearest point of any
        instance for every query point.  The answer minimises (distance, instance, triangle) over every triangle of
        every instance within `max_distance` (None = unbounded), measured to the world triangle whose vertices are
        the binary32 images A v + b (the sequence `intersects_closest` uses for `loc`); so it equals, bit for bit,
        `RayMeshIntersector.closest_point` on the scene flattened with those vertices, faces in instance order.
        `triangle_id` is the row of the instance's mesh faces and uv the weights of its vertices 0 and 1 (barycentrics
        survive affine maps, so the mesh's `interpolate` works).  A point with nothing in reach gets inst_idx =
        triangle_id = -1, distance inf, closest and uv 0.

        `distance` is differentiable with respect to `points`: (p - closest) / distance, 0 where the distance is 0 or
        inf.  There is no gradient with respect to the transforms or the member vertices."""
        self._check_current()
        md = float("inf") if max_distance is None else float(max_distance)
        side, _ = self._point_state(False)
        if torch.is_grad_enabled() and points.requires_grad:
            closest, distance, inst, tri, uv = _SceneClosestPointFn.apply(points, self, side, md)
        else:
            closest, distance, inst, tri, uv = hops.scene_closest_point(self._table, self._tlas, side, points, md)
        if return_uv:
            return closest, distance, inst, tri, uv
        return closest, distance, inst, tri

    def signed_distance(self, points: torch.Tensor, sign: str = "pseudonormal") -> torch.Tensor:
        """Float32[*b] — distance to the nearest instance, positive inside: one walk per point, with the sign of the
        angle-weighted pseudo-normal of the closest feature (`RayMeshIntersector.signed_distance(sign="pseudonormal")`)
        carried to world space by A^-T, which keeps outward normals outward for every invertible A, mirrors
        included.  |value| is bit for bit `closest_point`'s distance; an exact 0 is +0; a point with no answer
        (non-finite, or an empty scene) gives -inf.  One identity instance reproduces its mesh's signed distance.

        The sign is inside/outside when every mesh is closed, manifold and consistently oriented, every transform is
        a similarity (rotation times uniform scale, mirrors allowed) and the instances do not overlap.  Under
        non-uniform scale or shear the vertex and edge pseudo-normals lose their equal weights and the sign may be
        wrong near those features; where instances overlap it is the sign of the closest feature's instance, not of
        the union.  It is always defined and deterministic.  Only sign="pseudonormal" exists on scenes.

        Differentiable with respect to `points` like `closest_point`'s distance; not with respect to the transforms
        or the member vertices."""
        if sign != "pseudonormal":
            raise ValueError(f'only sign="pseudonormal" is supported on scenes (got {sign!r})')
        self._check_current()
        side, normals = self._point_state(True)
        if torch.is_grad_enabled() and points.requires_grad:
            return _SceneSignedDistanceFn.apply(points, self, side, normals)
        return hops.scene_signed_distance(self._table, self._tlas, side, normals, points)


def _scene_distance_backward(ctx, grad_value):
    points, value, closest, tri, uv = ctx.saved_tensors
    return hops.scene_distance_grad(points.detach(), grad_value, value, closest, tri, uv, ctx.n_faces)


class _SceneClosestPointFn(torch.autograd.Function):
    """RayMeshScene.closest_point with a distance differentiable with respect to the points."""

    @staticmethod
    def forward(ctx, points, scene, side, max_distance):
        out = hops.scene_closest_point(scene._table, scene._tlas, side, points.detach(), max_distance)
        closest, distance, inst, tri, uv = out
        ctx.mark_non_differentiable(closest, inst, tri, uv)
        ctx.save_for_backward(points, distance, closest, tri, uv)
        ctx.n_faces = scene._n_faces()
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_closest, grad_distance, grad_inst, grad_tri, grad_uv):
        return _scene_distance_backward(ctx, grad_distance), None, None, None


class _SceneSignedDistanceFn(torch.autograd.Function):
    """RayMeshScene.signed_distance with its gradient with respect to the points: one walk gives the sign and the
    closest feature."""

    @staticmethod
    def forward(ctx, points, scene, side, normals):
        sd, closest, _, tri, uv = hops.scene_signed_distance(scene._table, scene._tlas, side, normals, points.detach(),
                                                             return_closest=True)
        ctx.save_for_backward(points, sd, closest, tri, uv)
        ctx.n_faces = scene._n_faces()
        return sd

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_sd):
        return _scene_distance_backward(ctx, grad_sd), None, None, None
