"""RayMeshScene — closest, any and count ray queries against many instances of meshes, each instance with its own
affine transform, in one launch (the instance acceleration structures of OptiX, which the reference never exposed).

Point queries: `closest_point` and the pseudo-normal `signed_distance` over every instance in one launch (DESIGN.md
§4.12).

Gradients (DESIGN.md §4.13): `intersects_closest`'s `loc` and `uv` with respect to the rays, and the point queries'
distance and signed value with respect to the points, are also differentiable with respect to the transforms last
given to `update()` and every member's `mesh_vertices`, so poses can be fitted to point clouds or depth images
without flattening the scene.

Out of scope: gradients with respect to tmax or max_distance, visibility (edge) gradients, all-hits
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
    then.  No all-hits or containment queries (see the module docstring).

    Gradients: when `transforms` is a tensor that requires grad, the scene keeps a differentiable handle on it (the
    [:, :3, :] view of a 4x4, as float32), and the closest hit and the point queries return gradients to it in its own
    shape, dtype and device (a 4x4's last row gets 0).  Every member's `mesh_vertices` is an autograd input too.  A
    query's backward uses the table and the member tensors as of that query, so a backward after `update()` still
    differentiates the pose the forward saw.  After an in-place change of grad-requiring transforms (an optimiser
    step) call `update(transforms)` again: a query raises until then, rather than differentiate a pose the scene does
    not show.
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
        self._transforms_src = None      # what update() was last given (the autograd input), and its version
        self._transforms_version = 0
        self._member_table = None        # (key, device table, total vertex count), see _grad_members()
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
        if transforms is not None:
            src = transforms if isinstance(transforms, torch.Tensor) else None
            self._transforms_src, self._transforms_version = src, (src._version if src is not None else 0)
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
        src = self._transforms_src
        if src is not None and src.requires_grad and src._version != self._transforms_version:
            raise RuntimeError("the transforms given to update() were modified in place since (an optimiser step?): "
                               "call scene.update(transforms) so that the scene shows the pose being differentiated")

    # ------------------------------------------------------------------ gradients (DESIGN.md §4.13)
    def _transforms_handle(self):
        """The float32 [I,3,4] autograd handle of the transforms last given to update(), or None when they do not
        require grad.  Its values are those of the table (_check_current guards the version)."""
        src = self._transforms_src
        if src is None or not src.requires_grad or not torch.is_grad_enabled():
            return None
        return (src[:, :3, :] if src.shape[1] == 4 else src).to(torch.float32)

    def _vertices(self) -> list:
        return [m.mesh_vertices for m in self.meshes]

    def _tracks_grad(self, *tensors) -> bool:
        src = self._transforms_src
        return torch.is_grad_enabled() and (any(t.requires_grad for t in tensors)
                                            or (src is not None and src.requires_grad)
                                            or any(v.requires_grad for v in self._vertices()))

    def _grad_members(self):
        """(device member table, total vertex count, the member tensors it points to) for the current members; cached
        on the scene until a member's tensors change."""
        tensors = [(m.mesh_vertices.detach(), m.mesh_faces) for m in self.meshes]
        key = tuple((v.data_ptr(), v.shape[0], f.data_ptr(), f.shape[0]) for v, f in tensors)
        if self._member_table is None or self._member_table[0] != key:
            table, n_verts = hops.scene_members(tensors)
            self._member_table = (key, table, n_verts, tensors)
        return self._member_table[1:]

    def _trace(self, origins, directions, mode):
        self._check_current()
        return hops.scene_trace(self._table, self._tlas, origins, directions, mode, self.tmax)

    def intersects_closest(self, origins: torch.Tensor, directions: torch.Tensor, stream_compaction: bool = False):
        """Closest hit per ray over all instances.

        stream_compaction=False -> (hit[*b], front[*b], inst_idx[*b], tri_idx[*b], loc[*b,3], uv[*b,2])
        stream_compaction=True  -> (hit[*b], front[h], ray_idx[h], inst_idx[h], tri_idx[h], loc[h,3], uv[h,2])
        Misses: inst_idx = tri_idx = -1, loc and uv 0.

        `loc` and `uv` are differentiable with respect to `origins`, `directions`, the transforms last given to
        `update()` and every member's `mesh_vertices`: the gradient of the hit inside the visible triangle, recomputed
        on the world triangle A v + b of the forward's pose and vertices (DESIGN.md §4.13).  Visibility changes
        contribute nothing: a silhouette, an occlusion boundary or a hit that would move to another triangle or
        instance has no gradient.  Misses and degenerate triangles give 0.  `hit`, `front`, `ray_idx`, `inst_idx` and
        `tri_idx` are not differentiable.  Nothing of this runs unless grad mode is on and one of those requires grad;
        the gradients are deterministic to the bit."""
        if self._tracks_grad(origins, directions):
            return _SceneClosestHitFn.apply(self, stream_compaction, origins, directions, self._transforms_handle(),
                                            *self._vertices())
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

        `distance` is differentiable with respect to `points` ((p - closest) / distance, 0 where the distance is 0 or
        inf), the transforms last given to `update()` and every member's `mesh_vertices`: the gradient of the distance
        to the closest point, held at its triangle and barycentrics (DESIGN.md §4.13).  A closest point that would
        move to another triangle or instance contributes nothing beyond that."""
        self._check_current()
        md = float("inf") if max_distance is None else float(max_distance)
        side, _ = self._point_state(False)
        if self._tracks_grad(points):
            closest, distance, inst, tri, uv = _SceneClosestPointFn.apply(points, self, side, md,
                                                                          self._transforms_handle(), *self._vertices())
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

        Differentiable like `closest_point`'s distance, with respect to `points`, the transforms and every member's
        `mesh_vertices`; the sign is held."""
        if sign != "pseudonormal":
            raise ValueError(f'only sign="pseudonormal" is supported on scenes (got {sign!r})')
        self._check_current()
        side, normals = self._point_state(True)
        if self._tracks_grad(points):
            return _SceneSignedDistanceFn.apply(points, self, side, normals, self._transforms_handle(),
                                                *self._vertices())
        return hops.scene_signed_distance(self._table, self._tlas, side, normals, points)


def _save_scene(ctx, scene):
    """What the backward needs of the scene as of the forward: the table, the member table and its tensors."""
    ctx.table = scene._table
    ctx.n_inst = scene.instance_mesh.numel()
    ctx.members, ctx.n_verts, ctx.member_tensors = scene._grad_members()


def _split_vertices(ctx, gv, first: int):
    """grad_vertices [n_verts,3] as one gradient per member input (ctx.needs_input_grad[first:])"""
    out, base = [], 0
    for k, (v, _) in enumerate(ctx.member_tensors):
        n = v.shape[0]
        out.append(gv[base:base + n] if gv is not None and ctx.needs_input_grad[first + k] else None)
        base += n
    return out


def _transforms_grad(ctx, gt):
    """grad_transforms on the device of the transforms handle (autograd chains it back to what update() was given)"""
    return None if gt is None else gt.to(ctx.transforms_device)


def _scene_distance_backward(ctx, grad_value):
    """(grad_points, grad_transforms, grad_vertices per member) of a scene distance or signed distance; inputs
    (points, scene, side, extra, transforms, *vertices)"""
    points, value, closest, inst, tri, uv = ctx.saved_tensors
    need = ctx.needs_input_grad
    want_t, want_v = need[4], any(need[5:])
    if not want_t and not want_v:
        gp = hops.scene_distance_grad(points.detach(), grad_value, value, closest, tri, uv, ctx.n_faces)
        return gp, None, [None] * len(ctx.member_tensors)
    gp, gt, gv = hops.scene_point_grad(ctx.table, ctx.n_inst, ctx.members, ctx.n_verts, points.detach(), grad_value,
                                       value, closest, inst, tri, uv, points_grad=need[0], transforms_grad=want_t,
                                       vertices_grad=want_v)
    return gp, _transforms_grad(ctx, gt), _split_vertices(ctx, gv, 5)


def _save_point_forward(ctx, scene, transforms, points, value, closest, inst, tri, uv):
    ctx.save_for_backward(points, value, closest, inst, tri, uv)
    ctx.n_faces = scene._n_faces()
    ctx.transforms_device = None if transforms is None else transforms.device
    _save_scene(ctx, scene)


class _SceneClosestPointFn(torch.autograd.Function):
    """RayMeshScene.closest_point with a distance differentiable with respect to the points, the transforms handle
    and the members' vertices (DESIGN.md §4.13); those are only autograd inputs, the forward walks the scene."""

    @staticmethod
    def forward(ctx, points, scene, side, max_distance, transforms, *vertices):
        out = hops.scene_closest_point(scene._table, scene._tlas, side, points.detach(), max_distance)
        closest, distance, inst, tri, uv = out
        ctx.mark_non_differentiable(closest, inst, tri, uv)
        _save_point_forward(ctx, scene, transforms, points, distance, closest, inst, tri, uv)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_closest, grad_distance, grad_inst, grad_tri, grad_uv):
        gp, gt, gv = _scene_distance_backward(ctx, grad_distance)
        return gp, None, None, None, gt, *gv


class _SceneSignedDistanceFn(torch.autograd.Function):
    """RayMeshScene.signed_distance with its gradient with respect to the points, the transforms handle and the
    members' vertices: one walk gives the sign and the closest feature."""

    @staticmethod
    def forward(ctx, points, scene, side, normals, transforms, *vertices):
        sd, closest, inst, tri, uv = hops.scene_signed_distance(scene._table, scene._tlas, side, normals,
                                                                points.detach(), return_closest=True)
        _save_point_forward(ctx, scene, transforms, points, sd, closest, inst, tri, uv)
        return sd

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_sd):
        gp, gt, gv = _scene_distance_backward(ctx, grad_sd)
        return gp, None, None, None, gt, *gv


class _SceneClosestHitFn(torch.autograd.Function):
    """RayMeshScene.intersects_closest with differentiable loc and uv (DESIGN.md §4.13), dense or compacted; inputs
    (scene, compaction, origins, dirs, transforms handle or None, *member vertices)."""

    @staticmethod
    def forward(ctx, scene, compaction, origins, dirs, transforms, *vertices):
        hit, front, inst, tri, loc, uv = scene._trace(origins.detach(), dirs.detach(), hops.SCENE_CLOSEST)
        ray_idx = None
        if compaction:
            front, ray_idx, tri, loc, uv = hops.compact_closest(hit, front, tri, loc, uv)
            inst = inst.reshape(-1)[ray_idx.long()]
        ctx.mark_non_differentiable(*(t for t in (hit, front, ray_idx, inst, tri) if t is not None))
        ctx.save_for_backward(origins, dirs, inst, tri, ray_idx)
        ctx.transforms_device = None if transforms is None else transforms.device
        _save_scene(ctx, scene)
        if compaction:
            return hit, front, ray_idx, inst, tri, loc, uv
        return hit, front, inst, tri, loc, uv

    @staticmethod
    @once_differentiable
    def backward(ctx, *grads):
        origins, dirs, inst, tri, ray_idx = ctx.saved_tensors
        need = ctx.needs_input_grad
        h = tri.numel()
        grad_loc, grad_uv = grads[-2], grads[-1]
        go, gd, gt, gv = hops.scene_ray_grad(ctx.table, ctx.n_inst, ctx.members, ctx.n_verts, origins.detach(),
                                             dirs.detach(), inst.reshape(h), tri.reshape(h), grad_loc.reshape(h, 3),
                                             None if grad_uv is None else grad_uv.reshape(h, 2), ray_idx=ray_idx,
                                             origins_grad=need[2], directions_grad=need[3], transforms_grad=need[4],
                                             vertices_grad=any(need[5:]))
        return None, None, go, gd, _transforms_grad(ctx, gt), *_split_vertices(ctx, gv, 5)
