"""RayMeshIntersector — trimesh.ray-compatible façade over the B200 kernels.

Keeps the public surface of the reference class `triro.ray.ray_optix.RayMeshIntersector`
(reference triro/ray/ray_optix.py:18-279) verbatim: constructor keywords, attributes
(`mesh_vertices`, `mesh_faces`, `mesh_aabb`, `as_wrapper`), method names, argument order and
defaults, dtypes and tuple orders of the results.  What changed is underneath: one fused
kernel launch (plus a prefix-sum/scatter pair where a result is variable-length) per call
instead of OptiX launches glued together with torch indexing.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

import triro.backend.ops as hops


class RayMeshIntersector:
    """Ray/mesh queries against a static triangle mesh.

    Either ``mesh=`` (any object with ``.vertices`` / ``.faces`` array-likes, e.g. a
    ``trimesh.Trimesh``) or ``vertices=`` and ``faces=`` (torch tensors on any device) must be
    given (reference ray_optix.py:24-41).
    """

    def __init__(self, **kwargs):
        if "mesh" in kwargs:
            mesh = kwargs["mesh"]
            vertices = torch.as_tensor(mesh.vertices)
            faces = torch.as_tensor(mesh.faces)
        elif "vertices" in kwargs and "faces" in kwargs:
            vertices = kwargs["vertices"]
            faces = kwargs["faces"]
        else:
            raise ValueError("Either 'mesh' or 'vertices' and 'faces' must be provided.")
        # Extensions (SURVEY §8f): the reference hard-codes tmax = 1e7 (shaders.cu:86) and at most 8 hits per ray
        # (LaunchParams.h:8); both stay the defaults.
        self.tmax = float(kwargs.get("tmax", hops.TMAX_DEFAULT))
        self.max_hits = int(kwargs.get("max_hits", hops.MAX_ANYHIT_SIZE))
        if not (self.tmax > 0.0) or not (1 <= self.max_hits <= hops.MAX_HITS_LIMIT):
            raise ValueError(f"tmax must be positive and 1 <= max_hits <= {hops.MAX_HITS_LIMIT}")
        self.as_wrapper = OptixAccelStructureWrapper()
        self.as_wrapper._inner.tmax = self.tmax
        self.update_raw(vertices, faces)

    def update_raw(self, vertices: torch.Tensor, faces: torch.Tensor):
        """Replace the mesh and rebuild the acceleration structure (reference ray_optix.py:55-69)."""
        # [n, 3] float32 / [f, 3] int32 on the device: a CUDA input keeps its device, a host input goes to the
        # current one (the reference's `.cuda()`, ray_optix.py:57-58); both must end up on the same device
        self.mesh_vertices = vertices.float().contiguous()
        if not self.mesh_vertices.is_cuda:
            self.mesh_vertices = self.mesh_vertices.cuda()
        self.mesh_faces = faces.int().contiguous().to(self.mesh_vertices.device)
        if self.mesh_vertices.shape[0] > 0:
            self.mesh_aabb = (
                torch.min(self.mesh_vertices, dim=0)[0],
                torch.max(self.mesh_vertices, dim=0)[0],
            )
        else:
            z = torch.zeros(3, dtype=torch.float32, device=self.mesh_vertices.device)
            self.mesh_aabb = (z, z.clone())
        self._aabb_host = (self.mesh_aabb[0].tolist(), self.mesh_aabb[1].tolist())
        self.as_wrapper.build_accel_structure(self.mesh_vertices, self.mesh_faces)

    def refit(self, vertices: torch.Tensor):
        """Extension (SURVEY §8f): move the vertices of the SAME topology and re-fit the BVH in place
        instead of rebuilding it (`update_raw`, like the reference, always rebuilds).  Results are
        exact for the deformed mesh; traversal efficiency degrades if the deformation is large."""
        self.mesh_vertices = vertices.float().contiguous().to(self.as_wrapper.blob.device)
        self.mesh_aabb = (torch.min(self.mesh_vertices, dim=0)[0], torch.max(self.mesh_vertices, dim=0)[0])
        self._aabb_host = (self.mesh_aabb[0].tolist(), self.mesh_aabb[1].tolist())
        self.as_wrapper._inner.refit(self.mesh_vertices, self.mesh_faces)

    def save_bvh(self, path: str):
        """Extension (SURVEY §8f): write the flat BVH blob to disk."""
        self.as_wrapper._inner.save(path)

    # ------------------------------------------------------------------ queries
    def intersects_any(self, origins: torch.Tensor, directions: torch.Tensor) -> torch.Tensor:
        """Bool[*b] — does each ray hit the mesh (reference :77-82)."""
        return hops.intersects_any(self.as_wrapper, origins, directions)

    def intersects_first(self, origins: torch.Tensor, directions: torch.Tensor) -> torch.Tensor:
        """Int32[*b] — index of the first triangle hit, -1 on a miss (reference :90-95)."""
        return hops.intersects_first(self.as_wrapper, origins, directions)

    def intersects_closest(self, origins: torch.Tensor, directions: torch.Tensor, stream_compaction: bool = False):
        """Closest hit per ray (reference :117-146).

        stream_compaction=False -> (hit[*b], front[*b], tri_idx[*b], loc[*b,3], uv[*b,2])
        stream_compaction=True  -> (hit[*b], front[h], ray_idx[h], tri_idx[h], loc[h,3], uv[h,2])
        with ray_idx the flattened row-major ray index in ascending order (int32).
        """
        hit, front, tri_idx, loc, uv = hops.intersects_closest(self.as_wrapper, origins, directions)
        if stream_compaction:
            front_c, ray_idx, tri_c, loc_c, uv_c = hops.compact_closest(hit, front, tri_idx, loc, uv)
            return hit, front_c, ray_idx, tri_c, loc_c, uv_c
        return hit, front, tri_idx, loc, uv

    def intersects_closest_pinhole(self, cam_mat, cam_origin, width: int, height: int, focal: float,
                                   stream_compaction: bool = False):
        """Extension (SURVEY §8f): `intersects_closest` for the pinhole camera of the reference's benchmark
        (`gen_rays`, test/performance_test.py:10-20) with the rays generated inside the kernel.  Same tuples as
        `intersects_closest`, batch shape [height, width]."""
        hit, front, tri_idx, loc, uv = hops.intersects_closest_pinhole(self.as_wrapper, cam_mat, cam_origin, width, height, focal)
        if stream_compaction:
            front_c, ray_idx, tri_c, loc_c, uv_c = hops.compact_closest(hit, front, tri_idx, loc, uv)
            return hit, front_c, ray_idx, tri_c, loc_c, uv_c
        return hit, front, tri_idx, loc, uv

    def interpolate(self, vertex_attribute: torch.Tensor, tri_idx: torch.Tensor, uv: torch.Tensor) -> torch.Tensor:
        """Extension (SURVEY §8f): barycentric interpolation of a per-vertex attribute at hit points, the post-op of
        the reference demo (test/test.py:35-42): uv0 * a[f0] + uv1 * a[f1] + (1 - uv0 - uv1) * a[f2]."""
        a = vertex_attribute.to(self.mesh_vertices.device)[self.mesh_faces[tri_idx.long()].long()]
        w0, w1 = uv[..., :1], uv[..., 1:]
        return w0 * a[..., 0, :] + w1 * a[..., 1, :] + (1 - w0 - w1) * a[..., 2, :]

    def intersects_location(self, origins: torch.Tensor, directions: torch.Tensor
                            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """(loc[h,3], ray_idx[h], tri_idx[h]) for every hit, at most 8 per ray (reference :157-164)."""
        return hops.intersects_location(self.as_wrapper, origins, directions, getattr(self, "max_hits", hops.MAX_ANYHIT_SIZE))

    def intersects_count(self, origins: torch.Tensor, directions: torch.Tensor) -> torch.Tensor:
        """Int32[*b] — number of triangles each ray crosses (reference :172-177)."""
        return hops.intersects_count(self.as_wrapper, origins, directions)

    def intersects_id(self, origins: torch.Tensor, directions: torch.Tensor, return_locations: bool = False,
                      multiple_hits: bool = True):
        """(tri_idx[h], ray_idx[h][, loc[h,3]]) (reference :191-223)."""
        if multiple_hits:
            loc, ray_idx, tri_idx = hops.intersects_location(self.as_wrapper, origins, directions,
                                                             getattr(self, "max_hits", hops.MAX_ANYHIT_SIZE))
            if return_locations:
                return tri_idx, ray_idx, loc
            return tri_idx, ray_idx
        hit, front, tri_idx, loc, uv = hops.intersects_closest(self.as_wrapper, origins, directions)
        _, ray_idx, tri_c, loc_c, _ = hops.compact_closest(hit, front, tri_idx, loc, uv)
        if return_locations:
            return tri_c, ray_idx, loc_c
        return tri_c, ray_idx

    def closest_point(self, points: torch.Tensor, max_distance: Optional[float] = None, return_uv: bool = False):
        """(closest[*b,3], distance[*b], triangle_id[*b][, uv[*b,2]]) — the nearest point of the mesh surface for
        every query point, in the order of trimesh.proximity.closest_point.  Triangles farther than `max_distance`
        (None = unbounded) are ignored; a point with no triangle in reach gets triangle_id -1, distance inf and
        closest 0.  Equal distances go to the smaller triangle index.  uv are the weights of the triangle's vertices
        0 and 1 like intersects_closest's, so `interpolate(attr, triangle_id, uv)` transfers attributes."""
        md = float("inf") if max_distance is None else float(max_distance)
        closest, distance, tri, uv = hops.closest_point(self.as_wrapper, points, md)
        if return_uv:
            return closest, distance, tri, uv
        return closest, distance, tri

    def signed_distance(self, points: torch.Tensor) -> torch.Tensor:
        """Float32[*b] — distance to the surface, positive inside and negative outside (trimesh.proximity.signed_distance).
        The sign is `contains_points` (with its documented decision procedure); an exact 0 is returned as +0.0."""
        _, d, _ = self.closest_point(points)
        inside = self.contains_points(points.reshape(-1, 3)).reshape(d.shape)
        return torch.where(inside | (d == 0), d, -d)

    DEFAULT_CHECK_DIRECTION = (0.4395064455, 0.617598629942, 0.652231566745)   # reference :245-247

    def contains_parity(self, points: torch.Tensor, direction, active: Optional[torch.Tensor] = None, out=None,
                        stop_when_broken: bool = False):
        """Fused core of `contains_points`: (contain, broken, flags[2] = [any inside the AABB, any broken]) for one
        direction; with `active` / `out` a masked in-place update (see hops.contains_parity)."""
        return hops.contains_parity(self.as_wrapper, points, direction, self._aabb_host[0], self._aabb_host[1], active, out,
                                    stop_when_broken)

    def contains_points(self, points: torch.Tensor, check_direction: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Bool[n] — is each point inside the (closed) mesh (reference :231-279).

        Same decision procedure as the reference: a point is inside iff it lies strictly within
        the mesh AABB and the crossing counts along +dir and -dir are both odd; points whose two
        counts disagree with one of them zero are 'broken' and retried once with a random
        direction when no direction was given.  When a direction IS given and some point is
        broken the reference returns its initial all-False tensor (:279) — kept.
        The two count traversals, the AABB test and the parity logic run in one kernel.
        """
        return contains_points_flow(self.contains_parity, points, check_direction)


def contains_points_flow(parity, points: torch.Tensor, check_direction, reduce_flags=None, draw_direction=None):
    """Control flow of the reference's `contains_points` (ray_optix.py:236-279) around the fused parity kernel.

    `parity(points, direction, active, out)` is RayMeshIntersector.contains_parity.  A ray-sharded caller
    (triro.distributed) passes `reduce_flags` (OR of the two decision flags over all ranks) and `draw_direction`
    (one retry direction for all ranks), so that N ranks take the branches one process would take."""
    zeros = lambda: torch.zeros(points.shape[:-1], dtype=torch.bool, device=points.device)   # noqa: E731  (:236)
    read = reduce_flags if reduce_flags is not None else (lambda f: tuple(int(x) for x in f.tolist()))
    direction = (RayMeshIntersector.DEFAULT_CHECK_DIRECTION if check_direction is None
                 else check_direction.detach().flatten().tolist())
    contain, broken, flags = parity(points, direction, None, None)
    any_inside, any_broken = read(flags)                              # one host sync for both decisions
    if not any_inside:                                                # reference :243-244
        return zeros()
    if not any_broken:                                                # reference :269-270
        return contain
    if check_direction is not None:                                   # reference :236,:279
        return zeros()
    # reference :272-277: contains[broken] = self.contains_points(points[broken], new_direction) — as ONE masked,
    # in-place launch: only the broken points are traced again and only their entries are rewritten (no
    # points[broken] gather, no boolean-index scatter).  The recursive call's own early returns are kept: it
    # yields all False for the subset when none of the broken points lies inside the AABB (:243-244) or when
    # some point is broken again (a direction was given, :279); otherwise the subset's parity result.
    new_direction = draw_direction() if draw_direction is not None else (torch.rand(3) - 0.5).tolist()   # CPU generator, as :273
    # The retry's per-point results only matter when NO point is broken again, so the launch may stop at the first one
    # (typical: every ordinary outside point is 'broken' by the reference's definition, and stays so).
    was_broken = broken.clone()
    _, _, flags = parity(points, new_direction, broken, (contain, broken), True)
    sub_inside, sub_broken = read(flags)
    if not sub_inside or sub_broken:
        contain.logical_and_(was_broken.logical_not_())      # contains[broken] = False, as two elementwise kernels
    return contain


class OptixAccelStructureWrapper:
    """Name kept from the reference (ray_optix.py:282-294); wraps the flat BVH8 blob."""

    def __init__(self):
        self._inner = hops.AccelStructure()

    def build_accel_structure(self, vertices: torch.Tensor, faces: torch.Tensor):
        self._inner.build(vertices, faces)

    @property
    def blob(self):
        return self._inner.blob

    @property
    def header(self):
        return self._inner.header
