"""numpy adapter with the calling convention of trimesh.ray (SURVEY §8f rank 2).

The reference mirrors `trimesh.ray` but speaks torch CUDA tensors (reference README.md:3); its own
benchmark calls the CPU side as `mesh.ray.intersects_location(origins, directions, multiple_hits=False)`
with numpy arrays (test/performance_test.py:75).  This class takes and returns numpy arrays with
trimesh's conventions (positional mesh argument, float64 locations, int64 indices, (n,) bool
masks) so that code written against `mesh.ray` can run on the B200 kernels unchanged.

Differences from trimesh that remain (inherited from the reference, SURVEY Appendix A.9): at most
8 hits per ray with multiple_hits=True; `contains_points` uses the reference's decision procedure.
"""
from __future__ import annotations

import numpy as np
import torch

from triro.ray.ray_optix import RayMeshIntersector as _TorchIntersector


class RayMeshIntersector:
    def __init__(self, geometry=None, vertices=None, faces=None, device="cuda"):
        if geometry is not None:
            vertices, faces = geometry.vertices, geometry.faces
        if vertices is None or faces is None:
            raise ValueError("a mesh or vertices and faces must be provided")
        self.device = torch.device(device)
        # mesh, BVH and rays all live on `device` (the intersector keeps a CUDA input's device)
        self._rmi = _TorchIntersector(vertices=torch.as_tensor(np.asarray(vertices, dtype=np.float32)).to(self.device),
                                      faces=torch.as_tensor(np.asarray(faces).astype(np.int32)).to(self.device))

    def _rays(self, ray_origins, ray_directions):
        o = np.asarray(ray_origins, dtype=np.float32).reshape(-1, 3)
        d = np.asarray(ray_directions, dtype=np.float32).reshape(-1, 3)
        if o.shape != d.shape:
            raise ValueError("ray_origins and ray_directions must both be (n, 3)")
        return torch.from_numpy(np.ascontiguousarray(o)).to(self.device), torch.from_numpy(np.ascontiguousarray(d)).to(self.device)

    def intersects_location(self, ray_origins, ray_directions, multiple_hits=True, **kwargs):
        """-> (locations (h,3) float64, index_ray (h,) int64, index_tri (h,) int64)"""
        o, d = self._rays(ray_origins, ray_directions)
        if multiple_hits:
            loc, ray_idx, tri_idx = self._rmi.intersects_location(o, d)
        else:
            tri_idx, ray_idx, loc = self._rmi.intersects_id(o, d, return_locations=True, multiple_hits=False)
        return (loc.cpu().numpy().astype(np.float64), ray_idx.cpu().numpy().astype(np.int64),
                tri_idx.cpu().numpy().astype(np.int64))

    def intersects_id(self, ray_origins, ray_directions, multiple_hits=True, max_hits=20, return_locations=False, **kwargs):
        """-> index_tri, index_ray[, locations]"""
        loc, ray_idx, tri_idx = self.intersects_location(ray_origins, ray_directions, multiple_hits=multiple_hits)
        return (tri_idx, ray_idx, loc) if return_locations else (tri_idx, ray_idx)

    def intersects_first(self, ray_origins, ray_directions, **kwargs):
        o, d = self._rays(ray_origins, ray_directions)
        return self._rmi.intersects_first(o, d).cpu().numpy().astype(np.int64)

    def intersects_any(self, ray_origins, ray_directions, **kwargs):
        o, d = self._rays(ray_origins, ray_directions)
        return self._rmi.intersects_any(o, d).cpu().numpy()

    def contains_points(self, points):
        p = torch.from_numpy(np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 3))).to(self.device)
        return self._rmi.contains_points(p).cpu().numpy()

    def _points(self, points):
        return torch.from_numpy(np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, 3))).to(self.device)

    def closest_point(self, points):
        """trimesh.proximity.closest_point -> (closest (n,3) float64, distance (n,) float64, triangle_id (n,) int64)"""
        c, d, t = self._rmi.closest_point(self._points(points))
        return c.cpu().numpy().astype(np.float64), d.cpu().numpy().astype(np.float64), t.cpu().numpy().astype(np.int64)

    def signed_distance(self, points):
        """trimesh.proximity.signed_distance -> (n,) float64, positive inside the mesh"""
        return self._rmi.signed_distance(self._points(points)).cpu().numpy().astype(np.float64)
