"""Operator layer over the C ABI of libtriro_b200.so (include/raymesh_b200.h).

Drop-in for the reference's op shim `triro/backend/ops.py:12-192`: same function names and
argument meaning (`intersects_any/first/closest/count/location(accel, origins, dirs)`,
`get_module()`, the five init functions called at import), but instead of JIT-compiling a
pybind11/OptiX module it loads a prebuilt CUDA library through ctypes.  torch only provides
device memory and the stream; every computation is a hand-written sm_100a kernel.

There is NO CPU fallback: if the library is missing or no CUDA device is present the
functions raise.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
from typing import Tuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libtriro_b200.so"
MAX_ANYHIT_SIZE = 8          # reference LaunchParams.h:8
MAX_BATCH_DIMS = 3           # reference LaunchParams.h:9 (MAX_SIZE_LENGTH = 4 incl. the trailing 3)
TRACE_SCRATCH_BYTES = 256
BLOB_HEADER_BYTES = 256
BLOB_MAGIC = 0x38485642
MAX_DEPTH = 60               # rt_core.cuh kMaxDepth
HOST_CHUNK = 1 << 20
ABI_VERSION = 2
ALLHITS_STAGING_BYTES = 2 << 30   # all-hits staging per launch window (nray_window * max_hits * 16 B)

_lib = None


class RayDesc(C.Structure):
    """rt_ray_desc — mirrors RayInput (reference LaunchParams.h:11-28)."""

    _fields_ = [
        ("nray", C.c_int64),
        ("shape", C.c_int64 * 4),
        ("origins", C.c_void_p),
        ("o_stride", C.c_int64 * 4),
        ("directions", C.c_void_p),
        ("d_stride", C.c_int64 * 4),
    ]


class TraceOpts(C.Structure):
    """rt_trace_opts — per-call options of every trace entry point (include/raymesh_b200.h)."""

    _fields_ = [("tmax", C.c_float), ("schedule", C.c_int32), ("ray_first", C.c_int64), ("ray_count", C.c_int64),
                ("flags", C.c_uint32), ("refill_threshold", C.c_int32), ("tri_threshold", C.c_int32),
                ("grid_div", C.c_int32), ("reserved", C.c_int32 * 4)]


SCHED_AUTO, SCHED_DIRECT, SCHED_COOP_COHERENT, SCHED_COOP_INCOHERENT = 0, 1, 3, 4
SCHED_QUEUED, SCHED_SLOTS = 2, 5     # removed schedules: the library runs SCHED_COOP_INCOHERENT for them (ABI v2 aliases)
OPT_SCRATCH_ZEROED = 1
OPT_STOP_WHEN_BROKEN = 2
OPT_NO_LANE_SHARING = 4
OPT_NO_TILE_ORDER = 8


class Pinhole(C.Structure):
    """rt_pinhole — camera of the fused ray-generation entry point."""

    _fields_ = [("width", C.c_int64), ("height", C.c_int64), ("focal", C.c_float), ("cam_mat", C.c_float * 9),
                ("origin", C.c_float * 3)]


def _declare(lib):
    vp, i64, sz, ci = C.c_void_p, C.c_int64, C.c_size_t, C.c_int
    psz = C.POINTER(C.c_size_t)
    prd = C.POINTER(RayDesc)
    pto = C.POINTER(TraceOpts)
    pf = C.POINTER(C.c_float)
    sig = {
        "rt_last_error": (C.c_char_p, []),
        "rt_abi_version": (ci, []),
        "rt_device_sm_count": (ci, []),
        "rt_bvh_sizes": (ci, [i64, i64, psz, psz]),
        "rt_bvh_build": (ci, [vp, i64, vp, i64, vp, sz, vp, sz, vp]),
        "rt_bvh_refit_sizes": (ci, [i64, psz]),
        "rt_bvh_refit": (ci, [vp, i64, vp, i64, vp, sz, vp, sz, vp]),
        "rt_sort_sizes": (ci, [i64, psz]),
        "rt_sort_pairs_u64": (ci, [vp, vp, i64, vp, sz, vp]),
        "rt_trace_any": (ci, [vp, prd, pto, vp, vp, vp]),
        "rt_trace_first": (ci, [vp, prd, pto, vp, vp, vp]),
        "rt_trace_closest": (ci, [vp, prd, pto, vp, vp, vp, vp, vp, vp, vp]),
        "rt_trace_count": (ci, [vp, prd, pto, vp, vp, vp]),
        "rt_trace_closest_pinhole": (ci, [vp, C.POINTER(Pinhole), pto, vp, vp, vp, vp, vp, vp, vp]),
        "rt_compact_sizes": (ci, [i64, psz]),
        "rt_compact_scan": (ci, [vp, i64, vp, sz, vp, vp]),
        "rt_compact_scatter": (ci, [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "rt_allhits_sizes": (ci, [i64, ci, psz, psz]),
        "rt_allhits_trace": (ci, [vp, prd, pto, ci, vp, vp, vp, sz, vp, vp, vp]),
        "rt_allhits_scatter": (ci, [i64, ci, vp, vp, vp, vp, vp, vp, vp]),
        "rt_allhits_scatter_at": (ci, [i64, ci, vp, vp, vp, i64, ci, vp, vp, vp, vp]),
        "rt_compact_scatter_at": (ci, [vp, i64, vp, vp, vp, vp, vp, i64, ci, vp, vp, vp, vp, vp, vp]),
        "rt_contains_parity": (ci, [vp, prd, pto, pf, pf, pf, vp, vp, vp, vp, vp, vp]),
        "rt_trace_stats": (ci, [vp, prd, pto, ci, vp, vp, vp]),
        "rt_closest_point": (ci, [vp, prd, pto, C.c_float, vp, vp, vp, vp, vp, vp, vp]),
        "rt_winding_moments_sizes": (ci, [i64, psz, psz]),
        "rt_winding_moments": (ci, [vp, vp, sz, vp, sz, vp]),
        "rt_winding_number": (ci, [vp, vp, prd, pto, C.c_float, vp, vp, vp, vp]),
        "rt_pseudonormals_sizes": (ci, [i64, psz, psz]),
        "rt_pseudonormals": (ci, [vp, vp, sz, vp, sz, vp, vp]),
        "rt_signed_distance": (ci, [vp, vp, prd, pto, vp, vp, vp, vp]),
        "rt_signed_distance_closest": (ci, [vp, vp, prd, pto, vp, vp, vp, vp, vp, vp, vp]),
        "rt_distance_grad_sizes": (ci, [i64, i64, psz]),
        "rt_distance_grad": (ci, [prd, pto, vp, vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, sz, vp]),
        "rt_ray_grad_sizes": (ci, [i64, i64, psz]),
        "rt_ray_grad": (ci, [prd, pto, i64, vp, vp, vp, vp, vp, i64, vp, i64, vp, vp, vp, vp, sz, vp]),
        "rt_scene_prepare_sizes": (ci, [i64, i64, psz]),
        "rt_scene_prepare": (ci, [i64, vp, i64, vp, vp, vp, sz, vp, vp, vp]),
        "rt_scene_trace": (ci, [vp, vp, prd, pto, ci, vp, vp, vp, vp, vp, vp, vp, vp]),
        "rt_scene_point_sizes": (ci, [i64, psz]),
        "rt_scene_point_prepare": (ci, [vp, i64, vp, sz, vp]),
        "rt_scene_closest_point": (ci, [vp, vp, vp, prd, pto, C.c_float, vp, vp, vp, vp, vp, vp]),
        "rt_scene_signed_distance": (ci, [vp, vp, vp, vp, prd, pto, vp, vp, vp, vp, vp, vp]),
        "rt_scene_grad_sizes": (ci, [i64, i64, i64, ci, psz]),
        "rt_scene_ray_grad": (ci, [vp, i64, vp, i64, i64, prd, pto, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "rt_scene_distance_grad": (ci, [vp, i64, vp, i64, i64, prd, pto, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz,
                                        vp]),
        "rt_host_closest_sizes": (ci, [i64, psz]),
        "rt_host_trace_closest": (ci, [vp, i64, vp, ci, vp, pto, vp, vp, vp, vp, vp, vp, sz]),
        "rt_host_trace_closest_compact": (ci, [vp, i64, vp, ci, vp, pto, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_int64), vp, sz]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)   # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    return sig


EXPORTS = None


def get_module():
    """Load libtriro_b200.so (reference: get_module(), ops.py:12-46, which JIT-builds instead)."""
    global _lib, EXPORTS
    if _lib is not None:
        return _lib
    path = os.environ.get("TRIRO_B200_LIB", os.path.join(_HERE, LIB_NAME))
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    EXPORTS = _declare(lib)
    if lib.rt_abi_version() != ABI_VERSION:
        raise RuntimeError(f"{path}: ABI version {lib.rt_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return _lib


# The reference initialises OptiX at import (triro/ray/__init__.py:17-22).  There is no OptiX
# here; the five entry points are kept so that code calling them keeps working.  They make sure
# the native library is loadable, which is the equivalent "import = ready" guarantee.
def init_optix():
    get_module()


def create_optix_context():
    get_module()


def create_optix_module():
    get_module()


def create_optix_pipelines():
    get_module()


def build_sbts():
    get_module()


def _check(rc: int, what: str):
    if rc != 0:
        msg = get_module().rt_last_error().decode("utf-8", "replace")
        if rc in (-1, -3):
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what}: {msg} (status {rc})")


TMAX_DEFAULT = 1.0e7        # reference: tmax of every optixTrace, shaders.cu:86
MAX_HITS_LIMIT = 64


def _env_int(name: str) -> int:
    try:
        return int(os.environ.get(name, "0"))
    except ValueError:
        return 0


# Scheduling knobs for experiments (tools/), read ONCE at import; 0 = the library's defaults.  The C library itself
# reads no environment variable on the trace path: everything a launch depends on is in rt_trace_opts.
_KNOBS = dict(schedule=_env_int("TRIRO_SCHED"), refill_threshold=_env_int("TRIRO_REFILL_THRESHOLD"),
              tri_threshold=_env_int("TRIRO_TRI_THRESHOLD"), grid_div=_env_int("TRIRO_GRID_DIV"),
              no_lane_sharing=_env_int("TRIRO_NO_LANE_SHARING"), no_tile_order=_env_int("TRIRO_NO_TILE_ORDER"))


def set_knobs(**kw) -> dict:
    """Override the experiment knobs (schedule, refill_threshold, tri_threshold, grid_div, no_lane_sharing, no_tile_order) for later calls of this
    process; returns the previous values.  Every schedule gives bit-identical results."""
    old = dict(_KNOBS)
    for k, v in kw.items():
        if k not in _KNOBS:
            raise KeyError(k)
        _KNOBS[k] = int(v)
    return old


_opts_cache: dict = {}


def trace_opts(accel=None, ray_first: int = 0, ray_count: int = -1, scratch_zeroed: bool = True) -> TraceOpts:
    """rt_trace_opts of one call: the accel's tmax (default 1e7 = the reference's hard-coded value), the ray window,
    and the experiment knobs.  The whole-batch form is cached per (tmax, knobs)."""
    if ray_first == 0 and ray_count < 0 and scratch_zeroed:
        tm = float(getattr(getattr(accel, "_inner", accel), "tmax", TMAX_DEFAULT)) if accel is not None else TMAX_DEFAULT
        key = (tm, *_KNOBS.values())
        o = _opts_cache.get(key)
        if o is None:
            o = _opts_cache[key] = _trace_opts(accel, 0, -1, True)
        return o
    return _trace_opts(accel, ray_first, ray_count, scratch_zeroed)


def _trace_opts(accel, ray_first: int, ray_count: int, scratch_zeroed: bool) -> TraceOpts:
    o = TraceOpts()
    o.tmax = float(getattr(getattr(accel, "_inner", accel), "tmax", TMAX_DEFAULT)) if accel is not None else TMAX_DEFAULT
    o.schedule = _KNOBS["schedule"]
    o.ray_first, o.ray_count = int(ray_first), max(int(ray_count), 0)     # 0 = up to the end of the batch
    o.flags = (OPT_SCRATCH_ZEROED if scratch_zeroed else 0) | (OPT_NO_LANE_SHARING if _KNOBS["no_lane_sharing"] else 0) | (OPT_NO_TILE_ORDER if _KNOBS["no_tile_order"] else 0)
    o.refill_threshold, o.tri_threshold, o.grid_div = _KNOBS["refill_threshold"], _KNOBS["tri_threshold"], _KNOBS["grid_div"]
    return o


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_scratch_cache: dict = {}


def _scratch(device, stream: int | None = None) -> torch.Tensor:
    """RT_TRACE_SCRATCH_BYTES of zeroed device memory private to (device, current stream).  Every launch leaves its
    scratch zeroed again (the last CTA resets it), so with RT_OPT_SCRATCH_ZEROED a trace call is exactly one kernel
    launch; launches that share a scratch are ordered by their stream."""
    dev = device if isinstance(device, torch.device) else torch.device(device)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), _stream(dev) if stream is None else stream)
    t = _scratch_cache.get(key)
    if t is None:
        t = torch.zeros(TRACE_SCRATCH_BYTES, dtype=torch.uint8, device=dev)
        _scratch_cache[key] = t
    return t


class _on_device:
    """`with torch.cuda.device(dev)` only when `dev` is not already current (the context manager costs ~3 us per call)."""

    __slots__ = ("ctx",)

    def __init__(self, dev):
        self.ctx = None if dev.index is None or torch.cuda.current_device() == dev.index else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            return self.ctx.__exit__(*a)


def _ptr(t: torch.Tensor | None):
    return None if t is None else C.c_void_p(t.data_ptr())


def tensor_input_check(*ts: torch.Tensor):
    """Reference tensorInputCheck (ray.cpp:104-123) checks is_cuda + strided layout and, on
    failure, prints to stderr and returns an empty tensor; here the same conditions (plus the
    dtype the reference silently reinterprets) raise ValueError."""
    for t in ts:
        if not isinstance(t, torch.Tensor):
            raise ValueError("input must be a torch.Tensor")
        if not t.is_cuda:
            raise ValueError("input tensors must reside in cuda device.")
        if t.layout != torch.strided:
            raise ValueError("input tensor layout must be torch.strided.")
        if t.dtype != torch.float32:
            raise ValueError(f"input tensors must be float32 (got {t.dtype})")


_desc_cache = (None, None)      # (key, value), replaced as ONE object so that threads never pair a key with another call's value


def make_ray_desc(origins: torch.Tensor, dirs: torch.Tensor | None) -> Tuple[RayDesc, tuple]:
    """fillArray of the reference (ray.cpp:151-159): right-align shape/strides into 4 slots.
    The batch shape is that of `origins` (ray.cpp:177-179).  A call with the same addresses, shapes and strides as the
    previous one (a render loop) reuses its descriptor: filling a ctypes struct costs more than the rest of the host side."""
    key = (origins.data_ptr(), origins.shape, origins.stride(), origins.device,
           None if dirs is None else (dirs.data_ptr(), dirs.shape, dirs.stride(), dirs.device))
    global _desc_cache
    cached = _desc_cache
    if cached[0] == key:
        return cached[1]
    val = _make_ray_desc(origins, dirs)
    if val[0]._keepalive is None:          # reshaped copies must not outlive their call through the cache
        _desc_cache = (key, val)
    return val


def _make_ray_desc(origins: torch.Tensor, dirs: torch.Tensor | None) -> Tuple[RayDesc, tuple]:
    if origins.dim() < 1 or origins.shape[-1] != 3:
        raise ValueError(f"origins must have shape [*b, 3], got {tuple(origins.shape)}")
    if dirs is not None and tuple(dirs.shape) != tuple(origins.shape):
        raise ValueError(f"directions {tuple(dirs.shape)} must have the shape of origins {tuple(origins.shape)}")
    if dirs is not None and dirs.device != origins.device:
        raise ValueError("origins and directions must be on the same device")
    batch = tuple(origins.shape[:-1])
    keep = None
    if len(batch) > MAX_BATCH_DIMS:
        # The reference keeps only the last 4 sizes/strides and silently reads wrong data (ray.cpp:151-159,
        # SURVEY A.1).  Here the surplus leading dimensions are merged into one (a view when the strides allow
        # it, otherwise a copy); results are reshaped back to the full batch shape by the callers.
        origins = origins.reshape(-1, *origins.shape[-3:])
        dirs = dirs.reshape(-1, *dirs.shape[-3:]) if dirs is not None else None
        keep = (origins, dirs)
    rd = RayDesc()
    rd._keepalive = keep
    n = 1
    for s in batch:
        n *= s
    rd.nray = n
    pad = 4 - origins.dim()
    for i in range(4):
        j = i - pad
        rd.shape[i] = origins.shape[j] if j >= 0 else 1
        rd.o_stride[i] = origins.stride(j) if j >= 0 else 0
        rd.d_stride[i] = (dirs.stride(j) if j >= 0 else 0) if dirs is not None else 0
    rd.origins = origins.data_ptr()
    rd.directions = dirs.data_ptr() if dirs is not None else None
    return rd, batch


class AccelStructure:
    """Flat, relocatable BVH8 blob owned by torch (reference: OptixAccelStructureWrapperCPP,
    ray.h:11-16, whose GAS is an opaque buffer owned by C++)."""

    def __init__(self):
        self.tmax: float = TMAX_DEFAULT      # rays are clipped to (0, tmax)
        self.blob: torch.Tensor | None = None
        self.header: dict | None = None
        self.build_ms: float | None = None
        self.winding_moments: torch.Tensor | None = None   # ops.winding_moments() cache, dropped with the blob's contents
        self.pseudo_normals: tuple | None = None           # ops.pseudo_normals() cache, likewise
        self.generation: int = 0                           # counts build() and refit(): scenes detect stale members

    def build(self, vertices: torch.Tensor, faces: torch.Tensor, timing: bool = False):
        lib = get_module()
        if not (vertices.is_cuda and faces.is_cuda):
            raise ValueError("vertices and faces must reside in cuda device.")
        if vertices.device != faces.device:
            raise ValueError("vertices and faces must be on the same device")
        if vertices.dtype != torch.float32 or faces.dtype != torch.int32:
            raise ValueError("vertices must be float32 and faces int32")
        if vertices.dim() != 2 or vertices.shape[1] != 3 or faces.dim() != 2 or faces.shape[1] != 3:
            raise ValueError("vertices must be [n,3] and faces [f,3]")
        vertices = vertices.contiguous()
        faces = faces.contiguous()
        dev = vertices.device
        nv, nf = vertices.shape[0], faces.shape[0]
        ws_b, blob_b = C.c_size_t(), C.c_size_t()
        _check(lib.rt_bvh_sizes(nv, nf, C.byref(ws_b), C.byref(blob_b)), "rt_bvh_sizes")
        with torch.cuda.device(dev):
            ws = torch.empty(ws_b.value, dtype=torch.uint8, device=dev)
            blob = torch.empty(blob_b.value, dtype=torch.uint8, device=dev)
            if timing:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
            _check(lib.rt_bvh_build(_ptr(vertices), nv, _ptr(faces), nf, _ptr(ws), ws_b.value, _ptr(blob),
                                    blob_b.value, _stream(dev)), "rt_bvh_build")
            if timing:
                e1.record()
            # the reference's build is synchronous too (2x cudaDeviceSynchronize, ray.cpp:85,95)
            hdr = parse_header(blob[:BLOB_HEADER_BYTES].cpu().numpy().tobytes())
            if timing:
                self.build_ms = e0.elapsed_time(e1)
        del ws
        if hdr["magic"] != BLOB_MAGIC:
            raise RuntimeError("rt_bvh_build produced an invalid blob header")
        if hdr["bad_index_faces"]:
            raise ValueError(f"{hdr['bad_index_faces']} faces reference vertices outside [0, {nv})")
        validate_header(hdr, blob.numel())
        self.blob = blob
        self.header = hdr
        self.winding_moments = None
        self.pseudo_normals = None
        self.generation += 1
        return self

    def refit(self, vertices: torch.Tensor, faces: torch.Tensor):
        """Same topology, new vertex positions: rewrite the triangle records and re-fit all node
        boxes bottom-up in place (rt_bvh_refit) — no sort, no hierarchy emission.  Works on any valid blob
        (built here, received by broadcast, loaded from disk): the used prefix carries the parent links."""
        lib = get_module()
        if self.blob is None:
            raise RuntimeError("acceleration structure has not been built")
        if vertices.dtype != torch.float32 or faces.dtype != torch.int32 or not (vertices.is_cuda and faces.is_cuda):
            raise ValueError("vertices must be float32 and faces int32 CUDA tensors")
        if vertices.device != self.blob.device or faces.device != self.blob.device:
            raise ValueError(f"refit: vertices / faces must be on the blob's device {self.blob.device}")
        if faces.shape[0] != self.header["n_tris"]:
            raise ValueError(f"refit needs the same topology: {faces.shape[0]} faces, BVH was built for {self.header['n_tris']}")
        vertices = vertices.contiguous()
        faces = faces.contiguous()
        dev = self.blob.device
        wb = C.c_size_t()
        _check(lib.rt_bvh_refit_sizes(faces.shape[0], C.byref(wb)), "rt_bvh_refit_sizes")
        with torch.cuda.device(dev):
            ws = torch.empty(max(wb.value, 256), dtype=torch.uint8, device=dev)
            _check(lib.rt_bvh_refit(_ptr(vertices), vertices.shape[0], _ptr(faces), faces.shape[0], _ptr(ws), ws.numel(),
                                    _ptr(self.blob), self.blob.numel(), _stream(dev)), "rt_bvh_refit")
            self.header = parse_header(self.blob[:BLOB_HEADER_BYTES].cpu().numpy().tobytes())
        self.winding_moments = None
        self.pseudo_normals = None
        self.generation += 1
        return self

    def save(self, path: str):
        """Serialise the used prefix of the blob (header + triangles + nodes + parent links)."""
        torch.save({"format": "triro_b200_bvh8", "abi_version": ABI_VERSION, "blob": self.used().cpu()}, path)

    def load(self, path: str, device="cuda"):
        d = torch.load(path, map_location="cpu")
        if d.get("format") != "triro_b200_bvh8" or d.get("abi_version") != ABI_VERSION:
            raise ValueError(f"{path} is not a BVH blob of this ABI version")
        return self.adopt(d["blob"].to(device))

    def adopt(self, blob: torch.Tensor):
        """Attach to a blob received from elsewhere (NCCL broadcast, torch.load).  The header is validated against
        the tensor exactly like a freshly built one: a truncated, foreign or corrupt blob is refused here instead of
        overrunning the traversal stack or reading out of bounds in a kernel."""
        if blob.dtype != torch.uint8 or blob.dim() != 1 or blob.numel() < BLOB_HEADER_BYTES or not blob.is_contiguous():
            raise ValueError("a BVH blob is a contiguous 1-D uint8 tensor of at least 256 bytes")
        if blob.is_cuda and blob.data_ptr() % 256 != 0:
            raise ValueError("a BVH blob must be 256-byte aligned")
        hdr = parse_header(blob[:BLOB_HEADER_BYTES].cpu().numpy().tobytes())
        if hdr["magic"] != BLOB_MAGIC or hdr["abi_version"] != ABI_VERSION:
            raise ValueError("not a BVH blob of this ABI version")
        validate_header(hdr, blob.numel())
        self.blob = blob
        self.header = hdr
        self.winding_moments = None
        self.pseudo_normals = None
        return self

    def used(self) -> torch.Tensor:
        """Prefix of the blob that must travel (header + triangles + nodes in use + their parent links)."""
        return self.blob[: self.header["used_bytes"]]

    def free(self):
        self.blob = None
        self.header = None
        self.winding_moments = None
        self.pseudo_normals = None


def parse_header(raw: bytes) -> dict:
    magic, abi, n_tris, n_nodes, depth, cap = struct.unpack_from("<6I", raw, 0)
    tris_off, nodes_off, used = struct.unpack_from("<3Q", raw, 24)
    aabb = struct.unpack_from("<6f", raw, 48)
    bad, overflow = struct.unpack_from("<2I", raw, 72)
    (parents_off,) = struct.unpack_from("<Q", raw, 80)
    return dict(magic=magic, abi_version=abi, n_tris=n_tris, n_nodes=n_nodes, depth=depth, n_nodes_cap=cap,
                tris_offset=tris_off, nodes_offset=nodes_off, used_bytes=used, aabb_lo=aabb[:3], aabb_hi=aabb[3:],
                bad_index_faces=bad, node_overflow=overflow, parents_offset=parents_off)


def validate_header(hdr: dict, blob_bytes: int) -> None:
    """What the build path guarantees, checked for every blob before a kernel may walk it."""
    if hdr["node_overflow"]:
        raise RuntimeError("BVH node pool overflow (internal error)")
    if hdr["depth"] > MAX_DEPTH:
        raise RuntimeError(f"BVH depth {hdr['depth']} exceeds the traversal stack ({MAX_DEPTH}); mesh too degenerate")
    nt, nn = hdr["n_tris"], hdr["n_nodes"]
    ok = (nn >= 1 and hdr["tris_offset"] == BLOB_HEADER_BYTES and hdr["tris_offset"] % 16 == 0
          and hdr["nodes_offset"] % 16 == 0 and hdr["nodes_offset"] >= hdr["tris_offset"] + 48 * nt
          and hdr["parents_offset"] % 4 == 0 and hdr["parents_offset"] >= hdr["nodes_offset"] + 80 * nn
          and hdr["used_bytes"] >= hdr["parents_offset"] + 4 * nn and hdr["used_bytes"] <= blob_bytes)
    if not ok:
        raise ValueError(f"inconsistent BVH blob header for a tensor of {blob_bytes} bytes (truncated or corrupt blob)")


def _blob_of(accel, device=None) -> torch.Tensor:
    inner = getattr(accel, "_inner", accel)
    if inner.blob is None:
        raise RuntimeError("acceleration structure has not been built")
    if device is not None and inner.blob.device != device:
        raise ValueError(f"the acceleration structure lives on {inner.blob.device} but the rays are on {device}")
    return inner.blob


# ------------------------------------------------------------------ operators (reference ops.py:84-192)
def intersects_any(accel_structure, origins: torch.Tensor, dirs: torch.Tensor) -> torch.Tensor:
    """Bool[*b]: does each ray hit anything with 0 < t < 1e7 (reference ops.py:84-101)."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, batch = make_ray_desc(origins, dirs)
    dev = origins.device
    with _on_device(dev):
        out = torch.empty(batch, dtype=torch.bool, device=dev)
        st = _stream(dev)
        _check(get_module().rt_trace_any(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure)), _ptr(out),
                                         _ptr(_scratch(dev, st)), st), "rt_trace_any")
    return out


def intersects_first(accel_structure, origins: torch.Tensor, dirs: torch.Tensor) -> torch.Tensor:
    """Int32[*b]: index of the nearest hit triangle or -1 (reference ops.py:104-119)."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, batch = make_ray_desc(origins, dirs)
    dev = origins.device
    with _on_device(dev):
        out = torch.empty(batch, dtype=torch.int32, device=dev)
        st = _stream(dev)
        _check(get_module().rt_trace_first(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure)), _ptr(out),
                                           _ptr(_scratch(dev, st)), st), "rt_trace_first")
    return out


def intersects_closest(accel_structure, origins: torch.Tensor, dirs: torch.Tensor, ray_first: int = 0, ray_count: int = -1):
    """(hit Bool[*b], front Bool[*b], tri Int32[*b], loc Float32[*b,3], uv Float32[*b,2])
    (reference ops.py:122-149, ray.cpp:231-289).  With a ray window [ray_first, ray_first + ray_count) of the
    flattened batch only those rays are traced and the outputs are 1-D over the window."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, batch = make_ray_desc(origins, dirs)
    if ray_first != 0 or ray_count >= 0:
        batch = (_window(rd.nray, ray_first, ray_count),)
    dev = origins.device
    with _on_device(dev):
        hit = torch.empty(batch, dtype=torch.bool, device=dev)
        front = torch.empty(batch, dtype=torch.bool, device=dev)
        tri = torch.empty(batch, dtype=torch.int32, device=dev)
        loc = torch.empty((*batch, 3), dtype=torch.float32, device=dev)
        uv = torch.empty((*batch, 2), dtype=torch.float32, device=dev)
        if hit.numel() == 0:
            return hit, front, tri, loc, uv
        st = _stream(dev)
        _check(get_module().rt_trace_closest(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure, ray_first, ray_count)),
                                             _ptr(hit), _ptr(front), _ptr(tri), _ptr(loc), _ptr(uv), _ptr(_scratch(dev, st)),
                                             st), "rt_trace_closest")
    return hit, front, tri, loc, uv


def _window(nray: int, ray_first: int, ray_count: int) -> int:
    if ray_first < 0 or ray_first > nray or (ray_count >= 0 and ray_first + ray_count > nray):
        raise ValueError(f"ray window [{ray_first}, +{ray_count}) outside the batch of {nray} rays")
    return nray - ray_first if ray_count < 0 else ray_count


def _query_batch(points: torch.Tensor, dirs: torch.Tensor | None, ray_first: int, ray_count: int,
                 counters: torch.Tensor | None = None, table: torch.Tensor | None = None):
    """Prelude of the point and scene queries: checks the batch (and the counters, and that a scene table lives on the
    batch's device) and returns (descriptor, output batch shape): the batch's, or 1-D over the window
    [ray_first, ray_first + ray_count).  An empty window zeroes the counters; the caller launches nothing."""
    tensor_input_check(points, *(() if dirs is None else (dirs,)))
    if table is not None and table.device != points.device:
        kind = "points" if dirs is None else "rays"
        raise ValueError(f"the scene lives on {table.device} but the {kind} are on {points.device}")
    rd, batch = make_ray_desc(points, dirs)
    n = rd.nray
    if ray_first != 0 or ray_count >= 0:
        n = _window(rd.nray, ray_first, ray_count)
        batch = (n,)
    if counters is not None:
        if (counters.dtype != torch.int64 or counters.device != points.device or counters.numel() != 4
                or not counters.is_contiguous()):
            raise ValueError("counters must be a contiguous int64 tensor of 4 elements on the points' device")
        if n == 0:
            counters.zero_()
    return rd, batch


def intersects_closest_into(accel_structure, origins: torch.Tensor, dirs: torch.Tensor, hit_ptr: int, front_ptr: int,
                            tri_ptr: int, loc_ptr: int, uv_ptr: int, ray_first: int = 0, ray_count: int = -1) -> None:
    """rt_trace_closest with caller-provided RAW output addresses (u8 hit, u8 front, i32 tri, f32 loc[3], f32 uv[2]
    per ray, dense).  The addresses may be peer-GPU memory mapped into this process (NVLink P2P / symmetric
    memory): the kernel then stores its results straight into another rank's tensors - the fused trace + gather
    of triro.distributed.  Asynchronous on the current stream."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, _ = make_ray_desc(origins, dirs)
    dev = origins.device
    if _window(rd.nray, ray_first, ray_count) == 0:
        return
    with torch.cuda.device(dev):
        _check(get_module().rt_trace_closest(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure, ray_first, ray_count)),
                                             C.c_void_p(hit_ptr), C.c_void_p(front_ptr), C.c_void_p(tri_ptr),
                                             C.c_void_p(loc_ptr), C.c_void_p(uv_ptr), _ptr(_scratch(dev)), _stream(dev)),
               "rt_trace_closest")


def intersects_closest_pinhole(accel_structure, cam_mat, cam_origin, width: int, height: int, focal: float):
    """Closest hit of the pinhole camera rays of the reference's benchmark (gen_rays,
    test/performance_test.py:10-20) generated inside the kernel: no ray tensors are built or read.
    Returns (hit[h,w], front[h,w], tri[h,w], loc[h,w,3], uv[h,w,2])."""
    blob = _blob_of(accel_structure)
    dev = blob.device
    cam = Pinhole()
    cam.width, cam.height, cam.focal = int(width), int(height), float(focal)
    m = [float(x) for x in torch.as_tensor(cam_mat).reshape(-1).tolist()]
    o = [float(x) for x in torch.as_tensor(cam_origin).reshape(-1).tolist()]
    if len(m) != 9 or len(o) != 3:
        raise ValueError("cam_mat must be 3x3 and cam_origin a 3-vector")
    for i in range(9):
        cam.cam_mat[i] = m[i]
    for i in range(3):
        cam.origin[i] = o[i]
    batch = (int(height), int(width))
    with torch.cuda.device(dev):
        hit = torch.empty(batch, dtype=torch.bool, device=dev)
        front = torch.empty(batch, dtype=torch.bool, device=dev)
        tri = torch.empty(batch, dtype=torch.int32, device=dev)
        loc = torch.empty((*batch, 3), dtype=torch.float32, device=dev)
        uv = torch.empty((*batch, 2), dtype=torch.float32, device=dev)
        _check(get_module().rt_trace_closest_pinhole(_ptr(blob), C.byref(cam), C.byref(trace_opts(accel_structure)), _ptr(hit),
                                                     _ptr(front), _ptr(tri), _ptr(loc), _ptr(uv), _ptr(_scratch(dev)),
                                                     _stream(dev)), "rt_trace_closest_pinhole")
    return hit, front, tri, loc, uv


def compact_closest(hit, front, tri, loc, uv):
    """Order-preserving stream compaction of dense closest-hit results: returns
    (front[h], ray_idx[h] int32, tri[h], loc[h,3], uv[h,2]) — what the reference computes with
    arange + five boolean-mask gathers (ray_optix.py:142-144)."""
    lib = get_module()
    dev = hit.device
    n = hit.numel()
    with torch.cuda.device(dev):
        ws_b = C.c_size_t()
        _check(lib.rt_compact_sizes(n, C.byref(ws_b)), "rt_compact_sizes")
        ws = torch.empty(max(ws_b.value, 256), dtype=torch.uint8, device=dev)
        total = torch.empty(1, dtype=torch.int64, device=dev)
        _check(lib.rt_compact_scan(_ptr(hit), n, _ptr(ws), ws.numel(), _ptr(total), _stream(dev)), "rt_compact_scan")
        h = int(total.item())   # the one host sync the API needs: output sizes
        front_c = torch.empty(h, dtype=torch.bool, device=dev)
        ray_idx = torch.empty(h, dtype=torch.int32, device=dev)
        tri_c = torch.empty(h, dtype=torch.int32, device=dev)
        loc_c = torch.empty((h, 3), dtype=torch.float32, device=dev)
        uv_c = torch.empty((h, 2), dtype=torch.float32, device=dev)
        if h > 0:
            _check(lib.rt_compact_scatter(_ptr(hit), n, _ptr(ws), _ptr(front), _ptr(tri), _ptr(loc), _ptr(uv),
                                          _ptr(front_c), _ptr(ray_idx), _ptr(tri_c), _ptr(loc_c), _ptr(uv_c),
                                          _stream(dev)), "rt_compact_scatter")
    return front_c, ray_idx, tri_c, loc_c, uv_c


def compact_scan(hit: torch.Tensor):
    """First half of compact_closest: (workspace, number of hits) - the host reads the total."""
    lib = get_module()
    dev = hit.device
    n = hit.numel()
    with torch.cuda.device(dev):
        ws_b = C.c_size_t()
        _check(lib.rt_compact_sizes(n, C.byref(ws_b)), "rt_compact_sizes")
        ws = torch.empty(max(ws_b.value, 256), dtype=torch.uint8, device=dev)
        total = torch.zeros(1, dtype=torch.int64, device=dev)
        _check(lib.rt_compact_scan(_ptr(hit), n, _ptr(ws), ws.numel(), _ptr(total), _stream(dev)), "rt_compact_scan")
        return ws, int(total.item())


def compact_scatter_at(hit, ws, front, tri, loc, uv, ray_base: int, ray_idx_bytes: int, front_ptr: int, ray_ptr: int,
                       tri_ptr: int, loc_ptr: int, uv_ptr: int) -> None:
    """Second half with RAW output addresses (possibly peer-GPU memory) already offset to this shard's first packed
    row; ray indices are written as ray_base + local index (rt_compact_scatter_at)."""
    dev = hit.device
    with torch.cuda.device(dev):
        _check(get_module().rt_compact_scatter_at(_ptr(hit), hit.numel(), _ptr(ws), _ptr(front), _ptr(tri), _ptr(loc),
                                                  _ptr(uv), int(ray_base), int(ray_idx_bytes), C.c_void_p(front_ptr),
                                                  C.c_void_p(ray_ptr), C.c_void_p(tri_ptr), C.c_void_p(loc_ptr),
                                                  C.c_void_p(uv_ptr), _stream(dev)), "rt_compact_scatter_at")


def allhits_window_rays(max_hits: int, budget_bytes: int | None = None) -> int:
    """Rays per all-hits launch so that the staging buffer (rays * max_hits * 16 B) stays within `budget_bytes`."""
    budget = ALLHITS_STAGING_BYTES if budget_bytes is None else int(budget_bytes)
    return max(1024, budget // (16 * max_hits))


def allhits_trace(accel_structure, origins: torch.Tensor, dirs: torch.Tensor, max_hits: int = 8, ray_first: int = 0,
                  ray_count: int = -1):
    """First half of intersects_location for one ray window: one traversal + scan -> (state for allhits_scatter_at,
    number of hits)."""
    tensor_input_check(origins, dirs)
    lib = get_module()
    blob = _blob_of(accel_structure, origins.device)
    rd, _ = make_ray_desc(origins, dirs)
    dev = origins.device
    n = _window(rd.nray, ray_first, ray_count)
    with torch.cuda.device(dev):
        st_b, ws_b = C.c_size_t(), C.c_size_t()
        _check(lib.rt_allhits_sizes(n, max_hits, C.byref(st_b), C.byref(ws_b)), "rt_allhits_sizes")
        staging = torch.empty(max(st_b.value, 16), dtype=torch.uint8, device=dev)
        ws = torch.empty(max(ws_b.value, 256), dtype=torch.uint8, device=dev)
        counts = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        total = torch.zeros(1, dtype=torch.int64, device=dev)
        if n == 0:
            return (0, max_hits, counts, staging, ws), 0
        _check(lib.rt_allhits_trace(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure, ray_first, n)), max_hits,
                                    _ptr(counts), _ptr(staging), _ptr(ws), ws.numel(), _ptr(total), _ptr(_scratch(dev)),
                                    _stream(dev)), "rt_allhits_trace")
        return (n, max_hits, counts, staging, ws), int(total.item())


def allhits_scatter_at(state, ray_base: int, ray_idx_bytes: int, loc_ptr: int, ray_ptr: int, tri_ptr: int) -> None:
    n, max_hits, counts, staging, ws = state
    dev = counts.device
    with torch.cuda.device(dev):
        _check(get_module().rt_allhits_scatter_at(n, max_hits, _ptr(counts), _ptr(staging), _ptr(ws), int(ray_base),
                                                  int(ray_idx_bytes), C.c_void_p(loc_ptr), C.c_void_p(ray_ptr),
                                                  C.c_void_p(tri_ptr), _stream(dev)), "rt_allhits_scatter_at")


def intersects_count(accel_structure, origins: torch.Tensor, dirs: torch.Tensor) -> torch.Tensor:
    """Int32[*b]: number of triangles hit with 0 < t < 1e7 (reference ops.py:152-168)."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, batch = make_ray_desc(origins, dirs)
    dev = origins.device
    with _on_device(dev):
        out = torch.empty(batch, dtype=torch.int32, device=dev)
        st = _stream(dev)
        _check(get_module().rt_trace_count(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure)), _ptr(out),
                                           _ptr(_scratch(dev, st)), st), "rt_trace_count")
    return out


def intersects_location(accel_structure, origins: torch.Tensor, dirs: torch.Tensor, max_hits: int = MAX_ANYHIT_SIZE,
                        ray_idx_base: int = 0, ray_idx_dtype=torch.int32, staging_bytes: int | None = None,
                        ray_first: int = 0, ray_count: int = -1):
    """(loc Float32[h,3], ray_idx Int32[h], tri_idx Int32[h]): up to 8 hits per ray, grouped by
    ray in ascending ray order (reference ops.py:171-192, ray.cpp:324-378) — one traversal
    instead of the reference's two.

    The reference sizes its output from a count pass; here hits are staged at max_hits * 16 B per ray during the
    single traversal, so a large batch is traced window by window (rt_trace_opts.ray_first / ray_count: no copy of
    the rays, any strides) with at most ALLHITS_STAGING_BYTES of staging alive; the windows' packed results are
    concatenated, which preserves the ray order.  Ray indices are `ray_idx_base` + the index in the flattened batch;
    `ray_first` / `ray_count` restrict the call to a slice of the batch (sharded callers)."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, _ = make_ray_desc(origins, dirs)
    dev = origins.device
    n = _window(rd.nray, ray_first, ray_count)
    rb = 8 if ray_idx_dtype == torch.int64 else 4
    per = allhits_window_rays(max_hits, staging_bytes)
    parts = []
    with torch.cuda.device(dev):
        for first in range(ray_first, ray_first + n, per):
            m = min(per, ray_first + n - first)
            state, h = allhits_trace(accel_structure, origins, dirs, max_hits, first, m)
            loc = torch.empty((h, 3), dtype=torch.float32, device=dev)
            ray_idx = torch.empty(h, dtype=ray_idx_dtype, device=dev)
            tri_idx = torch.empty(h, dtype=torch.int32, device=dev)
            if h > 0:
                allhits_scatter_at(state, ray_idx_base + first, rb, loc.data_ptr(), ray_idx.data_ptr(), tri_idx.data_ptr())
            parts.append((loc, ray_idx, tri_idx))
            del state
        if not parts:
            return (torch.empty((0, 3), dtype=torch.float32, device=dev), torch.empty(0, dtype=ray_idx_dtype, device=dev),
                    torch.empty(0, dtype=torch.int32, device=dev))
        if len(parts) == 1:
            return parts[0]
        return tuple(torch.cat([p[i] for p in parts], dim=0) for i in range(3))


def contains_parity(accel_structure, points: torch.Tensor, direction, aabb_lo, aabb_hi, active: torch.Tensor | None = None,
                    out=None, stop_when_broken: bool = False):
    """Fused core of contains_points (reference ray_optix.py:238-267): returns
    (contain Bool[*b], broken Bool[*b], flags Int32[2] = [any(inside_aabb), any(broken)]).
    With `active` (Bool[*b]) only the masked points are traced and written, in place into `out` = (contain, broken);
    `active` may be the `broken` tensor itself (the retry of ray_optix.py:272-277 without gather / scatter).
    `stop_when_broken`: the launch may end as soon as flags[1] is known to be 1 (per-point results unspecified then)."""
    tensor_input_check(points)
    blob = _blob_of(accel_structure, points.device)
    rd, batch = make_ray_desc(points, None)
    dev = points.device
    d3 = (C.c_float * 3)(*[float(x) for x in direction])
    lo3 = (C.c_float * 3)(*[float(x) for x in aabb_lo])
    hi3 = (C.c_float * 3)(*[float(x) for x in aabb_hi])
    with torch.cuda.device(dev):
        if out is None:
            if active is not None:
                raise ValueError("contains_parity: a masked call updates existing (contain, broken) tensors: pass out=")
            contain = torch.empty(batch, dtype=torch.bool, device=dev)
            broken = torch.empty(batch, dtype=torch.bool, device=dev)
        else:
            contain, broken = out
            for t in (contain, broken) + ((active,) if active is not None else ()):
                if t.dtype != torch.bool or t.device != dev or not t.is_contiguous() or t.numel() != rd.nray:
                    raise ValueError("contains_parity: masks must be contiguous bool tensors over the point batch")
        flags = torch.empty(2, dtype=torch.int32, device=dev)
        opts = trace_opts(accel_structure)
        if stop_when_broken:
            opts = _trace_opts(accel_structure, 0, -1, True)       # a private copy: the whole-batch form is a shared cached object
            opts.flags |= OPT_STOP_WHEN_BROKEN
        _check(get_module().rt_contains_parity(_ptr(blob), C.byref(rd), C.byref(opts), d3, lo3, hi3,
                                               _ptr(active), _ptr(contain), _ptr(broken), _ptr(flags), _ptr(_scratch(dev)),
                                               _stream(dev)), "rt_contains_parity")
    return contain, broken, flags


def trace_stats(accel_structure, origins: torch.Tensor, dirs: torch.Tensor, mode: str = "closest") -> dict:
    """Instrumented traversal: mean BVH8 nodes / triangles fetched per ray (roofline input)."""
    tensor_input_check(origins, dirs)
    blob = _blob_of(accel_structure, origins.device)
    rd, _ = make_ray_desc(origins, dirs)
    dev = origins.device
    with torch.cuda.device(dev):
        counters = torch.zeros(4, dtype=torch.int64, device=dev)
        _check(get_module().rt_trace_stats(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure)),
                                           {"closest": 0, "any": 1, "count": 2}[mode], _ptr(counters), _ptr(_scratch(dev)),
                                           _stream(dev)), "rt_trace_stats")
        c = counters.cpu().tolist()
    rays = max(c[2], 1)
    return dict(nodes=c[0], tris=c[1], rays=c[2], hits=c[3], nodes_per_ray=c[0] / rays, tris_per_ray=c[1] / rays,
                hit_fraction=c[3] / rays)


def closest_point(accel_structure, points: torch.Tensor, max_distance: float = float("inf"), ray_first: int = 0,
                  ray_count: int = -1, counters: torch.Tensor | None = None):
    """Closest point on the mesh for every query point (trimesh.proximity.closest_point): returns
    (closest Float32[*b,3], distance Float32[*b], tri Int32[*b], uv Float32[*b,2]) with uv = weights of the triangle's
    vertices 0 and 1.  Only triangles within `max_distance` count; a point with none (or a non-finite point, or an
    empty mesh) gets tri -1, distance +inf, closest 0, uv 0.  Equal distances go to the smaller triangle index.
    With a window [ray_first, ray_first + ray_count) of the flattened batch the outputs are 1-D over the window.
    `counters` (Int64[4] on the device, optional) selects the instrumented kernel: nodes fetched, triangles tested,
    points, points with an answer."""
    md = float(max_distance)
    if md != md or md < 0.0:
        raise ValueError(f"max_distance must be >= 0 or inf (got {max_distance})")
    rd, batch = _query_batch(points, None, ray_first, ray_count, counters)
    blob = _blob_of(accel_structure, points.device)
    dev = points.device
    with _on_device(dev):
        closest = torch.empty((*batch, 3), dtype=torch.float32, device=dev)
        distance = torch.empty(batch, dtype=torch.float32, device=dev)
        tri = torch.empty(batch, dtype=torch.int32, device=dev)
        uv = torch.empty((*batch, 2), dtype=torch.float32, device=dev)
        if tri.numel() == 0:
            return closest, distance, tri, uv
        st = _stream(dev)
        _check(get_module().rt_closest_point(_ptr(blob), C.byref(rd), C.byref(trace_opts(accel_structure, ray_first, ray_count)),
                                             md, _ptr(closest), _ptr(distance), _ptr(tri), _ptr(uv), _ptr(counters),
                                             _ptr(_scratch(dev, st)), st), "rt_closest_point")
    return closest, distance, tri, uv


def winding_moments(accel_structure) -> torch.Tensor:
    """Float32[nodes, 16]: the per-node moments rt_winding_number reads (area-weighted centroid, radius bound, sum of
    area vectors, first-moment tensor), one row per node of the blob.  Computed on first use and cached on
    the AccelStructure until its blob changes (build, refit, adopt / load)."""
    inner = getattr(accel_structure, "_inner", accel_structure)
    blob = _blob_of(inner)
    if inner.winding_moments is not None:
        return inner.winding_moments
    lib = get_module()
    # rt_winding_moments_sizes bounds the node count from the triangle count alone (for any leaf size, ~2.7x the
    # default build's); the header already gives the exact count, and the kernel checks it against the buffers.
    # Workspace: two 256-byte aligned arrays of one u32 / f32 per node.
    nn = max(int(inner.header["n_nodes"]), 1)
    mb, wb = nn * 64, 2 * (-(-nn * 4 // 256) * 256)
    dev = blob.device
    with _on_device(dev):
        moments = torch.empty((nn, 16), dtype=torch.float32, device=dev)
        ws = torch.empty(wb, dtype=torch.uint8, device=dev)
        _check(lib.rt_winding_moments(_ptr(blob), _ptr(moments), mb, _ptr(ws), wb, _stream(dev)), "rt_winding_moments")
    inner.winding_moments = moments
    return inner.winding_moments


def winding_number(accel_structure, points: torch.Tensor, beta: float = 2.0, ray_first: int = 0, ray_count: int = -1,
                   counters: torch.Tensor | None = None) -> torch.Tensor:
    """Float32[*b]: generalized winding number of every query point (sum of the triangles' signed solid angles / 4 pi,
    orientation from the face order): ~1 inside and ~0 outside a closed outward-facing mesh, fractional near holes,
    additive over nested shells.  Leaf triangles are summed exactly; a BVH subtree farther than `beta` times its radius
    adds its far-field expansion (Barill et al. 2018).  beta >= 1; beta = inf is exact.  A non-finite point gives NaN,
    an empty mesh 0.  With a window [ray_first, ray_first + ray_count) of the flattened batch the output is 1-D over the
    window.  `counters` (Int64[4] on the device, optional) selects the instrumented kernel: nodes visited, triangles
    summed exactly, points, far-field terms."""
    b = float(beta)
    if not (b >= 1.0):
        raise ValueError(f"beta must be >= 1 or inf (got {beta})")
    rd, batch = _query_batch(points, None, ray_first, ray_count, counters)
    blob = _blob_of(accel_structure, points.device)
    dev = points.device
    with _on_device(dev):
        w = torch.empty(batch, dtype=torch.float32, device=dev)
        if w.numel() == 0:
            return w
        moments = winding_moments(accel_structure)
        st = _stream(dev)
        _check(get_module().rt_winding_number(_ptr(blob), _ptr(moments), C.byref(rd),
                                              C.byref(trace_opts(accel_structure, ray_first, ray_count)), b, _ptr(w),
                                              _ptr(counters), _ptr(_scratch(dev, st)), st), "rt_winding_number")
    return w


def pseudo_normals(accel_structure) -> tuple[torch.Tensor, torch.Tensor]:
    """(normals Float32[n_tris, 24], edge_counts Int64[3]) of rt_pseudonormals: per triangle record the angle-weighted
    pseudo-normals of its vertices a, b, c and of its edges ab, ac, bc (one float4 each), with corners welded by
    equal coordinates; and the counts of boundary, non-manifold and inconsistently oriented edges, kept on the device.
    Computed on first use and cached on the AccelStructure until its blob changes (build, refit, adopt / load)."""
    inner = getattr(accel_structure, "_inner", accel_structure)
    blob = _blob_of(inner)
    if inner.pseudo_normals is not None:
        return inner.pseudo_normals
    lib = get_module()
    nt = int(inner.header["n_tris"])
    nb, wb = C.c_size_t(), C.c_size_t()
    _check(lib.rt_pseudonormals_sizes(nt, C.byref(nb), C.byref(wb)), "rt_pseudonormals_sizes")
    dev = blob.device
    with _on_device(dev):
        normals = torch.zeros((max(nt, 1), 24), dtype=torch.float32, device=dev)
        ws = torch.empty(max(wb.value, 256), dtype=torch.uint8, device=dev)
        counts = torch.empty(3, dtype=torch.int64, device=dev)
        _check(lib.rt_pseudonormals(_ptr(blob), _ptr(normals), nt * 96, _ptr(ws), ws.numel(), _ptr(counts), _stream(dev)),
               "rt_pseudonormals")
    inner.pseudo_normals = (normals[:nt], counts)
    return inner.pseudo_normals


def signed_distance_pseudonormal(accel_structure, points: torch.Tensor, ray_first: int = 0, ray_count: int = -1,
                                 counters: torch.Tensor | None = None, return_closest: bool = False):
    """Float32[*b]: distance to the surface, positive inside, with the sign of the angle-weighted pseudo-normal of the
    closest feature (Baerentzen & Aanaes 2005): one closest-point walk per point, no host sync once pseudo_normals()
    is cached.  |result| is bit for bit closest_point's distance; an exact 0 is +0; a non-finite point or an empty
    mesh gives -inf.  Batch, window and counters as closest_point.  return_closest=True returns
    (signed distance, closest, tri, uv) from the same walk, the last three exactly as closest_point's."""
    rd, batch = _query_batch(points, None, ray_first, ray_count, counters)
    blob = _blob_of(accel_structure, points.device)
    dev = points.device
    with _on_device(dev):
        sd = torch.empty(batch, dtype=torch.float32, device=dev)
        if return_closest:
            closest = torch.empty((*batch, 3), dtype=torch.float32, device=dev)
            tri = torch.empty(batch, dtype=torch.int32, device=dev)
            uv = torch.empty((*batch, 2), dtype=torch.float32, device=dev)
        if sd.numel() == 0:
            return (sd, closest, tri, uv) if return_closest else sd
        normals, _ = pseudo_normals(accel_structure)
        # an empty mesh has an empty (null) normals tensor: the kernel finds no triangle and reads no row
        nptr = _ptr(normals) if normals.numel() else _ptr(blob)
        st = _stream(dev)
        opts = C.byref(trace_opts(accel_structure, ray_first, ray_count))
        if return_closest:
            _check(get_module().rt_signed_distance_closest(_ptr(blob), nptr, C.byref(rd), opts, _ptr(sd), _ptr(closest),
                                                           _ptr(tri), _ptr(uv), _ptr(counters), _ptr(_scratch(dev, st)),
                                                           st), "rt_signed_distance_closest")
            return sd, closest, tri, uv
        _check(get_module().rt_signed_distance(_ptr(blob), nptr, C.byref(rd), opts, _ptr(sd), _ptr(counters),
                                               _ptr(_scratch(dev, st)), st), "rt_signed_distance")
    return sd


def _check_grad_inputs(dev, specs):
    """ValueError unless every (name, tensor, shape, dtype) of specs whose tensor is not None is dtype shape on dev"""
    for name, t, shape, dt in specs:
        if t is not None and (tuple(t.shape) != tuple(shape) or t.dtype != dt or t.device != dev):
            raise ValueError(f"{name} must be {dt} {tuple(shape)} on {dev}, got {t.dtype} {tuple(t.shape)} on {t.device}")


def _grad_workspace(dev, reduce: bool, sizes, workspace_bytes: int | None):
    """(workspace, its size in bytes) of a gradient call: none when it forms no vertex or transform sums, else
    workspace_bytes (default sizes(): one window for every row)"""
    if not reduce:
        return None, 0
    wb = sizes() if workspace_bytes is None else int(workspace_bytes)
    return torch.empty(max(wb, 256), dtype=torch.uint8, device=dev), wb


def distance_grad_workspace_bytes(n_points: int, n_verts: int) -> int:
    """Workspace rt_distance_grad needs to run a batch of n_points as one window."""
    wb = C.c_size_t()
    _check(get_module().rt_distance_grad_sizes(int(n_points), int(n_verts), C.byref(wb)), "rt_distance_grad_sizes")
    return wb.value


def distance_grad(points: torch.Tensor, grad_out: torch.Tensor, value: torch.Tensor, closest: torch.Tensor,
                  tri: torch.Tensor, uv: torch.Tensor, faces: torch.Tensor, n_verts: int, points_grad: bool = True,
                  vertices_grad: bool = True, workspace_bytes: int | None = None):
    """Backward of a distance (closest_point's) or signed distance (any sign mode) from the forward's outputs, with
    no BVH walk: (grad_points Float32[*b,3] or None, grad_vertices Float32[n_verts,3] or None).  With g = grad_out,
    s = the sign of value (+1 for +0), grad_points = g s (p - c) / |value| and every point adds -w_k times that to
    vertex faces[tri][k], w = (uv0, uv1, 1 - uv0 - uv1).  A point with value +-0, +-inf or NaN, or tri -1, gives 0.
    The vertex sums are a sort and a fixed-order tree (DESIGN.md §4.9): the same inputs give the same bits on every
    run.  `workspace_bytes` bounds the workspace (default: one window for the whole batch); a smaller one runs the
    batch as several point windows, whose sums are added in window order."""
    tensor_input_check(points)
    rd, batch = make_ray_desc(points, None)
    dev = points.device
    n = rd.nray
    _check_grad_inputs(dev, (("grad_out", grad_out, batch, torch.float32), ("value", value, batch, torch.float32),
                             ("closest", closest, (*batch, 3), torch.float32), ("tri", tri, batch, torch.int32),
                             ("uv", uv, (*batch, 2), torch.float32)))
    if faces.dtype != torch.int32 or faces.dim() != 2 or faces.shape[1] != 3 or faces.device != dev:
        raise ValueError("faces must be int32 [f, 3] on the points' device")
    grad_out, value, closest, tri, uv, faces = (t.contiguous() for t in (grad_out, value, closest, tri, uv, faces))
    with _on_device(dev):
        gp = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if points_grad else None
        gv = torch.empty((int(n_verts), 3), dtype=torch.float32, device=dev) if vertices_grad else None
        ws, wb = _grad_workspace(dev, vertices_grad, lambda: distance_grad_workspace_bytes(n, n_verts), workspace_bytes)
        _check(get_module().rt_distance_grad(C.byref(rd), C.byref(trace_opts()), _ptr(grad_out), _ptr(value),
                                             _ptr(closest), _ptr(tri), _ptr(uv), _ptr(faces), faces.shape[0],
                                             int(n_verts), _ptr(gp), _ptr(gv), _ptr(ws), wb, _stream(dev)),
               "rt_distance_grad")
    return gp, gv


def ray_grad_workspace_bytes(n_rows: int, n_verts: int) -> int:
    """Workspace rt_ray_grad needs to run n_rows hit rows as one window."""
    wb = C.c_size_t()
    _check(get_module().rt_ray_grad_sizes(int(n_rows), int(n_verts), C.byref(wb)), "rt_ray_grad_sizes")
    return wb.value


def ray_grad(origins: torch.Tensor, dirs: torch.Tensor, tri: torch.Tensor, grad_loc: torch.Tensor | None,
             grad_uv: torch.Tensor | None, vertices: torch.Tensor, faces: torch.Tensor,
             ray_idx: torch.Tensor | None = None, origins_grad: bool = True, directions_grad: bool = True,
             vertices_grad: bool = True, workspace_bytes: int | None = None):
    """Backward of the hit locations (and barycentrics) of intersects_closest, compact_closest or intersects_location,
    with no BVH walk: (grad_origins Float32[*b,3] or None, grad_directions Float32[*b,3] or None, grad_vertices
    Float32[n_verts,3] or None).  Row i is the hit of triangle tri[i] by ray ray_idx[i] (None: ray i, one row per
    ray) of the flattened batch; grad_loc Float32[h,3] and grad_uv Float32[h,2] are the incoming gradients (None: 0).
    Each row recomputes its hit with the Moeller-Trumbore sequence of DESIGN.md §4.10 from `vertices` and `faces`;
    the rows of one ray must be contiguous.  A row with no triangle, a degenerate triangle or a non-finite value
    gives 0.  Deterministic to the bit: per-ray sums in row order, vertex sums through the sort and fixed tree of
    distance_grad.  `workspace_bytes` bounds the workspace (default: one window for all rows); a smaller one runs
    the rows as several windows, whose vertex sums are added in window order."""
    tensor_input_check(origins, dirs, vertices)
    rd, batch = make_ray_desc(origins, dirs)
    dev = origins.device
    h = tri.shape[0] if tri.dim() == 1 else -1
    if ray_idx is None and h != rd.nray:
        raise ValueError(f"tri must have one row per ray ({rd.nray}) without ray_idx, got {tuple(tri.shape)}")
    _check_grad_inputs(dev, (("tri", tri, (h,), torch.int32), ("grad_loc", grad_loc, (h, 3), torch.float32),
                             ("grad_uv", grad_uv, (h, 2), torch.float32), ("ray_idx", ray_idx, (h,), torch.int32)))
    if vertices.dim() != 2 or vertices.shape[1] != 3 or vertices.device != dev:
        raise ValueError("vertices must be float32 [n, 3] on the rays' device")
    if faces.dtype != torch.int32 or faces.dim() != 2 or faces.shape[1] != 3 or faces.device != dev:
        raise ValueError("faces must be int32 [f, 3] on the rays' device")
    tri, grad_loc, grad_uv, ray_idx, vertices, faces = (None if t is None else t.contiguous() for t in
                                                        (tri, grad_loc, grad_uv, ray_idx, vertices, faces))
    n_verts = vertices.shape[0]
    with _on_device(dev):
        go = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if origins_grad else None
        gd = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if directions_grad else None
        gv = torch.empty((n_verts, 3), dtype=torch.float32, device=dev) if vertices_grad else None
        ws, wb = _grad_workspace(dev, vertices_grad, lambda: ray_grad_workspace_bytes(h, n_verts), workspace_bytes)
        _check(get_module().rt_ray_grad(C.byref(rd), C.byref(trace_opts()), h, _ptr(ray_idx), _ptr(tri), _ptr(grad_loc),
                                        _ptr(grad_uv), _ptr(vertices), n_verts, _ptr(faces), faces.shape[0], _ptr(go),
                                        _ptr(gd), _ptr(gv), _ptr(ws), wb, _stream(dev)), "rt_ray_grad")
    return go, gd, gv


def edge_counts(accel_structure) -> tuple[int, int, int]:
    """(boundary, non-manifold, inconsistent) edges of the welded surface (one host sync)."""
    return tuple(int(x) for x in pseudo_normals(accel_structure)[1].tolist())


def host_closest(accel_structure, origins_host: torch.Tensor, dirs_host: torch.Tensor, out: dict | None = None,
                 work: torch.Tensor | None = None, stream_compaction: bool = False):
    """End-to-end closest hit with HOST (ideally pinned) buffers: rt_host_trace_closest pipelines
    H2D copy, traversal and D2H copy over ray chunks.  origins_host may be [n,3] or a single
    [3]/[1,3] origin shared by all rays.  Returns a dict of host tensors (dense 5-tuple fields).
    stream_compaction=True (rt_host_trace_closest_compact) compacts on the device and copies back only the hit
    mask and the packed rows: the dict then holds hit[*b], n_hit and front / ray_idx / tri / loc / uv whose first
    n_hit rows are valid (views `*_c` are added for convenience)."""
    lib = get_module()
    blob = _blob_of(accel_structure)
    dev = blob.device
    d = dirs_host
    if d.is_cuda or d.dtype != torch.float32 or not d.is_contiguous() or d.shape[-1] != 3:
        raise ValueError("dirs_host must be a contiguous float32 host tensor [*b,3]")
    n = d.numel() // 3
    o = origins_host
    if o.is_cuda or o.dtype != torch.float32 or not o.is_contiguous():
        raise ValueError("origins_host must be a contiguous float32 host tensor")
    bcast = 1 if o.numel() == 3 else 0
    if not bcast and o.numel() != 3 * n:
        raise ValueError("origins_host must hold 3 or 3*nray floats")
    batch = tuple(d.shape[:-1])
    if work is None and out is not None:
        work = out.get("_work")
    if out is None:
        pin = torch.cuda.is_available()
        rows = (n,) if stream_compaction else batch
        out = dict(hit=torch.empty(batch, dtype=torch.bool, pin_memory=pin),
                   front=torch.empty(rows, dtype=torch.bool, pin_memory=pin),
                   tri=torch.empty(rows, dtype=torch.int32, pin_memory=pin),
                   loc=torch.empty((*rows, 3), dtype=torch.float32, pin_memory=pin),
                   uv=torch.empty((*rows, 2), dtype=torch.float32, pin_memory=pin))
        if stream_compaction:
            out["ray_idx"] = torch.empty(rows, dtype=torch.int32, pin_memory=pin)
    with torch.cuda.device(dev):
        wb = C.c_size_t()
        _check(lib.rt_host_closest_sizes(n, C.byref(wb)), "rt_host_closest_sizes")
        if work is None or work.numel() < wb.value:
            work = torch.empty(wb.value, dtype=torch.uint8, device=dev)
        torch.cuda.current_stream(dev).synchronize()   # blob must be complete before the private streams read it
        opts = trace_opts(accel_structure)
        if stream_compaction:
            nh = C.c_int64(0)
            _check(lib.rt_host_trace_closest_compact(_ptr(blob), n, C.c_void_p(o.data_ptr()), bcast, C.c_void_p(d.data_ptr()),
                                                     C.byref(opts), C.c_void_p(out["hit"].data_ptr()),
                                                     C.c_void_p(out["front"].data_ptr()), C.c_void_p(out["ray_idx"].data_ptr()),
                                                     C.c_void_p(out["tri"].data_ptr()), C.c_void_p(out["loc"].data_ptr()),
                                                     C.c_void_p(out["uv"].data_ptr()), C.byref(nh), _ptr(work), work.numel()),
                   "rt_host_trace_closest_compact")
            h = int(nh.value)
            out["n_hit"] = h
            for k in ("front", "ray_idx", "tri", "loc", "uv"):
                out[k + "_c"] = out[k][:h]
        else:
            _check(lib.rt_host_trace_closest(_ptr(blob), n, C.c_void_p(o.data_ptr()), bcast, C.c_void_p(d.data_ptr()),
                                             C.byref(opts), C.c_void_p(out["hit"].data_ptr()),
                                             C.c_void_p(out["front"].data_ptr()), C.c_void_p(out["tri"].data_ptr()),
                                             C.c_void_p(out["loc"].data_ptr()), C.c_void_p(out["uv"].data_ptr()), _ptr(work),
                                             work.numel()), "rt_host_trace_closest")
    out["_work"] = work
    return out


def sort_pairs_u64(keys: torch.Tensor, vals: torch.Tensor):
    """In-place onesweep radix sort of (uint64 keys as int64 storage, int32 values) — exposed for tests."""
    lib = get_module()
    dev = keys.device
    n = keys.numel()
    with torch.cuda.device(dev):
        wb = C.c_size_t()
        _check(lib.rt_sort_sizes(n, C.byref(wb)), "rt_sort_sizes")
        ws = torch.empty(max(wb.value, 256), dtype=torch.uint8, device=dev)
        _check(lib.rt_sort_pairs_u64(_ptr(keys), _ptr(vals), n, _ptr(ws), ws.numel(), _stream(dev)), "rt_sort_pairs_u64")
    return keys, vals


# ------------------------------------------------------------------ instanced scenes (DESIGN.md §4.11)
SCENE_CLOSEST, SCENE_ANY, SCENE_COUNT = 0, 1, 2


def scene_prepare(blobs: list, inst_mesh: torch.Tensor, transforms: torch.Tensor, device) -> tuple[torch.Tensor, AccelStructure]:
    """rt_scene_prepare + rt_bvh_build: (scene table, top-level AccelStructure) for the member blobs (device uint8
    tensors), the host int32 [I] mesh indices and the host float32 [I,3,4] object->world transforms.  Raises ValueError
    for a mesh index out of range, a non-finite or singular transform, or a blob on another device."""
    lib = get_module()
    dev = torch.device(device)
    for b in blobs:
        if not b.is_cuda or b.device != dev:
            raise ValueError(f"every mesh of a scene must live on {dev} (one is on {b.device})")
    inst_mesh = inst_mesh.to(torch.int32).contiguous()
    transforms = transforms.to(torch.float32).contiguous()
    n_inst, n_meshes = inst_mesh.numel(), len(blobs)
    tb = C.c_size_t()
    _check(lib.rt_scene_prepare_sizes(n_meshes, n_inst, C.byref(tb)), "rt_scene_prepare_sizes")
    addrs = (C.c_void_p * max(n_meshes, 1))(*[b.data_ptr() for b in blobs])
    with torch.cuda.device(dev):
        table = torch.empty(tb.value, dtype=torch.uint8, device=dev)
        tv = torch.empty((2 * n_inst, 3), dtype=torch.float32, device=dev)
        tf = torch.empty((n_inst, 3), dtype=torch.int32, device=dev)
        _check(lib.rt_scene_prepare(n_meshes, addrs, n_inst, C.c_void_p(inst_mesh.data_ptr()),
                                    C.c_void_p(transforms.data_ptr()), _ptr(table), table.numel(), _ptr(tv), _ptr(tf),
                                    _stream(dev)), "rt_scene_prepare")
        tlas = AccelStructure().build(tv, tf)
    return table, tlas


def scene_trace(table: torch.Tensor, tlas: AccelStructure, origins: torch.Tensor, dirs: torch.Tensor, mode: int,
                tmax: float = TMAX_DEFAULT, ray_first: int = 0, ray_count: int = -1):
    """rt_scene_trace.  closest: (hit, front, inst, tri, loc, uv); any: hit; count: count — shaped like the batch, or
    1-D over the window [ray_first, ray_first + ray_count)."""
    rd, batch = _query_batch(origins, dirs, ray_first, ray_count, table=table)
    dev = origins.device
    opts = TraceOpts()
    opts.tmax = float(tmax)
    opts.ray_first, opts.ray_count = int(ray_first), max(int(ray_count), 0)
    with _on_device(dev):
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)   # noqa: E731
        if mode == SCENE_CLOSEST:
            out = (e(batch, torch.bool), e(batch, torch.bool), e(batch, torch.int32), e(batch, torch.int32),
                   e((*batch, 3), torch.float32), e((*batch, 2), torch.float32))
            ptrs = (out[0], out[1], out[2], out[3], out[4], out[5], None)
        elif mode == SCENE_ANY:
            out = e(batch, torch.bool)
            ptrs = (out, None, None, None, None, None, None)
        else:
            out = e(batch, torch.int32)
            ptrs = (None, None, None, None, None, None, out)
        n = ptrs[0].numel() if ptrs[0] is not None else ptrs[6].numel()
        if n > 0:
            _check(get_module().rt_scene_trace(_ptr(table), _ptr(tlas.blob), C.byref(rd), C.byref(opts), int(mode),
                                               *[_ptr(p) for p in ptrs], _stream(dev)), "rt_scene_trace")
    return out


# ------------------------------------------------------------------ point queries on instanced scenes (DESIGN.md §4.12)
def scene_point_prepare(table: torch.Tensor, n_inst: int) -> torch.Tensor:
    """rt_scene_point_prepare: the side array (uint8 on the table's device) of the point queries: per instance a lower
    bound on the smallest singular value of its A and the margins of the instance walk's world bound."""
    lib = get_module()
    sb = C.c_size_t()
    _check(lib.rt_scene_point_sizes(int(n_inst), C.byref(sb)), "rt_scene_point_sizes")
    dev = table.device
    with _on_device(dev):
        side = torch.zeros(sb.value, dtype=torch.uint8, device=dev)
        _check(lib.rt_scene_point_prepare(_ptr(table), int(n_inst), _ptr(side), side.numel(), _stream(dev)),
               "rt_scene_point_prepare")
    return side


def scene_closest_point(table: torch.Tensor, tlas: AccelStructure, side: torch.Tensor, points: torch.Tensor,
                        max_distance: float = float("inf"), ray_first: int = 0, ray_count: int = -1):
    """rt_scene_closest_point: (closest Float32[*b,3], distance Float32[*b], inst Int32[*b], tri Int32[*b],
    uv Float32[*b,2]) over every instance, the key (d2, inst, tri) minimised; misses give inst = tri = -1, distance
    inf, closest and uv 0.  1-D over the window [ray_first, ray_first + ray_count) when one is given."""
    md = float(max_distance)
    if md != md or md < 0.0:
        raise ValueError(f"max_distance must be >= 0 or inf (got {max_distance})")
    rd, batch = _query_batch(points, None, ray_first, ray_count, table=table)
    opts = trace_opts(None, ray_first, ray_count)
    dev = points.device
    with _on_device(dev):
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)   # noqa: E731
        out = (e((*batch, 3), torch.float32), e(batch, torch.float32), e(batch, torch.int32), e(batch, torch.int32),
               e((*batch, 2), torch.float32))
        if out[1].numel() > 0:
            _check(get_module().rt_scene_closest_point(_ptr(table), _ptr(tlas.blob), _ptr(side), C.byref(rd),
                                                       C.byref(opts), md, *[_ptr(t) for t in out], _stream(dev)),
                   "rt_scene_closest_point")
    return out


def scene_signed_distance(table: torch.Tensor, tlas: AccelStructure, side: torch.Tensor, normals_table: torch.Tensor,
                          points: torch.Tensor, ray_first: int = 0, ray_count: int = -1, return_closest: bool = False):
    """rt_scene_signed_distance: Float32[*b], positive inside by the world pseudo-normal of the closest feature, -inf
    for a point without answer; return_closest=True returns (signed distance, closest, inst, tri, uv) from the same
    walk.  `normals_table`: int64 device tensor of each mesh's pseudo-normal rows address."""
    rd, batch = _query_batch(points, None, ray_first, ray_count, table=table)
    opts = trace_opts(None, ray_first, ray_count)
    dev = points.device
    with _on_device(dev):
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)   # noqa: E731
        sd = e(batch, torch.float32)
        extra = ((e((*batch, 3), torch.float32), e(batch, torch.int32), e(batch, torch.int32),
                  e((*batch, 2), torch.float32)) if return_closest else (None, None, None, None))
        if sd.numel() > 0:
            _check(get_module().rt_scene_signed_distance(_ptr(table), _ptr(tlas.blob), _ptr(side), _ptr(normals_table),
                                                         C.byref(rd), C.byref(opts), _ptr(sd),
                                                         *[_ptr(t) for t in extra], _stream(dev)),
                   "rt_scene_signed_distance")
    return (sd, *extra) if return_closest else sd


def scene_distance_grad(points: torch.Tensor, grad_out: torch.Tensor, value: torch.Tensor, closest: torch.Tensor,
                        tri: torch.Tensor, uv: torch.Tensor, n_faces: int) -> torch.Tensor:
    """grad_points of a scene distance or signed distance: rt_distance_grad without vertex gradient, g s (p - c) /
    |value| per point, 0 where value is +-0, +-inf or NaN or tri is outside [0, n_faces)."""
    tensor_input_check(points)
    rd, batch = make_ray_desc(points, None)
    dev = points.device
    grad_out, value, closest, tri, uv = (t.contiguous() for t in (grad_out, value, closest, tri, uv))
    with _on_device(dev):
        gp = torch.empty((*batch, 3), dtype=torch.float32, device=dev)
        if gp.numel() > 0:
            _check(get_module().rt_distance_grad(C.byref(rd), C.byref(trace_opts()), _ptr(grad_out), _ptr(value),
                                                 _ptr(closest), _ptr(tri), _ptr(uv), None, int(n_faces), 0, _ptr(gp),
                                                 None, None, 0, _stream(dev)), "rt_distance_grad")
    return gp


# ------------------------------------------------------------------ gradients on instanced scenes (DESIGN.md §4.13)
SCENE_GRAD_TRANSFORMS, SCENE_GRAD_VERTICES = 1, 2


def scene_members(members: list) -> tuple[torch.Tensor, int]:
    """The device member table of rt_scene_ray_grad / rt_scene_distance_grad for [(vertices Float32[v,3], faces
    Int32[f,3]), ...] (contiguous, on one CUDA device; the caller keeps them alive while the table is used): int64
    [M, 5] rows (vertices address, faces address, v, f, vertex base), and the total vertex count.  A member's vertex
    base is the sum of the vertex counts before it."""
    rows, base = [], 0
    for v, f in members:
        if v.dtype != torch.float32 or not v.is_contiguous() or f.dtype != torch.int32 or not f.is_contiguous():
            raise ValueError("member vertices must be contiguous float32 [v,3] and faces contiguous int32 [f,3]")
        rows.append([v.data_ptr(), f.data_ptr(), v.shape[0], f.shape[0], base])
        base += v.shape[0]
    dev = members[0][0].device if members else torch.device("cuda", torch.cuda.current_device())
    return torch.tensor(rows or [[0] * 5], dtype=torch.int64).to(dev), base


def scene_grad_workspace_bytes(n_rows: int, n_inst: int, n_verts: int, outputs: int) -> int:
    """Workspace rt_scene_ray_grad / rt_scene_distance_grad need to run n_rows rows as one window; `outputs` =
    SCENE_GRAD_TRANSFORMS | SCENE_GRAD_VERTICES as requested."""
    wb = C.c_size_t()
    _check(get_module().rt_scene_grad_sizes(int(n_rows), int(n_inst), int(n_verts), int(outputs), C.byref(wb)),
           "rt_scene_grad_sizes")
    return wb.value


def _scene_grad_outputs(dev, n_inst: int, n_verts: int, n_rows: int, transforms_grad: bool, vertices_grad: bool,
                        workspace_bytes: int | None):
    gt = torch.empty((n_inst, 3, 4), dtype=torch.float32, device=dev) if transforms_grad else None
    gv = torch.empty((n_verts, 3), dtype=torch.float32, device=dev) if vertices_grad else None
    outputs = (SCENE_GRAD_TRANSFORMS if transforms_grad else 0) | (SCENE_GRAD_VERTICES if vertices_grad else 0)
    ws, wb = _grad_workspace(dev, outputs != 0, lambda: scene_grad_workspace_bytes(n_rows, n_inst, n_verts, outputs),
                             workspace_bytes)
    return gt, gv, ws, wb


def _scene_member_args(table: torch.Tensor, n_inst: int, members: torch.Tensor, n_verts: int, dev):
    if table.device != dev or members.device != dev or members.dtype != torch.int64 or members.dim() != 2:
        raise ValueError(f"the scene table and the member table must be on {dev}")
    return _ptr(table), int(n_inst), _ptr(members), members.shape[0], int(n_verts)


def scene_ray_grad(table: torch.Tensor, n_inst: int, members: torch.Tensor, n_verts: int, origins: torch.Tensor,
                   dirs: torch.Tensor, inst: torch.Tensor, tri: torch.Tensor, grad_loc: torch.Tensor | None,
                   grad_uv: torch.Tensor | None, ray_idx: torch.Tensor | None = None, origins_grad: bool = True,
                   directions_grad: bool = True, transforms_grad: bool = True, vertices_grad: bool = True,
                   workspace_bytes: int | None = None):
    """Backward of RayMeshScene.intersects_closest's loc and uv (rt_scene_ray_grad): (grad_origins Float32[*b,3],
    grad_directions Float32[*b,3], grad_transforms Float32[I,3,4], grad_vertices Float32[n_verts,3]), each None when
    not asked for.  Row i is the hit of (inst[i], tri[i]) by ray ray_idx[i] (None: ray i) of the flattened batch;
    `members` and n_verts come from scene_members.  Each row recomputes its hit on the world triangle (DESIGN.md
    §4.13); sums are deterministic to the bit.  `workspace_bytes` bounds the workspace (default: one window)."""
    tensor_input_check(origins, dirs)
    rd, batch = make_ray_desc(origins, dirs)
    dev = origins.device
    h = tri.shape[0] if tri.dim() == 1 else -1
    if ray_idx is None and h != rd.nray:
        raise ValueError(f"tri must have one row per ray ({rd.nray}) without ray_idx, got {tuple(tri.shape)}")
    _check_grad_inputs(dev, (("inst", inst, (h,), torch.int32), ("tri", tri, (h,), torch.int32),
                             ("grad_loc", grad_loc, (h, 3), torch.float32), ("grad_uv", grad_uv, (h, 2), torch.float32),
                             ("ray_idx", ray_idx, (h,), torch.int32)))
    scene = _scene_member_args(table, n_inst, members, n_verts, dev)
    inst, tri, grad_loc, grad_uv, ray_idx = (None if t is None else t.contiguous() for t in
                                             (inst, tri, grad_loc, grad_uv, ray_idx))
    with _on_device(dev):
        go = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if origins_grad else None
        gd = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if directions_grad else None
        gt, gv, ws, wb = _scene_grad_outputs(dev, n_inst, n_verts, h, transforms_grad, vertices_grad, workspace_bytes)
        _check(get_module().rt_scene_ray_grad(*scene, C.byref(rd), C.byref(trace_opts()), h, _ptr(ray_idx), _ptr(inst),
                                              _ptr(tri), _ptr(grad_loc), _ptr(grad_uv), _ptr(go), _ptr(gd), _ptr(gt),
                                              _ptr(gv), _ptr(ws), wb, _stream(dev)), "rt_scene_ray_grad")
    return go, gd, gt, gv


def scene_point_grad(table: torch.Tensor, n_inst: int, members: torch.Tensor, n_verts: int, points: torch.Tensor,
                     grad_out: torch.Tensor, value: torch.Tensor, closest: torch.Tensor, inst: torch.Tensor,
                     tri: torch.Tensor, uv: torch.Tensor, points_grad: bool = True, transforms_grad: bool = True,
                     vertices_grad: bool = True, workspace_bytes: int | None = None):
    """Backward of RayMeshScene.closest_point's distance or signed_distance (rt_scene_distance_grad) from the forward's
    outputs: (grad_points Float32[*b,3], grad_transforms Float32[I,3,4], grad_vertices Float32[n_verts,3]), each None
    when not asked for (DESIGN.md §4.13)."""
    tensor_input_check(points)
    rd, batch = make_ray_desc(points, None)
    dev = points.device
    _check_grad_inputs(dev, (("grad_out", grad_out, batch, torch.float32), ("value", value, batch, torch.float32),
                             ("closest", closest, (*batch, 3), torch.float32), ("inst", inst, batch, torch.int32),
                             ("tri", tri, batch, torch.int32), ("uv", uv, (*batch, 2), torch.float32)))
    scene = _scene_member_args(table, n_inst, members, n_verts, dev)
    grad_out, value, closest, inst, tri, uv = (t.contiguous() for t in (grad_out, value, closest, inst, tri, uv))
    with _on_device(dev):
        gp = torch.empty((*batch, 3), dtype=torch.float32, device=dev) if points_grad else None
        gt, gv, ws, wb = _scene_grad_outputs(dev, n_inst, n_verts, rd.nray, transforms_grad, vertices_grad,
                                             workspace_bytes)
        _check(get_module().rt_scene_distance_grad(*scene, C.byref(rd), C.byref(trace_opts()), _ptr(grad_out),
                                                   _ptr(value), _ptr(closest), _ptr(inst), _ptr(tri), _ptr(uv), _ptr(gp),
                                                   _ptr(gt), _ptr(gv), _ptr(ws), wb, _stream(dev)),
               "rt_scene_distance_grad")
    return gp, gt, gv
