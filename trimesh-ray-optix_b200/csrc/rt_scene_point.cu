// rt_scene_point.cu — closest point and pseudo-normal signed distance on instanced scenes (DESIGN.md §4.12).
//
// rt_scene_point_prepare: one thread per instance (k_scene_point_prepare) writes the side array of the point queries,
// a lower bound on the smallest singular value of the instance's A and the margins of its world bound, from the
// scene table and its meshes' header boxes alone.
// rt_scene_closest_point / rt_scene_signed_distance: one thread per point (k_scene_point) walks the top-level tree with
// point_step (world slot bounds, padded instance boxes at the leaves), and every instance within reach with its own
// tree (object-space slot bounds carried to world, world triangles at the leaves).  The answer is the minimum of the
// total order (d2, inst, prim), so the host simulator under tests/scene/, a brute-force loop and the flattened mesh
// give the same bits.
#include "rt_api.h"
#include "rt_scene.cuh"

namespace rt {

constexpr int kScenePointThreads = 128;

__global__ void __launch_bounds__(128) k_scene_point_prepare(const uint8_t* table, uint32_t n_inst, ScenePointSide* side) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inst) return;
    const SceneView sv = scene_view(table);
    const SceneInst s = sv.inst[i];
    side[i] = prepare_point_side(reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]), s);
}

struct ScenePointParams {
    const uint8_t* table;
    const uint8_t* tlas;
    const ScenePointSide* side;
    const uint64_t* normals;     // signed distance: the rt_pseudonormals rows of each mesh
    rt_ray_desc points;
    int64_t first, n;            // window [first, first + n) of the batch; outputs indexed by (r - first)
    float max_d2;
    float* closest;
    float* distance;
    int32_t* inst;
    int32_t* tri;
    float* uv;
    float* signed_distance;
};

struct ScenePointStack {
    PointStackEntry e[kMaxDepth];
    __device__ __forceinline__ void push(int sp, const PointStackEntry& v) { e[sp] = v; }
    __device__ __forceinline__ void pop(int sp, PointStackEntry& v) { v = e[sp]; }
};

// SIGNED: write the signed distance; CLOSEST: write closest, inst, tri and uv (and the distance when not SIGNED).
template <bool SIGNED, bool CLOSEST>
__global__ void __launch_bounds__(kScenePointThreads) k_scene_point(const __grid_constant__ ScenePointParams p) {
    const int64_t i = (int64_t)blockIdx.x * kScenePointThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t o = scene_offset(p.points.shape, p.points.o_stride, p.first + i);
    const int64_t os = p.points.o_stride[3];
    const rt_blob_header* th = reinterpret_cast<const rt_blob_header*>(p.tlas);
    ScenePointStack top, below;
    SceneTopSpace<ScenePointStack> sp{scene_view(p.table), p.side, &below};
    PointTrav t;
    point_init(t, p.points.origins[o], p.points.origins[o + os], p.points.origins[o + 2 * os], p.max_d2);
    NoStats st;
    while (!point_step(p.tlas + th->nodes_offset, p.tlas + th->tris_offset, t, st, top, sp)) {}
    if (sp.inst >= 0) {
        float v[9];
        const PointHit h = scene_point_attr(sp.sv, sp.inst, sp.slot, t.x, t.y, t.z, v);
        const float d = fsqrt(t.best);
        if (SIGNED) {
            const SceneInst& s = sp.sv.inst[sp.inst];
            const uint8_t* normals = reinterpret_cast<const uint8_t*>(p.normals[s.mesh]);
            p.signed_distance[i] = scene_pseudonormal_sign(s, normals, sp.slot, h, t.x, t.y, t.z, v, d);
        } else {
            p.distance[i] = d;
        }
        if (CLOSEST) {
            p.closest[3 * i] = h.cx; p.closest[3 * i + 1] = h.cy; p.closest[3 * i + 2] = h.cz;
            p.inst[i] = sp.inst; p.tri[i] = sp.prim;
            p.uv[2 * i] = h.w0; p.uv[2 * i + 1] = h.w1;
        }
    } else {
        if (SIGNED) p.signed_distance[i] = as_float(0xff800000u);
        else p.distance[i] = as_float(0x7f800000u);
        if (CLOSEST) {
            p.closest[3 * i] = 0.0f; p.closest[3 * i + 1] = 0.0f; p.closest[3 * i + 2] = 0.0f;
            p.inst[i] = -1; p.tri[i] = -1;
            p.uv[2 * i] = 0.0f; p.uv[2 * i + 1] = 0.0f;
        }
    }
}

}  // namespace rt

using namespace rt;

extern "C" int rt_scene_point_sizes(int64_t n_inst, size_t* side_bytes) {
    RT_REQUIRE(n_inst >= 0 && n_inst <= ((int64_t)1 << 30) && side_bytes, RT_ERR_INVALID, "rt_scene_point_sizes: bad arguments");
    *side_bytes = align_up_sz((size_t)(n_inst > 0 ? n_inst : 1) * sizeof(ScenePointSide), 256);
    return RT_OK;
}

extern "C" int rt_scene_point_prepare(const void* table, int64_t n_inst, void* side, size_t side_bytes, void* stream) {
    const char* fn = "rt_scene_point_prepare";
    size_t need = 0;
    RT_REQUIRE(rt_scene_point_sizes(n_inst, &need) == RT_OK, RT_ERR_INVALID, "%s: bad instance count", fn);
    RT_REQUIRE(table != nullptr && ((uintptr_t)table & 255) == 0, RT_ERR_INVALID, "%s: table null or not 256-byte aligned", fn);
    RT_REQUIRE(side != nullptr && ((uintptr_t)side & 15) == 0, RT_ERR_INVALID, "%s: side null or not 16-byte aligned", fn);
    RT_REQUIRE(side_bytes >= need, RT_ERR_SIZE, "%s: side array %zu < %zu bytes", fn, side_bytes, need);
    if (n_inst == 0) return RT_OK;
    k_scene_point_prepare<<<(unsigned)((n_inst + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint8_t*>(table), (uint32_t)n_inst, reinterpret_cast<ScenePointSide*>(side));
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

// Checks shared by both queries and the batch part of the launch parameters; *count = points in the window.
static int scene_point_params(const char* fn, const void* table, const void* tlas_blob, const void* side,
                              const rt_ray_desc* points, const rt_trace_opts* opts, ScenePointParams& p, int64_t* count) {
    RT_REQUIRE(table != nullptr && ((uintptr_t)table & 255) == 0, RT_ERR_INVALID, "%s: table null or not 256-byte aligned", fn);
    RT_REQUIRE(tlas_blob != nullptr && ((uintptr_t)tlas_blob & 15) == 0, RT_ERR_INVALID,
               "%s: top-level blob null or not 16-byte aligned", fn);
    RT_REQUIRE(side != nullptr && ((uintptr_t)side & 15) == 0, RT_ERR_INVALID, "%s: side null or not 16-byte aligned", fn);
    RT_REQUIRE(points != nullptr, RT_ERR_INVALID, "%s: null point descriptor", fn);
    RT_REQUIRE(points->nray >= 0 && points->shape[3] == 3, RT_ERR_INVALID, "%s: point batch must be [*b, 3]", fn);
    RT_REQUIRE(points->shape[0] >= 0 && points->shape[1] >= 0 && points->shape[2] >= 0 &&
                   points->shape[0] * points->shape[1] * points->shape[2] == points->nray,
               RT_ERR_INVALID, "%s: nray %lld does not match shape", fn, (long long)points->nray);
    static const rt_trace_opts kDefaults = {};
    const rt_trace_opts& o = opts ? *opts : kDefaults;
    RT_REQUIRE(o.ray_first >= 0 && o.ray_first <= points->nray, RT_ERR_INVALID, "%s: ray_first %lld outside [0, %lld]", fn,
               (long long)o.ray_first, (long long)points->nray);
    const int64_t n = o.ray_count <= 0 ? points->nray - o.ray_first : o.ray_count;
    RT_REQUIRE(n <= points->nray - o.ray_first, RT_ERR_INVALID, "%s: window [%lld, +%lld) exceeds the batch of %lld", fn,
               (long long)o.ray_first, (long long)n, (long long)points->nray);
    *count = n;
    if (n == 0) return RT_OK;
    RT_REQUIRE(points->origins != nullptr, RT_ERR_INVALID, "%s: null points", fn);
    RT_REQUIRE((n + kScenePointThreads - 1) / kScenePointThreads < ((int64_t)1 << 31), RT_ERR_INVALID,
               "%s: batch of %lld points too large for one launch", fn, (long long)n);
    p = ScenePointParams{};
    p.table = reinterpret_cast<const uint8_t*>(table);
    p.tlas = reinterpret_cast<const uint8_t*>(tlas_blob);
    p.side = reinterpret_cast<const ScenePointSide*>(side);
    p.points = *points;
    p.first = o.ray_first;
    p.n = n;
    return RT_OK;
}

extern "C" int rt_scene_closest_point(const void* table, const void* tlas_blob, const void* side, const rt_ray_desc* points,
                                      const rt_trace_opts* opts, float max_distance, float* closest, float* distance,
                                      int32_t* inst_idx, int32_t* tri_idx, float* uv, void* stream) {
    const char* fn = "rt_scene_closest_point";
    RT_REQUIRE(!(max_distance != max_distance) && max_distance >= 0.0f, RT_ERR_INVALID,
               "%s: max_distance must be >= 0 or +inf (got %g)", fn, (double)max_distance);
    ScenePointParams p;
    int64_t count = 0;
    const int rc = scene_point_params(fn, table, tlas_blob, side, points, opts, p, &count);
    if (rc != RT_OK || count == 0) return rc;
    RT_REQUIRE(closest && distance && inst_idx && tri_idx && uv, RT_ERR_INVALID, "%s: null output", fn);
    p.max_d2 = fmul(max_distance, max_distance);
    p.closest = closest; p.distance = distance; p.inst = inst_idx; p.tri = tri_idx; p.uv = uv;
    k_scene_point<false, true><<<(unsigned)((count + kScenePointThreads - 1) / kScenePointThreads), kScenePointThreads, 0,
                                 (cudaStream_t)stream>>>(p);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

extern "C" int rt_scene_signed_distance(const void* table, const void* tlas_blob, const void* side, const void* normals_table,
                                        const rt_ray_desc* points, const rt_trace_opts* opts, float* signed_distance,
                                        float* closest, int32_t* inst_idx, int32_t* tri_idx, float* uv, void* stream) {
    const char* fn = "rt_scene_signed_distance";
    RT_REQUIRE(normals_table != nullptr && ((uintptr_t)normals_table & 7) == 0, RT_ERR_INVALID,
               "%s: normals table null or not 8-byte aligned", fn);
    const bool with_closest = closest || inst_idx || tri_idx || uv;
    RT_REQUIRE(!with_closest || (closest && inst_idx && tri_idx && uv), RT_ERR_INVALID,
               "%s: closest, inst_idx, tri_idx and uv must be all NULL or all set", fn);
    ScenePointParams p;
    int64_t count = 0;
    const int rc = scene_point_params(fn, table, tlas_blob, side, points, opts, p, &count);
    if (rc != RT_OK || count == 0) return rc;
    RT_REQUIRE(signed_distance != nullptr, RT_ERR_INVALID, "%s: null output", fn);
    p.max_d2 = as_float(0x7f800000u);
    p.normals = reinterpret_cast<const uint64_t*>(normals_table);
    p.signed_distance = signed_distance;
    p.closest = closest; p.inst = inst_idx; p.tri = tri_idx; p.uv = uv;
    const unsigned grid = (unsigned)((count + kScenePointThreads - 1) / kScenePointThreads);
    if (with_closest)
        k_scene_point<true, true><<<grid, kScenePointThreads, 0, (cudaStream_t)stream>>>(p);
    else
        k_scene_point<true, false><<<grid, kScenePointThreads, 0, (cudaStream_t)stream>>>(p);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
