// rt_closest.cu — closest point on the mesh for a batch of query points (rt_closest_point), the counterpart of
// trimesh.proximity.closest_point on the BVH8 blob the ray queries use.
//
// One thread per point: stack-based traversal of the BVH8 (point_step, rt_point.cuh), children nearest first by
// their lower bound, subtrees dropped when their bound exceeds the best squared distance found so far.  The answer is
// the minimum of the key (d2, prim) (DESIGN.md §4.6), so it depends neither on the traversal order nor on the launch
// geometry: the host simulator under tests/pointquery/ and a brute-force loop give the same bits.
#include <type_traits>
#include "rt_api.h"
#include "rt_point.cuh"

namespace rt {

constexpr int kPointThreads = 128;

struct PointParams {
    const uint8_t* blob;
    const float* origins;
    int64_t shape[4], stride[4];
    int packed;                  // row-major contiguous [.., 3]: offset 3 * r
    int64_t first, n;            // window [first, first + n) of the batch; outputs indexed by (r - first)
    float max_distance;
    float* closest;
    float* distance;
    int32_t* tri;
    float* uv;
    unsigned long long* counters;
};

struct PointStack {
    PointStackEntry e[kMaxDepth];
    __device__ __forceinline__ void push(int sp, const PointStackEntry& v) { e[sp] = v; }
    __device__ __forceinline__ void pop(int sp, PointStackEntry& v) { v = e[sp]; }
};

__device__ __forceinline__ int64_t point_offset(const PointParams& p, int64_t r) {
    if (p.packed) return 3 * r;
    const int64_t i2 = r % p.shape[2];
    const int64_t q = r / p.shape[2];
    const int64_t i1 = q % p.shape[1];
    const int64_t i0 = q / p.shape[1];
    return i0 * p.stride[0] + i1 * p.stride[1] + i2 * p.stride[2];
}

template <bool STATS>
__global__ void __launch_bounds__(kPointThreads) k_closest_point(const __grid_constant__ PointParams p) {
    using S = typename std::conditional<STATS, Stats, NoStats>::type;
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(p.blob);
    const uint8_t* tris = p.blob + hdr->tris_offset;
    const uint8_t* nodes = p.blob + hdr->nodes_offset;
    const int64_t i = (int64_t)blockIdx.x * kPointThreads + threadIdx.x;
    S st;
    bool found = false;
    if (i < p.n) {
        const int64_t o = point_offset(p, p.first + i);
        const int64_t os = p.stride[3];
        PointTrav t;
        point_init(t, p.origins[o], p.origins[o + os], p.origins[o + 2 * os], fmul(p.max_distance, p.max_distance));
        PointStack stack;
        while (!point_step(nodes, tris, t, st, stack)) {}
        found = t.prim != kNoPrim;
        if (found) {
            const uint8_t* tp = tris + (size_t)t.slot * 48u;
            const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
            const PointHit h = point_tri(t.x, t.y, t.z, as_float(a.x), as_float(a.y), as_float(a.z), as_float(b.x),
                                         as_float(b.y), as_float(b.z), as_float(c.x), as_float(c.y), as_float(c.z));
            p.closest[3 * i] = h.cx; p.closest[3 * i + 1] = h.cy; p.closest[3 * i + 2] = h.cz;
            p.distance[i] = fsqrt(t.best);
            p.tri[i] = t.prim;
            p.uv[2 * i] = h.w0; p.uv[2 * i + 1] = h.w1;
        } else {
            p.closest[3 * i] = 0.0f; p.closest[3 * i + 1] = 0.0f; p.closest[3 * i + 2] = 0.0f;
            p.distance[i] = as_float(0x7f800000u);
            p.tri[i] = -1;
            p.uv[2 * i] = 0.0f; p.uv[2 * i + 1] = 0.0f;
        }
    }
    if (STATS) {
        unsigned long long c0 = st.n_nodes(), c1 = st.n_tris(), c2 = i < p.n ? 1ull : 0ull, c3 = found ? 1ull : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c0 += __shfl_xor_sync(0xffffffffu, c0, o);
            c1 += __shfl_xor_sync(0xffffffffu, c1, o);
            c2 += __shfl_xor_sync(0xffffffffu, c2, o);
            c3 += __shfl_xor_sync(0xffffffffu, c3, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&p.counters[0], c0); atomicAdd(&p.counters[1], c1);
            atomicAdd(&p.counters[2], c2); atomicAdd(&p.counters[3], c3);
        }
    }
}

static bool points_packed(const int64_t shape[4], const int64_t stride[4]) {
    // row-major contiguous [s0, s1, s2, 3]; dimensions of extent 1 may carry any stride
    if (stride[3] != 1) return false;
    int64_t expect = 3;
    for (int i = 2; i >= 0; --i) {
        if (shape[i] != 1 && stride[i] != expect) return false;
        expect *= shape[i];
    }
    return true;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_closest_point(const void* blob, const rt_ray_desc* points, const rt_trace_opts* opts, float max_distance,
                                float* closest, float* distance, int32_t* tri_idx, float* uv, uint64_t* counters_dev,
                                void* scratch, void* stream) {
    (void)scratch;   // one thread per point: no work counter, the scratch is left as it was
    const char* fn = "rt_closest_point";
    RT_REQUIRE(blob != nullptr && ((uintptr_t)blob & 15) == 0, RT_ERR_INVALID, "%s: blob null or not 16-byte aligned", fn);
    RT_REQUIRE(points != nullptr, RT_ERR_INVALID, "%s: null point descriptor", fn);
    RT_REQUIRE(!(max_distance != max_distance) && max_distance >= 0.0f, RT_ERR_INVALID,
               "%s: max_distance must be >= 0 or +inf (got %g)", fn, (double)max_distance);
    RT_REQUIRE(points->nray >= 0 && points->shape[3] == 3, RT_ERR_INVALID, "%s: point batch must be [*b, 3]", fn);
    RT_REQUIRE(points->shape[0] >= 0 && points->shape[1] >= 0 && points->shape[2] >= 0 &&
                   points->shape[0] * points->shape[1] * points->shape[2] == points->nray,
               RT_ERR_INVALID, "%s: nray %lld does not match shape", fn, (long long)points->nray);
    static const rt_trace_opts kDefaults = {};
    const rt_trace_opts& o = opts ? *opts : kDefaults;
    RT_REQUIRE(o.ray_first >= 0 && o.ray_first <= points->nray, RT_ERR_INVALID, "%s: ray_first %lld outside [0, %lld]", fn,
               (long long)o.ray_first, (long long)points->nray);
    const int64_t count = o.ray_count <= 0 ? points->nray - o.ray_first : o.ray_count;
    RT_REQUIRE(count <= points->nray - o.ray_first, RT_ERR_INVALID, "%s: window [%lld, +%lld) exceeds the batch of %lld", fn,
               (long long)o.ray_first, (long long)count, (long long)points->nray);
    if (counters_dev) RT_CUDA_TRY(cudaMemsetAsync(counters_dev, 0, 4 * sizeof(uint64_t), (cudaStream_t)stream));
    if (count == 0) return RT_OK;
    RT_REQUIRE(points->origins != nullptr, RT_ERR_INVALID, "%s: null points", fn);
    RT_REQUIRE(closest && distance && tri_idx && uv, RT_ERR_INVALID, "%s: null output", fn);
    PointParams p = {};
    p.blob = reinterpret_cast<const uint8_t*>(blob);
    p.origins = points->origins;
    for (int a = 0; a < 4; ++a) { p.shape[a] = points->shape[a]; p.stride[a] = points->o_stride[a]; }
    p.packed = points_packed(points->shape, points->o_stride) ? 1 : 0;
    p.first = o.ray_first;
    p.n = count;
    p.max_distance = max_distance;
    p.closest = closest; p.distance = distance; p.tri = tri_idx; p.uv = uv;
    p.counters = reinterpret_cast<unsigned long long*>(counters_dev);
    const int64_t grid = (count + kPointThreads - 1) / kPointThreads;
    RT_REQUIRE(grid < ((int64_t)1 << 31), RT_ERR_INVALID, "%s: batch of %lld points too large for one launch", fn,
               (long long)count);
    if (counters_dev)
        k_closest_point<true><<<(unsigned)grid, kPointThreads, 0, (cudaStream_t)stream>>>(p);
    else
        k_closest_point<false><<<(unsigned)grid, kPointThreads, 0, (cudaStream_t)stream>>>(p);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
