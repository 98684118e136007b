// rt_scene.cu — instanced multi-mesh scenes: closest, any and count ray queries against many instances of BVH8
// blobs, each with its own affine transform (DESIGN.md §4.11).
//
// rt_scene_prepare: one thread per instance (k_scene_prepare) reads its mesh's header box from the device blob,
// computes the binary64 inverse transform and the padded world box, and writes the instance record and the instance's
// top-level "triangle" (lo, hi, lo).  The caller builds the top-level BVH from those with rt_bvh_build.
// rt_scene_trace: one thread per ray (k_scene_trace) walks the top-level tree (scene_step), and every instance whose
// box it crosses with its own tree under the object-space ray (traverse with the single-mesh visitors).  The answers
// are minima of total orders or sums, so the host simulator under tests/scene/ and a brute-force instance loop give
// the same bits.
#include "rt_api.h"
#include "rt_scene.cuh"

namespace rt {

constexpr int kSceneThreads = 128;

__global__ void __launch_bounds__(128) k_scene_prepare(uint8_t* table, uint32_t n_inst, float* tlas_v, int32_t* tlas_f) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inst) return;
    const SceneHeader* h = reinterpret_cast<const SceneHeader*>(table);
    SceneInst* inst = reinterpret_cast<SceneInst*>(table + h->inst_offset);
    const uint64_t* blobs = reinterpret_cast<const uint64_t*>(table + h->blobs_offset);
    SceneInst s = inst[i];
    prepare_instance(reinterpret_cast<const uint8_t*>(blobs[s.mesh]), s, i, tlas_v + 6 * (size_t)i, tlas_f + 3 * (size_t)i);
    inst[i] = s;
}

struct SceneParams {
    const uint8_t* table;
    const uint8_t* tlas;
    rt_ray_desc rays;
    int64_t first, n;            // window [first, first + n) of the batch; outputs indexed by (r - first)
    float tmax;
    uint8_t* hit;
    uint8_t* front;
    int32_t* inst;
    int32_t* tri;
    float* loc;
    float* uv;
    int32_t* count;
};

struct SceneStack {
    uint2 e[kMaxDepth];
    __device__ __forceinline__ void push(int sp, uint32_t x, uint32_t y) { e[sp] = make_uint2(x, y); }
    __device__ __forceinline__ void pop(int sp, uint32_t& x, uint32_t& y) { const uint2 v = e[sp]; x = v.x; y = v.y; }
};

template <int MODE>   // 0 closest, 1 any, 2 count
__global__ void __launch_bounds__(kSceneThreads) k_scene_trace(const __grid_constant__ SceneParams p) {
    const int64_t i = (int64_t)blockIdx.x * kSceneThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t r = p.first + i;
    const int64_t oo = scene_offset(p.rays.shape, p.rays.o_stride, r), dd = scene_offset(p.rays.shape, p.rays.d_stride, r);
    const int64_t os = p.rays.o_stride[3], ds = p.rays.d_stride[3];
    const float w[6] = {p.rays.origins[oo], p.rays.origins[oo + os], p.rays.origins[oo + 2 * os],
                        p.rays.directions[dd], p.rays.directions[dd + ds], p.rays.directions[dd + 2 * ds]};
    const rt_blob_header* th = reinterpret_cast<const rt_blob_header*>(p.tlas);
    const uint8_t* nodes = p.tlas + th->nodes_offset;
    const uint8_t* recs = p.tlas + th->tris_offset;
    const SceneView sv = scene_view(p.table);
    Ray wr;
    ray_setup(wr, w[0], w[1], w[2], w[3], w[4], w[5]);
    SceneStack top, below;
    Trav t;
    trav_init(t);
    if (MODE == 0) {
        SceneClosest<SceneStack> vis{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, p.tmax};
        vis.stack = &below;
        while (!scene_step(nodes, recs, wr, vis, top, t)) {}
        if (vis.inst >= 0) {
            const SceneHitOut a = scene_hit_attr(sv, vis.inst, vis.slot, w);
            p.hit[i] = 1; p.front[i] = a.front ? 1 : 0; p.inst[i] = vis.inst; p.tri[i] = vis.prim;
            p.loc[3 * i] = a.loc[0]; p.loc[3 * i + 1] = a.loc[1]; p.loc[3 * i + 2] = a.loc[2];
            p.uv[2 * i] = a.uv[0]; p.uv[2 * i + 1] = a.uv[1];
        } else {
            p.hit[i] = 0; p.front[i] = 0; p.inst[i] = -1; p.tri[i] = -1;
            p.loc[3 * i] = 0.0f; p.loc[3 * i + 1] = 0.0f; p.loc[3 * i + 2] = 0.0f;
            p.uv[2 * i] = 0.0f; p.uv[2 * i + 1] = 0.0f;
        }
    } else if (MODE == 1) {
        SceneAny<SceneStack> vis{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, p.tmax};
        vis.stack = &below;
        while (!scene_step(nodes, recs, wr, vis, top, t)) {}
        p.hit[i] = vis.found ? 1 : 0;
    } else {
        SceneCount<SceneStack> vis{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, p.tmax};
        vis.stack = &below;
        while (!scene_step(nodes, recs, wr, vis, top, t)) {}
        p.count[i] = vis.count;
    }
}

struct SceneLayout { size_t inst_offset, blobs_offset, total; };
static SceneLayout scene_layout(int64_t n_meshes, int64_t n_inst) {
    SceneLayout l;
    l.inst_offset = 256;
    l.blobs_offset = align_up_sz(l.inst_offset + (size_t)n_inst * sizeof(SceneInst), 256);
    l.total = align_up_sz(l.blobs_offset + (size_t)n_meshes * 8u, 256);
    return l;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_scene_prepare_sizes(int64_t n_meshes, int64_t n_inst, size_t* table_bytes) {
    RT_REQUIRE(n_meshes >= 0 && n_inst >= 0 && n_inst <= ((int64_t)1 << 30) && n_meshes <= ((int64_t)1 << 30) && table_bytes,
               RT_ERR_INVALID, "rt_scene_prepare_sizes: bad arguments");
    *table_bytes = scene_layout(n_meshes, n_inst).total;
    return RT_OK;
}

extern "C" int rt_scene_prepare(int64_t n_meshes, const void* const* blobs, int64_t n_inst, const int32_t* inst_mesh,
                                const float* transforms, void* table, size_t table_bytes, float* tlas_vertices,
                                int32_t* tlas_faces, void* stream_) {
    const char* fn = "rt_scene_prepare";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    size_t need = 0;
    RT_REQUIRE(rt_scene_prepare_sizes(n_meshes, n_inst, &need) == RT_OK, RT_ERR_INVALID, "%s: bad sizes", fn);
    RT_REQUIRE(table != nullptr && ((uintptr_t)table & 255) == 0, RT_ERR_INVALID, "%s: table null or not 256-byte aligned", fn);
    RT_REQUIRE(table_bytes >= need, RT_ERR_SIZE, "%s: table %zu < %zu bytes", fn, table_bytes, need);
    RT_REQUIRE(n_meshes == 0 || blobs != nullptr, RT_ERR_INVALID, "%s: null blob list", fn);
    RT_REQUIRE(n_inst == 0 || (inst_mesh && transforms && tlas_vertices && tlas_faces), RT_ERR_INVALID, "%s: null argument", fn);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    for (int64_t m = 0; m < n_meshes; ++m) {
        RT_REQUIRE(blobs[m] != nullptr && ((uintptr_t)blobs[m] & 15) == 0, RT_ERR_INVALID,
                   "%s: blob of mesh %lld null or not 16-byte aligned", fn, (long long)m);
        cudaPointerAttributes at;
        const cudaError_t e = cudaPointerGetAttributes(&at, blobs[m]);
        RT_REQUIRE(e == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == dev.device, RT_ERR_INVALID,
                   "%s: blob of mesh %lld is not memory of the current device %d", fn, (long long)m, dev.device);
    }
    SceneLayout l = scene_layout(n_meshes, n_inst);
    SceneHeader hdr = {};
    hdr.n_meshes = (uint64_t)n_meshes; hdr.n_inst = (uint64_t)n_inst;
    hdr.inst_offset = l.inst_offset; hdr.blobs_offset = l.blobs_offset;
    // The records start from the host: transform and mesh checked here (the kernel cannot report an error), the rest
    // is filled on the device from the blobs' headers.
    SceneInst* recs = n_inst > 0 ? (SceneInst*)calloc((size_t)n_inst, sizeof(SceneInst)) : nullptr;
    RT_REQUIRE(n_inst == 0 || recs != nullptr, RT_ERR_INVALID, "%s: out of host memory", fn);
    for (int64_t i = 0; i < n_inst; ++i) {
        SceneInst& s = recs[i];
        s.mesh = inst_mesh[i];
        for (int k = 0; k < 12; ++k) s.fwd[k] = transforms[12 * i + k];
        double det = 0.0, kappa = 0.0;
        const bool ok_mesh = s.mesh >= 0 && s.mesh < n_meshes;
        const bool ok_inv = invert_transform(s.fwd, s.inv, &det, &kappa);
        if (!ok_mesh || !ok_inv) {
            free(recs);
            if (!ok_mesh) return set_error(RT_ERR_INVALID, "%s: instance %lld: mesh index %d outside [0, %lld)", fn, (long long)i,
                                           (int)inst_mesh[i], (long long)n_meshes);
            return set_error(RT_ERR_INVALID, "%s: instance %lld: transform not finite, singular (det %g) or its inverse "
                             "overflows binary32", fn, (long long)i, det);
        }
    }
    cudaError_t e = cudaMemcpyAsync(table, &hdr, sizeof(hdr), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess && n_inst > 0)
        e = cudaMemcpyAsync((uint8_t*)table + l.inst_offset, recs, (size_t)n_inst * sizeof(SceneInst), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess && n_meshes > 0)
        e = cudaMemcpyAsync((uint8_t*)table + l.blobs_offset, blobs, (size_t)n_meshes * 8u, cudaMemcpyHostToDevice, stream);
    free(recs);   // pageable sources: cudaMemcpyAsync returns once it has staged them
    RT_CUDA_TRY(e);
    if (n_inst == 0) return RT_OK;
    k_scene_prepare<<<(unsigned)((n_inst + 127) / 128), 128, 0, stream>>>(reinterpret_cast<uint8_t*>(table), (uint32_t)n_inst,
                                                                          tlas_vertices, tlas_faces);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

extern "C" int rt_scene_trace(const void* table, const void* tlas_blob, const rt_ray_desc* rays, const rt_trace_opts* opts,
                              int mode, uint8_t* hit, uint8_t* front, int32_t* inst_idx, int32_t* tri_idx, float* loc,
                              float* uv, int32_t* count, void* stream) {
    const char* fn = "rt_scene_trace";
    RT_REQUIRE(table != nullptr && ((uintptr_t)table & 255) == 0, RT_ERR_INVALID, "%s: table null or not 256-byte aligned", fn);
    RT_REQUIRE(tlas_blob != nullptr && ((uintptr_t)tlas_blob & 15) == 0, RT_ERR_INVALID,
               "%s: top-level blob null or not 16-byte aligned", fn);
    RT_REQUIRE(mode >= RT_SCENE_CLOSEST && mode <= RT_SCENE_COUNT, RT_ERR_INVALID, "%s: unknown mode %d", fn, mode);
    RT_REQUIRE(rays != nullptr, RT_ERR_INVALID, "%s: null ray descriptor", fn);
    RT_REQUIRE(rays->nray >= 0 && rays->shape[3] == 3, RT_ERR_INVALID, "%s: ray batch must be [*b, 3]", fn);
    RT_REQUIRE(rays->shape[0] >= 0 && rays->shape[1] >= 0 && rays->shape[2] >= 0 &&
                   rays->shape[0] * rays->shape[1] * rays->shape[2] == rays->nray,
               RT_ERR_INVALID, "%s: nray %lld does not match shape", fn, (long long)rays->nray);
    static const rt_trace_opts kDefaults = {};
    const rt_trace_opts& o = opts ? *opts : kDefaults;
    RT_REQUIRE(o.ray_first >= 0 && o.ray_first <= rays->nray, RT_ERR_INVALID, "%s: ray_first %lld outside [0, %lld]", fn,
               (long long)o.ray_first, (long long)rays->nray);
    const int64_t n = o.ray_count <= 0 ? rays->nray - o.ray_first : o.ray_count;
    RT_REQUIRE(n <= rays->nray - o.ray_first, RT_ERR_INVALID, "%s: window [%lld, +%lld) exceeds the batch of %lld", fn,
               (long long)o.ray_first, (long long)n, (long long)rays->nray);
    if (n == 0) return RT_OK;
    RT_REQUIRE(rays->origins != nullptr && rays->directions != nullptr, RT_ERR_INVALID, "%s: null rays", fn);
    if (mode == RT_SCENE_CLOSEST)
        RT_REQUIRE(hit && front && inst_idx && tri_idx && loc && uv, RT_ERR_INVALID, "%s: null output", fn);
    else if (mode == RT_SCENE_ANY)
        RT_REQUIRE(hit != nullptr, RT_ERR_INVALID, "%s: null output", fn);
    else
        RT_REQUIRE(count != nullptr, RT_ERR_INVALID, "%s: null output", fn);
    const int64_t grid = (n + kSceneThreads - 1) / kSceneThreads;
    RT_REQUIRE(grid < ((int64_t)1 << 31), RT_ERR_INVALID, "%s: batch of %lld rays too large for one launch", fn, (long long)n);
    SceneParams p = {};
    p.table = reinterpret_cast<const uint8_t*>(table);
    p.tlas = reinterpret_cast<const uint8_t*>(tlas_blob);
    p.rays = *rays;
    p.first = o.ray_first;
    p.n = n;
    p.tmax = o.tmax > 0.0f ? o.tmax : RT_TMAX_DEFAULT;     // NaN and <= 0 select the default, as rt_trace_* do
    p.hit = hit; p.front = front; p.inst = inst_idx; p.tri = tri_idx; p.loc = loc; p.uv = uv; p.count = count;
    cudaStream_t st = (cudaStream_t)stream;
    if (mode == RT_SCENE_CLOSEST)
        k_scene_trace<0><<<(unsigned)grid, kSceneThreads, 0, st>>>(p);
    else if (mode == RT_SCENE_ANY)
        k_scene_trace<1><<<(unsigned)grid, kSceneThreads, 0, st>>>(p);
    else
        k_scene_trace<2><<<(unsigned)grid, kSceneThreads, 0, st>>>(p);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
