// rt_scene_grad.cu — gradients of the instanced-scene queries (DESIGN.md §4.13): the closest-hit loc and uv
// (rt_scene_ray_grad) and the point distance or signed distance (rt_scene_distance_grad), with respect to the rays or
// points, the instance transforms and the member vertices, from the forward's outputs alone.
//
// Per row window, with the arithmetic of rt_scenegrad.cuh:
//   1. one thread per row: the per-ray (head row of a ray) or per-point gradient and, when transform or vertex
//      gradients are wanted, the row's factors (q, q_obj, x, w: 44 B) and its pairs, three vertex keys and four
//      transform-column keys of the joint key space [member vertices | 4 I transform columns];
//   2. and 3. rt_distgrad.cu's sort and fixed tree (dg_reduce) with the scene's level-0 contribution, into one
//      accumulator of the key space;
// then one kernel copies the accumulator to grad_vertices and, transposed, to grad_transforms.  Nothing is atomic.
#include "rt_api.h"
#include "rt_scenegrad.cuh"

namespace rt {

struct SgPairsOut {
    float* rec;                  // [n, kSgRowFloats] or null (no transform or vertex gradient)
    uint64_t* keys;              // [n_slots n]
    uint32_t* vals;
    int slot0, n_slots;          // slots [slot0, slot0 + n_slots) of 0..6 are emitted
    uint64_t n_keys;
};

__device__ __forceinline__ void sg_emit(const SgPairsOut& o, int64_t i, bool live, const SgRow& r,
                                        const uint64_t vkey[3], int32_t inst, uint64_t n_verts) {
    sg_store(r, o.rec + (size_t)kSgRowFloats * i);
    for (int s = 0; s < o.n_slots; ++s) {
        o.keys[o.n_slots * i + s] = sg_key(live, vkey, inst, o.slot0 + s, n_verts, o.n_keys);
        o.vals[o.n_slots * i + s] = (uint32_t)(o.n_slots * i + s);
    }
}

struct SgSceneArgs {
    const uint8_t* table;
    int64_t n_inst, n_meshes, n_verts;
    const rt_scene_member* members;
};
__device__ __forceinline__ SgScene sg_scene_of(const SgSceneArgs& a) {
    return sg_scene(a.table, a.n_inst, a.members, a.n_meshes, a.n_verts);
}

struct SgHitParams {
    SgSceneArgs scene;
    const float* origins;
    const float* directions;
    int64_t shape[4], o_stride[4], d_stride[4];
    int o_packed, d_packed;
    int64_t first, window, n_rows;
    int64_t n, base;             // rows of this launch, [base, base + n)
    const int32_t* row_ray;      // [n_rows] or null (row j is ray j)
    const int32_t* inst;
    const int32_t* tri;
    const float* grad_loc;       // [n_rows, 3] or null
    const float* grad_uv;        // [n_rows, 2] or null
    float* grad_origins;         // [window, 3] or null
    float* grad_directions;
    SgPairsOut out;
};

__device__ __forceinline__ int64_t sg_ray_of(const SgHitParams& p, int64_t j) {
    const int64_t ray = p.row_ray ? (int64_t)p.row_ray[j] : j;
    return ray >= 0 && ray < p.window ? ray : -1;
}

__device__ __forceinline__ bool sg_hit_eval(const SgHitParams& p, const SgScene& sc, int64_t j, RgRow& rr, SgRow& r,
                                            uint64_t key[3]) {
    const int64_t ray = sg_ray_of(p, j);
    const float gz[3] = {0.0f, 0.0f, 0.0f};
    if (ray < 0) return sg_hit_row(sc, -1, -1, gz, gz, gz, 0.0f, 0.0f, rr, r, key);
    const int64_t b = p.first + ray;
    const int64_t oo = batch_offset(p.shape, p.o_stride, p.o_packed, b);
    const int64_t od = batch_offset(p.shape, p.d_stride, p.d_packed, b);
    const int64_t os = p.o_stride[3], ds = p.d_stride[3];
    const float o[3] = {p.origins[oo], p.origins[oo + os], p.origins[oo + 2 * os]};
    const float d[3] = {p.directions[od], p.directions[od + ds], p.directions[od + 2 * ds]};
    float gl[3] = {0.0f, 0.0f, 0.0f};
    float gu0 = 0.0f, gu1 = 0.0f;
    if (p.grad_loc) { gl[0] = p.grad_loc[3 * j]; gl[1] = p.grad_loc[3 * j + 1]; gl[2] = p.grad_loc[3 * j + 2]; }
    if (p.grad_uv) { gu0 = p.grad_uv[2 * j]; gu1 = p.grad_uv[2 * j + 1]; }
    return sg_hit_row(sc, p.inst[j], p.tri[j], o, d, gl, gu0, gu1, rr, r, key);
}

__global__ void __launch_bounds__(kDgThreads) k_sg_hit_rows(const __grid_constant__ SgHitParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t j = p.base + i;
    const SgScene sc = sg_scene_of(p.scene);
    if ((p.grad_origins || p.grad_directions) && rg_head(j, p.row_ray)) {
        const int64_t ray = sg_ray_of(p, j);
        if (ray >= 0) {
            float go[3], gd[3];
            rg_ray_sums(j, p.n_rows, p.row_ray, [&](int64_t k, RgRow& rr) {
                SgRow r;
                uint64_t key[3];
                sg_hit_eval(p, sc, k, rr, r, key);
            }, go, gd);
            if (p.grad_origins) {
                p.grad_origins[3 * ray] = go[0]; p.grad_origins[3 * ray + 1] = go[1]; p.grad_origins[3 * ray + 2] = go[2];
            }
            if (p.grad_directions) {
                p.grad_directions[3 * ray] = gd[0]; p.grad_directions[3 * ray + 1] = gd[1];
                p.grad_directions[3 * ray + 2] = gd[2];
            }
        }
    }
    if (p.out.rec) {
        RgRow rr;
        SgRow r;
        uint64_t key[3];
        const bool live = sg_hit_eval(p, sc, j, rr, r, key);
        sg_emit(p.out, i, live, r, key, live ? p.inst[j] : -1, (uint64_t)p.scene.n_verts);
    }
}

struct SgPointParams {
    SgSceneArgs scene;
    const float* points;
    int64_t shape[4], stride[4];
    int packed;
    int64_t first;               // batch index of window position 0
    int64_t n, base;             // points of this launch, window positions [base, base + n)
    const float* grad_out;
    const float* value;
    const float* closest;
    const int32_t* inst;
    const int32_t* tri;
    const float* uv;
    float* grad_points;          // [window, 3] or null
    SgPairsOut out;
};

__global__ void __launch_bounds__(kDgThreads) k_sg_point_rows(const __grid_constant__ SgPointParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t w = p.base + i;
    const int64_t o = batch_offset(p.shape, p.stride, p.packed, p.first + w);
    const int64_t os = p.stride[3];
    float q[3];
    SgRow r;
    uint64_t key[3];
    const int32_t inst = p.inst[w];
    const bool live = sg_point_row(sg_scene_of(p.scene), inst, p.tri[w], p.points[o], p.points[o + os], p.points[o + 2 * os],
                                   p.grad_out[w], p.value[w], p.closest[3 * w], p.closest[3 * w + 1],
                                   p.closest[3 * w + 2], p.uv[2 * w], p.uv[2 * w + 1], q, r, key);
    if (p.grad_points) {
        p.grad_points[3 * w] = q[0]; p.grad_points[3 * w + 1] = q[1]; p.grad_points[3 * w + 2] = q[2];
    }
    if (p.out.rec) sg_emit(p.out, i, live, r, key, inst, (uint64_t)p.scene.n_verts);
}

__global__ void __launch_bounds__(kDgThreads) k_sg_level0(const uint64_t* keys, const uint32_t* vals, int64_t m,
                                                          const uint32_t* start, uint64_t n_keys, const float* rec,
                                                          int slot0, int n_slots, float* acc, DgLevel next) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < m; j += stride)
        dg_level0_with((uint64_t)j, (uint64_t)m, keys, vals, start, n_keys,
                       [&](uint32_t e, float out[3]) { sg_contrib(rec, slot0, n_slots, e, out); }, acc, next);
}

__global__ void __launch_bounds__(kDgThreads) k_sg_outputs(const float* acc, int64_t n_verts, int64_t n_inst,
                                                           float* grad_vertices, float* grad_transforms) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    const int64_t nv = grad_vertices ? 3 * n_verts : 0, nt = grad_transforms ? 12 * n_inst : 0;
    for (int64_t e = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; e < nv + nt; e += stride) {
        if (e < nv) grad_vertices[e] = acc[e];
        else sg_transform_out(acc, (uint64_t)n_verts, (uint64_t)(e - nv), grad_transforms);
    }
}

// Workspace of a window of w rows with n_slots pairs each over n_keys keys: row factors, keys, values, sort
// workspace, run starts, two level buffers, the accumulator [n_keys, 3].
struct SgWorkspace {
    float* rec;
    DgPairs pairs;
    float* acc;
    size_t total;
};
static SgWorkspace carve_sg(void* base, int64_t w, int n_slots, int64_t n_keys) {
    const int64_t m = n_slots * w;
    const uint64_t slots = dg_next_size((uint64_t)m);
    size_t sb = 0;
    rt_sort_sizes(m, &sb);
    const size_t sizes[12] = {(size_t)w * 4u * kSgRowFloats, (size_t)m * 8u, (size_t)m * 4u, sb, (size_t)n_keys * 4u,
                              slots * 4u, slots * 4u, slots * 12u, slots * 4u, slots * 4u, slots * 12u,
                              (size_t)n_keys * 12u};
    size_t off[13];
    off[0] = 0;
    for (int i = 0; i < 12; ++i) off[i + 1] = off[i] + align_up_sz(sizes[i], 256);
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    auto at = [&](size_t o) { return p ? p + o : nullptr; };
    SgWorkspace ws;
    ws.rec = reinterpret_cast<float*>(at(off[0]));
    ws.pairs.keys = reinterpret_cast<uint64_t*>(at(off[1]));
    ws.pairs.vals = reinterpret_cast<uint32_t*>(at(off[2]));
    ws.pairs.sort_ws = at(off[3]);
    ws.pairs.start = reinterpret_cast<uint32_t*>(at(off[4]));
    ws.pairs.lv[0] = DgLevel{reinterpret_cast<uint32_t*>(at(off[5])), reinterpret_cast<uint32_t*>(at(off[6])),
                             reinterpret_cast<float*>(at(off[7]))};
    ws.pairs.lv[1] = DgLevel{reinterpret_cast<uint32_t*>(at(off[8])), reinterpret_cast<uint32_t*>(at(off[9])),
                             reinterpret_cast<float*>(at(off[10]))};
    ws.acc = reinterpret_cast<float*>(at(off[11]));
    ws.total = off[12];
    return ws;
}

// The slots a call emits: vertex slots 0..2 and / or transform slots 3..6
static void sg_slots(bool transforms, bool vertices, int* slot0, int* n_slots) {
    *slot0 = vertices ? 0 : 3;
    *n_slots = (vertices ? 3 : 0) + (transforms ? 4 : 0);
}

// The largest window of at most n (and kSgMaxRows) rows whose workspace fits workspace_bytes; 0 when not even one fits.
static int64_t sg_window(int64_t n, int n_slots, int64_t n_keys, size_t workspace_bytes) {
    int64_t win = n < kSgMaxRows ? n : kSgMaxRows;
    if (carve_sg(nullptr, win, n_slots, n_keys).total > workspace_bytes) {
        int64_t lo = 0, hi = win;                       // fits(lo), !fits(hi)
        while (hi - lo > 1) {
            const int64_t mid = lo + (hi - lo) / 2;
            (carve_sg(nullptr, mid, n_slots, n_keys).total <= workspace_bytes ? lo : hi) = mid;
        }
        win = lo;
    }
    return win;
}

struct SgLevel0Arg { const float* rec; int slot0, n_slots; };
static void sg_level0_launch(const void* arg, const uint64_t* keys, const uint32_t* vals, int64_t m,
                             const uint32_t* start, uint64_t n_keys, float* acc, DgLevel next, int grid,
                             cudaStream_t stream) {
    const SgLevel0Arg* a = static_cast<const SgLevel0Arg*>(arg);
    k_sg_level0<<<grid, kDgThreads, 0, stream>>>(keys, vals, m, start, n_keys, a->rec, a->slot0, a->n_slots, acc, next);
}

// Host checks shared by both entry points; *n_keys = n_verts + 4 n_inst.
static int sg_check_scene(const char* fn, const void* table, int64_t n_inst, const rt_scene_member* members,
                          int64_t n_meshes, int64_t n_verts, int64_t* n_keys) {
    RT_REQUIRE(n_inst >= 0 && n_meshes >= 0 && n_verts >= 0 && n_inst < kDgMaxVerts && n_verts < kDgMaxVerts &&
                   n_verts + 4 * n_inst < kDgMaxVerts,
               RT_ERR_INVALID, "%s: bad sizes (%lld instances, %lld meshes, %lld vertices)", fn, (long long)n_inst,
               (long long)n_meshes, (long long)n_verts);
    RT_REQUIRE(table != nullptr && (members != nullptr || n_meshes == 0), RT_ERR_INVALID, "%s: null table or members", fn);
    *n_keys = n_verts + 4 * n_inst;
    return RT_OK;
}

// Runs the row kernel `rows(n, base, out)` over windows and reduces the pairs into the outputs; without transform and
// vertex outputs one launch over every row.
template <class RowLaunch>
static int sg_run(const char* fn, int64_t n_rows, int64_t n_inst, int64_t n_verts, int64_t n_keys,
                  float* grad_transforms, float* grad_vertices, void* workspace, size_t workspace_bytes,
                  const RowLaunch& rows, cudaStream_t stream) {
    SgPairsOut out{};
    out.n_keys = (uint64_t)n_keys;
    if (!grad_transforms && !grad_vertices) {
        RT_REQUIRE((n_rows + kDgThreads - 1) / kDgThreads < ((int64_t)1 << 31), RT_ERR_INVALID,
                   "%s: %lld rows too many for one launch", fn, (long long)n_rows);
        rows(n_rows, 0, out);
        RT_CUDA_TRY(cudaGetLastError());
        return RT_OK;
    }
    int slot0 = 0, n_slots = 0;
    sg_slots(grad_transforms != nullptr, grad_vertices != nullptr, &slot0, &n_slots);
    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    const int64_t win = sg_window(n_rows, n_slots, n_keys, workspace_bytes);
    RT_REQUIRE(win > 0, RT_ERR_SIZE, "%s: workspace %zu < %zu (one row)", fn, workspace_bytes,
               carve_sg(nullptr, 1, n_slots, n_keys).total);
    const SgWorkspace w = carve_sg(workspace, win, n_slots, n_keys);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    RT_CUDA_TRY(cudaMemsetAsync(w.acc, 0, (size_t)n_keys * 12u, stream));
    const int passes = dg_sort_passes(n_keys);
    out.rec = w.rec; out.keys = w.pairs.keys; out.vals = w.pairs.vals; out.slot0 = slot0; out.n_slots = n_slots;
    const SgLevel0Arg arg{w.rec, slot0, n_slots};
    for (int64_t base = 0; base < n_rows; base += win) {
        const int64_t nw = n_rows - base < win ? n_rows - base : win;
        rows(nw, base, out);
        RT_CUDA_TRY(cudaGetLastError());
        const int rc = dg_reduce(w.pairs, n_slots * nw, n_keys, passes, dev.sm_count, sg_level0_launch, &arg, w.acc,
                                 stream);
        if (rc != RT_OK) return rc;
    }
    const int64_t total = (grad_vertices ? 3 * n_verts : 0) + (grad_transforms ? 12 * n_inst : 0);
    if (total > 0) {
        k_sg_outputs<<<grid_for(total, kDgThreads, dev.sm_count, 8), kDgThreads, 0, stream>>>(w.acc, n_verts, n_inst,
                                                                                             grad_vertices,
                                                                                             grad_transforms);
        RT_CUDA_TRY(cudaGetLastError());
    }
    return RT_OK;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_scene_grad_sizes(int64_t n_rows, int64_t n_inst, int64_t n_verts_total, int outputs,
                                   size_t* workspace_bytes) {
    RT_REQUIRE(n_rows >= 0 && n_inst >= 0 && n_verts_total >= 0 && n_inst < kDgMaxVerts && n_verts_total < kDgMaxVerts &&
                   n_verts_total + 4 * n_inst < kDgMaxVerts && (outputs & ~3) == 0 && workspace_bytes,
               RT_ERR_INVALID, "rt_scene_grad_sizes: bad arguments (n_verts_total + 4 n_inst below %lld)",
               (long long)kDgMaxVerts);
    if (outputs == 0) { *workspace_bytes = 0; return RT_OK; }
    int slot0 = 0, n_slots = 0;
    sg_slots((outputs & RT_SCENE_GRAD_TRANSFORMS) != 0, (outputs & RT_SCENE_GRAD_VERTICES) != 0, &slot0, &n_slots);
    const int64_t w = n_rows < kSgMaxRows ? n_rows : kSgMaxRows;
    *workspace_bytes = carve_sg(nullptr, w > 0 ? w : 1, n_slots, n_verts_total + 4 * n_inst).total;
    return RT_OK;
}

extern "C" int rt_scene_ray_grad(const void* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                                 int64_t n_verts_total, const rt_ray_desc* rays, const rt_trace_opts* opts,
                                 int64_t n_rows, const int32_t* row_ray, const int32_t* inst_idx,
                                 const int32_t* tri_idx, const float* grad_loc, const float* grad_uv,
                                 float* grad_origins, float* grad_directions, float* grad_transforms,
                                 float* grad_vertices, void* workspace, size_t workspace_bytes, void* stream_) {
    const char* fn = "rt_scene_ray_grad";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    int64_t first = 0, window = 0, n_keys = 0;
    int rc = batch_window(fn, rays, opts, &first, &window);
    if (rc != RT_OK) return rc;
    rc = sg_check_scene(fn, table, n_inst, members, n_meshes, n_verts_total, &n_keys);
    if (rc != RT_OK) return rc;
    RT_REQUIRE(n_rows >= 0, RT_ERR_INVALID, "%s: %lld rows", fn, (long long)n_rows);
    RT_REQUIRE(row_ray != nullptr || n_rows == window || n_rows == 0, RT_ERR_INVALID,
               "%s: without row_ray there must be one row per ray of the window (%lld rows, %lld rays)", fn,
               (long long)n_rows, (long long)window);
    RT_REQUIRE(n_rows == 0 || (rays->origins && rays->directions && inst_idx && tri_idx), RT_ERR_INVALID,
               "%s: null input", fn);
    if (grad_vertices) RT_CUDA_TRY(cudaMemsetAsync(grad_vertices, 0, (size_t)n_verts_total * 12u, stream));
    if (grad_transforms) RT_CUDA_TRY(cudaMemsetAsync(grad_transforms, 0, (size_t)n_inst * 48u, stream));
    if (row_ray || n_rows == 0) {       // rays without rows get +0
        if (grad_origins) RT_CUDA_TRY(cudaMemsetAsync(grad_origins, 0, (size_t)window * 12u, stream));
        if (grad_directions) RT_CUDA_TRY(cudaMemsetAsync(grad_directions, 0, (size_t)window * 12u, stream));
    }
    if (n_rows == 0 || (!grad_origins && !grad_directions && !grad_transforms && !grad_vertices)) return RT_OK;

    SgHitParams p{};
    p.scene = SgSceneArgs{reinterpret_cast<const uint8_t*>(table), n_inst, n_meshes, n_verts_total, members};
    p.origins = rays->origins; p.directions = rays->directions;
    for (int a = 0; a < 4; ++a) {
        p.shape[a] = rays->shape[a]; p.o_stride[a] = rays->o_stride[a]; p.d_stride[a] = rays->d_stride[a];
    }
    p.o_packed = batch_packed(rays->shape, rays->o_stride) ? 1 : 0;
    p.d_packed = batch_packed(rays->shape, rays->d_stride) ? 1 : 0;
    p.first = first; p.window = window; p.n_rows = n_rows;
    p.row_ray = row_ray; p.inst = inst_idx; p.tri = tri_idx; p.grad_loc = grad_loc; p.grad_uv = grad_uv;
    p.grad_origins = grad_origins; p.grad_directions = grad_directions;
    return sg_run(fn, n_rows, n_inst, n_verts_total, n_keys, grad_transforms, grad_vertices, workspace, workspace_bytes,
                  [&](int64_t n, int64_t base, const SgPairsOut& out) {
                      p.n = n; p.base = base; p.out = out;
                      k_sg_hit_rows<<<(unsigned)((n + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
                  }, stream);
}

extern "C" int rt_scene_distance_grad(const void* table, int64_t n_inst, const rt_scene_member* members,
                                      int64_t n_meshes, int64_t n_verts_total, const rt_ray_desc* points,
                                      const rt_trace_opts* opts, const float* grad_out, const float* value,
                                      const float* closest, const int32_t* inst_idx, const int32_t* tri_idx,
                                      const float* uv, float* grad_points, float* grad_transforms, float* grad_vertices,
                                      void* workspace, size_t workspace_bytes, void* stream_) {
    const char* fn = "rt_scene_distance_grad";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    int64_t first = 0, n = 0, n_keys = 0;
    int rc = batch_window(fn, points, opts, &first, &n);
    if (rc != RT_OK) return rc;
    rc = sg_check_scene(fn, table, n_inst, members, n_meshes, n_verts_total, &n_keys);
    if (rc != RT_OK) return rc;
    RT_REQUIRE(n == 0 || (points->origins && grad_out && value && closest && inst_idx && tri_idx && uv), RT_ERR_INVALID,
               "%s: null input", fn);
    if (grad_vertices) RT_CUDA_TRY(cudaMemsetAsync(grad_vertices, 0, (size_t)n_verts_total * 12u, stream));
    if (grad_transforms) RT_CUDA_TRY(cudaMemsetAsync(grad_transforms, 0, (size_t)n_inst * 48u, stream));
    if (n == 0 || (!grad_points && !grad_transforms && !grad_vertices)) return RT_OK;

    SgPointParams p{};
    p.scene = SgSceneArgs{reinterpret_cast<const uint8_t*>(table), n_inst, n_meshes, n_verts_total, members};
    p.points = points->origins;
    for (int a = 0; a < 4; ++a) { p.shape[a] = points->shape[a]; p.stride[a] = points->o_stride[a]; }
    p.packed = batch_packed(points->shape, points->o_stride) ? 1 : 0;
    p.first = first;
    p.grad_out = grad_out; p.value = value; p.closest = closest; p.inst = inst_idx; p.tri = tri_idx; p.uv = uv;
    p.grad_points = grad_points;
    return sg_run(fn, n, n_inst, n_verts_total, n_keys, grad_transforms, grad_vertices, workspace, workspace_bytes,
                  [&](int64_t nw, int64_t base, const SgPairsOut& out) {
                      p.n = nw; p.base = base; p.out = out;
                      k_sg_point_rows<<<(unsigned)((nw + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
                  }, stream);
}
