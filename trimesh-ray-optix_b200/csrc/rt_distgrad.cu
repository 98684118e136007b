// rt_distgrad.cu — the gradient of the point-to-mesh distance with respect to the query points and the mesh vertices
// (rt_distance_grad, DESIGN.md §4.9), from the outputs of rt_closest_point or rt_signed_distance_closest alone, and the
// gradient of hit locations and barycentrics with respect to the rays and the mesh vertices (rt_ray_grad, §4.10).
//
// Per point (or hit row) window, with the arithmetic of rt_distgrad.cuh (rt_raygrad.cuh):
//   1. one thread per point: grad_points and, when the vertex gradient is wanted, q (12 B) and three
//      (key = vertex, value = pair index 3 i + k) pairs; one thread per hit row: grad_origins and grad_directions of
//      the ray whose rows it heads, q, w (8 B) and three pairs;
//   2. the builder's stable onesweep sort of the pairs on the low bits of the key (ceil(log2(n_verts + 1)) bits,
//      at most 4 passes): each vertex's pairs become one run, in ascending pair order;
//   3. the run starts, then the tree reduction: level 0 sums groups of kDgGroup pairs of a run, every further level
//      groups of kDgGroup sums of the level below; a run that fits one group is added to grad_vertices.
// Nothing is atomic and every sum has one fixed order, so the result does not depend on the launch.
#include "rt_api.h"
#include "rt_distgrad.cuh"
#include "rt_raygrad.cuh"

namespace rt {

constexpr int kDgThreads = 256;

struct DgPointParams {
    const float* points;
    int64_t shape[4], stride[4];
    int packed;
    int64_t first;               // batch index of window position 0
    int64_t n;                   // points in this launch, window positions [base, base + n)
    int64_t base;
    const float* grad_out;
    const float* value;
    const float* closest;
    const int32_t* tri;
    const int32_t* faces;
    int64_t n_faces, n_verts;
    float* grad_points;          // [window, 3] or null
    float* q;                    // [n, 3] or null (no vertex gradient)
    uint64_t* keys;              // [3 n]
    uint32_t* vals;              // [3 n]
};

__global__ void __launch_bounds__(kDgThreads) k_dg_points(const __grid_constant__ DgPointParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t w = p.base + i;              // position in the caller's window
    const int64_t r = p.first + w;             // index in the batch
    const int64_t o = batch_offset(p.shape, p.stride, p.packed, r);
    const int64_t os = p.stride[3];
    const int32_t t = p.tri[w];
    float q[3];
    const bool live = dg_point_q(p.points[o], p.points[o + os], p.points[o + 2 * os], p.grad_out[w], p.value[w],
                                 p.closest[3 * w], p.closest[3 * w + 1], p.closest[3 * w + 2], t, p.n_faces, q);
    if (p.grad_points) {
        p.grad_points[3 * w] = q[0]; p.grad_points[3 * w + 1] = q[1]; p.grad_points[3 * w + 2] = q[2];
    }
    if (p.q) {
        p.q[3 * i] = q[0]; p.q[3 * i + 1] = q[1]; p.q[3 * i + 2] = q[2];
#pragma unroll
        for (uint32_t k = 0; k < 3; ++k) {
            p.keys[3 * i + k] = dg_key(live, p.faces, t, k, p.n_verts);
            p.vals[3 * i + k] = (uint32_t)(3 * i + k);
        }
    }
}

__global__ void __launch_bounds__(kDgThreads) k_dg_run_start(const uint64_t* keys, int64_t m, uint64_t n_verts,
                                                             uint32_t* start) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < m; j += stride)
        dg_run_start((uint64_t)j, keys, n_verts, start);
}

__global__ void __launch_bounds__(kDgThreads) k_dg_level0(const uint64_t* keys, const uint32_t* vals, int64_t m,
                                                          const uint32_t* start, uint64_t n_verts, const float* q,
                                                          const float* uv, float* grad_vertices, DgLevel next) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < m; j += stride)
        dg_level0_at((uint64_t)j, (uint64_t)m, keys, vals, start, n_verts, q, uv, grad_vertices, next);
}

__global__ void __launch_bounds__(kDgThreads) k_dg_level(DgLevel cur, int64_t size, float* grad_vertices, DgLevel next) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < size; j += stride)
        dg_level_at((uint64_t)j, (uint64_t)size, cur, grad_vertices, next);
}

struct RgRowParams {
    const float* origins;
    const float* directions;
    int64_t shape[4], o_stride[4], d_stride[4];
    int o_packed, d_packed;
    int64_t first;               // batch index of window ray 0
    int64_t window;              // rays in the window
    int64_t n_rows;
    int64_t n;                   // rows in this launch, [base, base + n)
    int64_t base;
    const int32_t* row_ray;      // [n_rows] or null (row i is ray i)
    const int32_t* tri;
    const float* grad_loc;       // [n_rows, 3] or null
    const float* grad_uv;        // [n_rows, 2] or null
    RgMesh mesh;
    float* grad_origins;         // [window, 3] or null
    float* grad_directions;      // [window, 3] or null
    float* q;                    // [n, 3] or null (no vertex gradient)
    float* w;                    // [n, 2]
    uint64_t* keys;              // [3 n]
    uint32_t* vals;              // [3 n]
};

// ray of row j in the window, or -1 for a row_ray outside [0, window)
__device__ __forceinline__ int64_t rg_ray_of(const RgRowParams& p, int64_t j) {
    const int64_t ray = p.row_ray ? (int64_t)p.row_ray[j] : j;
    return ray >= 0 && ray < p.window ? ray : -1;
}

__device__ __forceinline__ bool rg_eval(const RgRowParams& p, int64_t j, RgRow& r) {
    const int64_t ray = rg_ray_of(p, j);
    if (ray < 0) {
        const float gz[3] = {0.0f, 0.0f, 0.0f};
        return rg_row(gz, gz, gz, 0.0f, 0.0f, -1, p.mesh, r);
    }
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
    return rg_row(o, d, gl, gu0, gu1, p.tri[j], p.mesh, r);
}

__global__ void __launch_bounds__(kDgThreads) k_rg_rows(const __grid_constant__ RgRowParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t j = p.base + i;
    if ((p.grad_origins || p.grad_directions) && rg_head(j, p.row_ray)) {
        const int64_t ray = rg_ray_of(p, j);
        if (ray >= 0) {
            float go[3], gd[3];
            rg_ray_sums(j, p.n_rows, p.row_ray, [&](int64_t k, RgRow& r) { rg_eval(p, k, r); }, go, gd);
            if (p.grad_origins) {
                p.grad_origins[3 * ray] = go[0]; p.grad_origins[3 * ray + 1] = go[1]; p.grad_origins[3 * ray + 2] = go[2];
            }
            if (p.grad_directions) {
                p.grad_directions[3 * ray] = gd[0]; p.grad_directions[3 * ray + 1] = gd[1];
                p.grad_directions[3 * ray + 2] = gd[2];
            }
        }
    }
    if (p.q) {
        RgRow r;
        const bool live = rg_eval(p, j, r);
        p.q[3 * i] = r.q[0]; p.q[3 * i + 1] = r.q[1]; p.q[3 * i + 2] = r.q[2];
        p.w[2 * i] = r.w[0]; p.w[2 * i + 1] = r.w[1];
#pragma unroll
        for (uint32_t k = 0; k < 3; ++k) {
            p.keys[3 * i + k] = dg_key(live, p.mesh.faces, p.tri[j], k, p.mesh.n_verts);
            p.vals[3 * i + k] = (uint32_t)(3 * i + k);
        }
    }
}

// Workspace of a window of w points (hit rows): q, w (hit rows only), keys, values, sort workspace, run starts, two
// level buffers.
struct DgWorkspace {
    float* q;
    float* w;
    uint64_t* keys;
    uint32_t* vals;
    void* sort_ws;
    uint32_t* start;
    DgLevel lv[2];
    size_t total;
};
static DgWorkspace carve_dg(void* base, int64_t w, int64_t n_verts, bool with_w) {
    const int64_t m = 3 * w;
    const uint64_t slots = dg_next_size((uint64_t)m);
    size_t sb = 0;
    rt_sort_sizes(m, &sb);
    const size_t sizes[11] = {(size_t)w * 12u, with_w ? (size_t)w * 8u : 0u, (size_t)m * 8u, (size_t)m * 4u, sb,
                              (size_t)n_verts * 4u, slots * 4u, slots * 4u, slots * 12u, slots * 4u, slots * 4u};
    size_t off[12];
    off[0] = 0;
    for (int i = 0; i < 11; ++i) off[i + 1] = off[i] + align_up_sz(sizes[i], 256);
    // the last level buffer's values follow its idx array
    const size_t total = off[11] + align_up_sz(slots * 12u, 256);
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    auto at = [&](size_t o) { return p ? p + o : nullptr; };
    DgWorkspace ws;
    ws.q = reinterpret_cast<float*>(at(off[0]));
    ws.w = with_w ? reinterpret_cast<float*>(at(off[1])) : nullptr;
    ws.keys = reinterpret_cast<uint64_t*>(at(off[2]));
    ws.vals = reinterpret_cast<uint32_t*>(at(off[3]));
    ws.sort_ws = at(off[4]);
    ws.start = reinterpret_cast<uint32_t*>(at(off[5]));
    ws.lv[0] = DgLevel{reinterpret_cast<uint32_t*>(at(off[6])), reinterpret_cast<uint32_t*>(at(off[7])),
                       reinterpret_cast<float*>(at(off[8]))};
    ws.lv[1] = DgLevel{reinterpret_cast<uint32_t*>(at(off[9])), reinterpret_cast<uint32_t*>(at(off[10])),
                       reinterpret_cast<float*>(at(off[11]))};
    ws.total = total;
    return ws;
}

constexpr int64_t kDgMaxVerts = 0xffffffffll;     // vertex ids and the sentinel n_verts fit 32 bits

// The largest window of at most n (and kDgMaxPoints) points whose workspace fits workspace_bytes; 0 when not even
// one point fits.
static int64_t dg_window(int64_t n, int64_t n_verts, bool with_w, size_t workspace_bytes) {
    int64_t win = n < kDgMaxPoints ? n : kDgMaxPoints;
    if (carve_dg(nullptr, win, n_verts, with_w).total > workspace_bytes) {
        int64_t lo = 0, hi = win;                       // fits(lo), !fits(hi)
        while (hi - lo > 1) {
            const int64_t mid = lo + (hi - lo) / 2;
            (carve_dg(nullptr, mid, n_verts, with_w).total <= workspace_bytes ? lo : hi) = mid;
        }
        win = lo;
    }
    return win;
}

// Steps 2 and 3 for one window of nw points whose pairs are in w.keys / w.vals and whose q and uv (w for hit rows)
// are at w.q and uv: adds every vertex's sum of the window to grad_vertices.
static int dg_reduce_window(const DgWorkspace& w, int64_t nw, int64_t n_verts, const float* uv, int passes,
                            int sm_count, float* grad_vertices, cudaStream_t stream) {
    const int64_t m = 3 * nw;
    uint64_t* keys = nullptr;
    uint32_t* vals = nullptr;
    const int rc = sort_pairs_low(w.keys, w.vals, m, w.sort_ws, passes, &keys, &vals, stream);
    if (rc != RT_OK) return rc;
    const int grid = grid_for(m, kDgThreads, sm_count, 8);
    k_dg_run_start<<<grid, kDgThreads, 0, stream>>>(keys, m, (uint64_t)n_verts, w.start);
    // level l holds `size` slots; runs at most `len` long; it forwards into the next level while len > kDgGroup
    uint64_t size = (uint64_t)m, len = (uint64_t)m;
    int cur = 0;
    if (len > kDgGroup) RT_CUDA_TRY(cudaMemsetAsync(w.lv[0].key, 0xff, dg_next_size(size) * 4u, stream));
    k_dg_level0<<<grid, kDgThreads, 0, stream>>>(keys, vals, m, w.start, (uint64_t)n_verts, w.q, uv, grad_vertices,
                                                 w.lv[0]);
    RT_CUDA_TRY(cudaGetLastError());
    while (len > kDgGroup) {
        size = dg_next_size(size);
        len = (len + kDgGroup - 1) / kDgGroup;
        if (len > kDgGroup) RT_CUDA_TRY(cudaMemsetAsync(w.lv[cur ^ 1].key, 0xff, dg_next_size(size) * 4u, stream));
        k_dg_level<<<grid_for((int64_t)size, kDgThreads, sm_count, 8), kDgThreads, 0, stream>>>(
            w.lv[cur], (int64_t)size, grad_vertices, w.lv[cur ^ 1]);
        RT_CUDA_TRY(cudaGetLastError());
        cur ^= 1;
    }
    return RT_OK;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_distance_grad_sizes(int64_t n_points, int64_t n_verts, size_t* workspace_bytes) {
    RT_REQUIRE(n_points >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts && workspace_bytes, RT_ERR_INVALID,
               "rt_distance_grad_sizes: bad arguments (at most %lld vertices)", (long long)(kDgMaxVerts - 1));
    *workspace_bytes = carve_dg(nullptr, n_points < kDgMaxPoints ? n_points : kDgMaxPoints, n_verts, false).total;
    return RT_OK;
}

extern "C" int rt_distance_grad(const rt_ray_desc* points, const rt_trace_opts* opts, const float* grad_out,
                                const float* value, const float* closest, const int32_t* tri_idx, const float* uv,
                                const int32_t* faces, int64_t n_faces, int64_t n_verts, float* grad_points,
                                float* grad_vertices, void* workspace, size_t workspace_bytes, void* stream_) {
    const char* fn = "rt_distance_grad";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    int64_t first = 0, n = 0;
    const int rc = batch_window(fn, points, opts, &first, &n);
    if (rc != RT_OK) return rc;
    RT_REQUIRE(n_faces >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts, RT_ERR_INVALID,
               "%s: bad mesh size (%lld faces, %lld vertices)", fn, (long long)n_faces, (long long)n_verts);
    if (grad_vertices) RT_CUDA_TRY(cudaMemsetAsync(grad_vertices, 0, (size_t)n_verts * 12u, stream));
    if (n == 0 || (!grad_points && !grad_vertices)) return RT_OK;
    RT_REQUIRE(points->origins && grad_out && value && closest && tri_idx && uv, RT_ERR_INVALID, "%s: null input", fn);
    RT_REQUIRE(!grad_vertices || faces || n_faces == 0, RT_ERR_INVALID, "%s: null faces", fn);

    DgPointParams p{};
    p.points = points->origins;
    for (int a = 0; a < 4; ++a) { p.shape[a] = points->shape[a]; p.stride[a] = points->o_stride[a]; }
    p.packed = batch_packed(points->shape, points->o_stride) ? 1 : 0;
    p.first = first;
    p.grad_out = grad_out; p.value = value; p.closest = closest; p.tri = tri_idx; p.faces = faces;
    p.n_faces = n_faces; p.n_verts = n_verts;
    p.grad_points = grad_points;

    if (!grad_vertices) {   // one pass, no sort
        RT_REQUIRE((n + kDgThreads - 1) / kDgThreads < ((int64_t)1 << 31), RT_ERR_INVALID,
                   "%s: batch of %lld points too large for one launch", fn, (long long)n);
        p.n = n; p.base = 0;
        k_dg_points<<<(unsigned)((n + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
        RT_CUDA_TRY(cudaGetLastError());
        return RT_OK;
    }

    // the largest window whose workspace fits
    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    const int64_t win = dg_window(n, n_verts, false, workspace_bytes);
    RT_REQUIRE(win > 0, RT_ERR_SIZE, "%s: workspace %zu < %zu (one point)", fn, workspace_bytes,
               carve_dg(nullptr, 1, n_verts, false).total);
    const DgWorkspace w = carve_dg(workspace, win, n_verts, false);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    const int passes = dg_sort_passes(n_verts);
    p.q = w.q; p.keys = w.keys; p.vals = w.vals;
    for (int64_t base = 0; base < n; base += win) {
        const int64_t nw = n - base < win ? n - base : win;
        p.n = nw; p.base = base;
        k_dg_points<<<(unsigned)((nw + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
        RT_CUDA_TRY(cudaGetLastError());
        const int rc = dg_reduce_window(w, nw, n_verts, uv + 2 * base, passes, dev.sm_count, grad_vertices, stream);
        if (rc != RT_OK) return rc;
    }
    return RT_OK;
}

extern "C" int rt_ray_grad_sizes(int64_t n_rows, int64_t n_verts, size_t* workspace_bytes) {
    RT_REQUIRE(n_rows >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts && workspace_bytes, RT_ERR_INVALID,
               "rt_ray_grad_sizes: bad arguments (at most %lld vertices)", (long long)(kDgMaxVerts - 1));
    *workspace_bytes = carve_dg(nullptr, n_rows < kDgMaxPoints ? n_rows : kDgMaxPoints, n_verts, true).total;
    return RT_OK;
}

extern "C" int rt_ray_grad(const rt_ray_desc* rays, const rt_trace_opts* opts, int64_t n_rows, const int32_t* row_ray,
                           const int32_t* tri_idx, const float* grad_loc, const float* grad_uv, const float* vertices,
                           int64_t n_verts, const int32_t* faces, int64_t n_faces, float* grad_origins,
                           float* grad_directions, float* grad_vertices, void* workspace, size_t workspace_bytes,
                           void* stream_) {
    const char* fn = "rt_ray_grad";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    int64_t first = 0, window = 0;
    const int rc = batch_window(fn, rays, opts, &first, &window);
    if (rc != RT_OK) return rc;
    RT_REQUIRE(n_rows >= 0 && n_faces >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts, RT_ERR_INVALID,
               "%s: bad sizes (%lld rows, %lld faces, %lld vertices)", fn, (long long)n_rows, (long long)n_faces,
               (long long)n_verts);
    // no rows at all (every ray missed): any row_ray, NULL included, and every gradient is +0
    RT_REQUIRE(row_ray != nullptr || n_rows == window || n_rows == 0, RT_ERR_INVALID,
               "%s: without row_ray there must be one row per ray of the window (%lld rows, %lld rays)", fn,
               (long long)n_rows, (long long)window);
    if (grad_vertices) RT_CUDA_TRY(cudaMemsetAsync(grad_vertices, 0, (size_t)n_verts * 12u, stream));
    if (row_ray || n_rows == 0) {       // rays without rows get +0
        if (grad_origins) RT_CUDA_TRY(cudaMemsetAsync(grad_origins, 0, (size_t)window * 12u, stream));
        if (grad_directions) RT_CUDA_TRY(cudaMemsetAsync(grad_directions, 0, (size_t)window * 12u, stream));
    }
    if (n_rows == 0 || (!grad_origins && !grad_directions && !grad_vertices)) return RT_OK;
    RT_REQUIRE(rays->origins && rays->directions && tri_idx, RT_ERR_INVALID, "%s: null input", fn);
    RT_REQUIRE((vertices || n_verts == 0) && (faces || n_faces == 0), RT_ERR_INVALID, "%s: null mesh", fn);

    RgRowParams p{};
    p.origins = rays->origins; p.directions = rays->directions;
    for (int a = 0; a < 4; ++a) {
        p.shape[a] = rays->shape[a]; p.o_stride[a] = rays->o_stride[a]; p.d_stride[a] = rays->d_stride[a];
    }
    p.o_packed = batch_packed(rays->shape, rays->o_stride) ? 1 : 0;
    p.d_packed = batch_packed(rays->shape, rays->d_stride) ? 1 : 0;
    p.first = first; p.window = window; p.n_rows = n_rows;
    p.row_ray = row_ray; p.tri = tri_idx; p.grad_loc = grad_loc; p.grad_uv = grad_uv;
    p.mesh = RgMesh{vertices, n_verts, faces, n_faces};
    p.grad_origins = grad_origins; p.grad_directions = grad_directions;

    if (!grad_vertices) {   // one pass, no sort
        RT_REQUIRE((n_rows + kDgThreads - 1) / kDgThreads < ((int64_t)1 << 31), RT_ERR_INVALID,
                   "%s: %lld rows too many for one launch", fn, (long long)n_rows);
        p.n = n_rows; p.base = 0;
        k_rg_rows<<<(unsigned)((n_rows + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
        RT_CUDA_TRY(cudaGetLastError());
        return RT_OK;
    }

    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    const int64_t win = dg_window(n_rows, n_verts, true, workspace_bytes);
    RT_REQUIRE(win > 0, RT_ERR_SIZE, "%s: workspace %zu < %zu (one row)", fn, workspace_bytes,
               carve_dg(nullptr, 1, n_verts, true).total);
    const DgWorkspace w = carve_dg(workspace, win, n_verts, true);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    const int passes = dg_sort_passes(n_verts);
    p.q = w.q; p.w = w.w; p.keys = w.keys; p.vals = w.vals;
    for (int64_t base = 0; base < n_rows; base += win) {
        const int64_t nw = n_rows - base < win ? n_rows - base : win;
        p.n = nw; p.base = base;
        k_rg_rows<<<(unsigned)((nw + kDgThreads - 1) / kDgThreads), kDgThreads, 0, stream>>>(p);
        RT_CUDA_TRY(cudaGetLastError());
        const int rc = dg_reduce_window(w, nw, n_verts, w.w, passes, dev.sm_count, grad_vertices, stream);
        if (rc != RT_OK) return rc;
    }
    return RT_OK;
}
