// rt_distgrad.cu — every backward pass of the C ABI, from the forward's outputs alone:
//   rt_distance_grad  the point-to-mesh distance w.r.t. the query points and the mesh vertices (DESIGN.md §4.9), from
//                     the outputs of rt_closest_point or rt_signed_distance_closest;
//   rt_ray_grad       hit locations and barycentrics w.r.t. the rays and the mesh vertices (§4.10);
//   rt_scene_ray_grad, rt_scene_distance_grad
//                     the instanced-scene closest hit and point distance w.r.t. the rays or points, the instance
//                     transforms and the member vertices (§4.13).
//
// Per row window, with the arithmetic of rt_distgrad.cuh, rt_raygrad.cuh and rt_scenegrad.cuh:
//   1. one thread per row: the row's own gradient (grad_points, or grad_origins and grad_directions of the ray whose
//      rows it heads) and, when a vertex or transform gradient is wanted, the row's record (mesh points q: 12 B; hit
//      rows q and w: 12 + 8 B; scene rows q, q_obj, x, w: 44 B) and its (key, pair index) pairs: three vertex keys,
//      and for scene rows four transform-column keys of the joint key space [member vertices | 4 I transform columns];
//   2. the builder's stable onesweep sort of the pairs on the low bits of the key (ceil(log2(n_keys + 1)) bits, at
//      most 4 passes): each key's pairs become one run, in ascending pair order;
//   3. the run starts, then the tree reduction: level 0 sums groups of kDgGroup pairs of a run, every further level
//      groups of kDgGroup sums of the level below; a run that fits one group is added to the accumulator (mesh rows:
//      grad_vertices; scene rows: a workspace accumulator that one kernel finally copies to grad_vertices and,
//      transposed, to grad_transforms).
// Nothing is atomic and every sum has one fixed order, so the result does not depend on the launch.
#include "rt_api.h"
#include "rt_distgrad.cuh"
#include "rt_raygrad.cuh"
#include "rt_scenegrad.cuh"

namespace rt {

constexpr int kDgThreads = 256;

// blocks of a launch with one thread per row
inline unsigned row_blocks(int64_t n) { return (unsigned)((n + kDgThreads - 1) / kDgThreads); }

// Shape, strides and batch_packed of the origins and directions of an rt_ray_desc, as the row kernels read them
struct BatchLayout {
    int64_t shape[4], o_stride[4], d_stride[4];
    int o_packed, d_packed;
};
static BatchLayout batch_layout(const rt_ray_desc* d) {
    BatchLayout b;
    for (int a = 0; a < 4; ++a) { b.shape[a] = d->shape[a]; b.o_stride[a] = d->o_stride[a]; b.d_stride[a] = d->d_stride[a]; }
    b.o_packed = batch_packed(d->shape, d->o_stride) ? 1 : 0;
    b.d_packed = batch_packed(d->shape, d->d_stride) ? 1 : 0;
    return b;
}

// ------------------------------------------------------------------ row kernels (step 1)
struct DgPointParams {
    const float* points;
    BatchLayout b;
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
    const int64_t o = batch_offset(p.b.shape, p.b.o_stride, p.b.o_packed, r);
    const int64_t os = p.b.o_stride[3];
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

// The hit rows of rt_ray_grad and rt_scene_ray_grad: the rays, the row -> ray map, the incoming gradients and the
// per-ray outputs.
struct HitRows {
    const float* origins;
    const float* directions;
    BatchLayout b;
    int64_t first;               // batch index of window ray 0
    int64_t window;              // rays in the window
    int64_t n_rows;
    const int32_t* row_ray;      // [n_rows] or null (row j is ray j)
    const float* grad_loc;       // [n_rows, 3] or null
    const float* grad_uv;        // [n_rows, 2] or null
    float* grad_origins;         // [window, 3] or null
    float* grad_directions;      // [window, 3] or null
};

// ray of row j in the window, or -1 for a row_ray outside [0, window)
__device__ __forceinline__ int64_t hit_ray(const HitRows& h, int64_t j) {
    const int64_t ray = h.row_ray ? (int64_t)h.row_ray[j] : j;
    return ray >= 0 && ray < h.window ? ray : -1;
}

// What hit row j reads: its ray (or -1), o, d, g_L and g_U; all +0 for ray -1
struct HitIn { int64_t ray; float o[3], d[3], gl[3], gu0, gu1; };

__device__ __forceinline__ HitIn hit_in(const HitRows& h, int64_t j) {
    HitIn in;
    in.ray = hit_ray(h, j);
    for (int c = 0; c < 3; ++c) in.o[c] = in.d[c] = in.gl[c] = 0.0f;
    in.gu0 = in.gu1 = 0.0f;
    if (in.ray < 0) return in;
    const int64_t b = h.first + in.ray;
    const int64_t oo = batch_offset(h.b.shape, h.b.o_stride, h.b.o_packed, b);
    const int64_t od = batch_offset(h.b.shape, h.b.d_stride, h.b.d_packed, b);
    const int64_t os = h.b.o_stride[3], ds = h.b.d_stride[3];
    in.o[0] = h.origins[oo]; in.o[1] = h.origins[oo + os]; in.o[2] = h.origins[oo + 2 * os];
    in.d[0] = h.directions[od]; in.d[1] = h.directions[od + ds]; in.d[2] = h.directions[od + 2 * ds];
    if (h.grad_loc) { in.gl[0] = h.grad_loc[3 * j]; in.gl[1] = h.grad_loc[3 * j + 1]; in.gl[2] = h.grad_loc[3 * j + 2]; }
    if (h.grad_uv) { in.gu0 = h.grad_uv[2 * j]; in.gu1 = h.grad_uv[2 * j + 1]; }
    return in;
}

// When row j heads its ray's rows: the ray's grad_origins and grad_directions (rg_ray_sums; eval(k, RgRow&) evaluates
// row k)
template <class Eval>
__device__ __forceinline__ void hit_ray_grads(const HitRows& h, int64_t j, const Eval& eval) {
    if ((!h.grad_origins && !h.grad_directions) || !rg_head(j, h.row_ray)) return;
    const int64_t ray = hit_ray(h, j);
    if (ray < 0) return;
    float go[3], gd[3];
    rg_ray_sums(j, h.n_rows, h.row_ray, eval, go, gd);
    if (h.grad_origins) {
        h.grad_origins[3 * ray] = go[0]; h.grad_origins[3 * ray + 1] = go[1]; h.grad_origins[3 * ray + 2] = go[2];
    }
    if (h.grad_directions) {
        h.grad_directions[3 * ray] = gd[0]; h.grad_directions[3 * ray + 1] = gd[1]; h.grad_directions[3 * ray + 2] = gd[2];
    }
}

struct RgRowParams {
    HitRows h;
    int64_t n;                   // rows in this launch, [base, base + n)
    int64_t base;
    const int32_t* tri;
    RgMesh mesh;
    float* q;                    // [n, 3] or null (no vertex gradient)
    float* w;                    // [n, 2]
    uint64_t* keys;              // [3 n]
    uint32_t* vals;              // [3 n]
};

__device__ __forceinline__ bool rg_eval(const RgRowParams& p, int64_t j, RgRow& r) {
    const HitIn in = hit_in(p.h, j);
    if (in.ray < 0) return rg_row(in.o, in.d, in.gl, in.gu0, in.gu1, -1, p.mesh, r);
    return rg_row(in.o, in.d, in.gl, in.gu0, in.gu1, p.tri[j], p.mesh, r);
}

__global__ void __launch_bounds__(kDgThreads) k_rg_rows(const __grid_constant__ RgRowParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t j = p.base + i;
    hit_ray_grads(p.h, j, [&](int64_t k, RgRow& r) { rg_eval(p, k, r); });
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
    HitRows h;
    int64_t n, base;             // rows of this launch, [base, base + n)
    const int32_t* inst;
    const int32_t* tri;
    SgPairsOut out;
};

__device__ __forceinline__ bool sg_hit_eval(const SgHitParams& p, const SgScene& sc, int64_t j, RgRow& rr, SgRow& r,
                                            uint64_t key[3]) {
    const HitIn in = hit_in(p.h, j);
    if (in.ray < 0) return sg_hit_row(sc, -1, -1, in.o, in.d, in.gl, in.gu0, in.gu1, rr, r, key);
    return sg_hit_row(sc, p.inst[j], p.tri[j], in.o, in.d, in.gl, in.gu0, in.gu1, rr, r, key);
}

__global__ void __launch_bounds__(kDgThreads) k_sg_hit_rows(const __grid_constant__ SgHitParams p) {
    const int64_t i = (int64_t)blockIdx.x * kDgThreads + threadIdx.x;
    if (i >= p.n) return;
    const int64_t j = p.base + i;
    const SgScene sc = sg_scene_of(p.scene);
    hit_ray_grads(p.h, j, [&](int64_t k, RgRow& rr) {
        SgRow r;
        uint64_t key[3];
        sg_hit_eval(p, sc, k, rr, r, key);
    });
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
    BatchLayout b;
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
    const int64_t o = batch_offset(p.b.shape, p.b.o_stride, p.b.o_packed, p.first + w);
    const int64_t os = p.b.o_stride[3];
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

// ------------------------------------------------------------------ reduction kernels (step 3) and the scene outputs
// The level-0 contribution of pair e: -w_k q_i of mesh rows (q and uv of the window; w for hit rows), sg_contrib of
// scene rows.
struct MeshContrib {
    const float* q;
    const float* uv;
    __device__ void operator()(uint32_t e, float out[3]) const { dg_contrib(q, uv, e, out); }
};
struct SceneContrib {
    const float* rec;
    int slot0, n_slots;
    __device__ void operator()(uint32_t e, float out[3]) const { sg_contrib(rec, slot0, n_slots, e, out); }
};

__global__ void __launch_bounds__(kDgThreads) k_dg_run_start(const uint64_t* keys, int64_t m, uint64_t n_keys,
                                                             uint32_t* start) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < m; j += stride)
        dg_run_start((uint64_t)j, keys, n_keys, start);
}

template <class Contrib>
__global__ void __launch_bounds__(kDgThreads) k_dg_level0(const uint64_t* keys, const uint32_t* vals, int64_t m,
                                                          const uint32_t* start, uint64_t n_keys, const Contrib contrib,
                                                          float* acc, DgLevel next) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < m; j += stride)
        dg_level0_with((uint64_t)j, (uint64_t)m, keys, vals, start, n_keys, contrib, acc, next);
}

__global__ void __launch_bounds__(kDgThreads) k_dg_level(DgLevel cur, int64_t size, float* acc, DgLevel next) {
    const int64_t stride = (int64_t)gridDim.x * kDgThreads;
    for (int64_t j = (int64_t)blockIdx.x * kDgThreads + threadIdx.x; j < size; j += stride)
        dg_level_at((uint64_t)j, (uint64_t)size, cur, acc, next);
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

// ------------------------------------------------------------------ the windowed driver
// What a window of rows needs: per-row record regions, pairs per row over n_keys keys, the window limit and whether
// the workspace holds the accumulator [n_keys, 3] (scene rows; mesh rows sum into grad_vertices).
struct DgLayout {
    size_t rec_bytes[2];
    int pairs;
    int64_t max_rows;            // a window's pairs must fit one sort call
    int64_t n_keys;
    bool acc;
};
static DgLayout mesh_layout(int64_t n_verts, bool hit_rows) {
    return DgLayout{{12u, hit_rows ? 8u : 0u}, 3, kDgMaxPoints, n_verts, false};
}

// Workspace of a window of w rows: the record regions, keys, values, sort workspace, run starts, two level buffers,
// the accumulator.  Regions of 0 bytes take no space.
struct DgWorkspace {
    void* rec[2];
    uint64_t* keys;
    uint32_t* vals;
    void* sort_ws;
    uint32_t* start;
    DgLevel lv[2];
    float* acc;
    size_t total;
};
static DgWorkspace carve_dg(void* base, int64_t w, const DgLayout& l) {
    const int64_t m = l.pairs * w;
    const uint64_t slots = dg_next_size((uint64_t)m);
    size_t sb = 0;
    rt_sort_sizes(m, &sb);
    const size_t sizes[13] = {(size_t)w * l.rec_bytes[0], (size_t)w * l.rec_bytes[1], (size_t)m * 8u, (size_t)m * 4u,
                              sb, (size_t)l.n_keys * 4u, slots * 4u, slots * 4u, slots * 12u, slots * 4u, slots * 4u,
                              slots * 12u, l.acc ? (size_t)l.n_keys * 12u : 0u};
    size_t off[14];
    off[0] = 0;
    for (int i = 0; i < 13; ++i) off[i + 1] = off[i] + align_up_sz(sizes[i], 256);
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    auto at = [&](int i) { return p ? p + off[i] : nullptr; };
    DgWorkspace ws;
    ws.rec[0] = at(0);
    ws.rec[1] = l.rec_bytes[1] ? at(1) : nullptr;
    ws.keys = reinterpret_cast<uint64_t*>(at(2));
    ws.vals = reinterpret_cast<uint32_t*>(at(3));
    ws.sort_ws = at(4);
    ws.start = reinterpret_cast<uint32_t*>(at(5));
    for (int b = 0; b < 2; ++b)
        ws.lv[b] = DgLevel{reinterpret_cast<uint32_t*>(at(6 + 3 * b)), reinterpret_cast<uint32_t*>(at(7 + 3 * b)),
                           reinterpret_cast<float*>(at(8 + 3 * b))};
    ws.acc = l.acc ? reinterpret_cast<float*>(at(12)) : nullptr;
    ws.total = off[13];
    return ws;
}

// The largest window of at most n (and max_rows) rows whose workspace fits workspace_bytes; 0 when not even one fits.
static int64_t dg_window(int64_t n, const DgLayout& l, size_t workspace_bytes) {
    int64_t win = n < l.max_rows ? n : l.max_rows;
    if (carve_dg(nullptr, win, l).total > workspace_bytes) {
        int64_t lo = 0, hi = win;                       // fits(lo), !fits(hi)
        while (hi - lo > 1) {
            const int64_t mid = lo + (hi - lo) / 2;
            (carve_dg(nullptr, mid, l).total <= workspace_bytes ? lo : hi) = mid;
        }
        win = lo;
    }
    return win;
}

// Steps 2 and 3 for the m pairs of one window at w.keys / w.vals: the sort on the low 8 * passes key bits, the run
// starts, level 0 with the window's contributions and the further levels.  Each key below n_keys adds its sum to
// acc[key].
template <class Contrib>
static int dg_reduce(const DgWorkspace& w, int64_t m, int64_t n_keys, int passes, int sm_count, const Contrib& contrib,
                     float* acc, cudaStream_t stream) {
    uint64_t* keys = nullptr;
    uint32_t* vals = nullptr;
    const int rc = sort_pairs_low(w.keys, w.vals, m, w.sort_ws, passes, &keys, &vals, stream);
    if (rc != RT_OK) return rc;
    const int grid = grid_for(m, kDgThreads, sm_count, 8);
    k_dg_run_start<<<grid, kDgThreads, 0, stream>>>(keys, m, (uint64_t)n_keys, w.start);
    // level l holds `size` slots; runs at most `len` long; it forwards into the next level while len > kDgGroup
    uint64_t size = (uint64_t)m, len = (uint64_t)m;
    int cur = 0;
    if (len > kDgGroup) RT_CUDA_TRY(cudaMemsetAsync(w.lv[0].key, 0xff, dg_next_size(size) * 4u, stream));
    k_dg_level0<<<grid, kDgThreads, 0, stream>>>(keys, vals, m, w.start, (uint64_t)n_keys, contrib, acc, w.lv[0]);
    RT_CUDA_TRY(cudaGetLastError());
    while (len > kDgGroup) {
        size = dg_next_size(size);
        len = (len + kDgGroup - 1) / kDgGroup;
        if (len > kDgGroup) RT_CUDA_TRY(cudaMemsetAsync(w.lv[cur ^ 1].key, 0xff, dg_next_size(size) * 4u, stream));
        k_dg_level<<<grid_for((int64_t)size, kDgThreads, sm_count, 8), kDgThreads, 0, stream>>>(
            w.lv[cur], (int64_t)size, acc, w.lv[cur ^ 1]);
        RT_CUDA_TRY(cudaGetLastError());
        cur ^= 1;
    }
    return RT_OK;
}

// Runs the row launch rows(n, base, ws) over rows [0, n_rows).  Without a sum to form (reduce false): one launch over
// every row, ws null.  Else window by window: each launch writes its window's records and pairs into *ws and returns
// the contribution of its pairs (MeshContrib or SceneContrib), which dg_reduce adds into acc, or into the workspace
// accumulator (zeroed first) when the layout holds one; then finish(acc, sm_count).  The error texts call a row a
// point when `points`.
template <class Rows, class Finish>
static int dg_run(const char* fn, bool points, int64_t n_rows, bool reduce, const DgLayout& l, void* workspace,
                  size_t workspace_bytes, float* acc, const Rows& rows, const Finish& finish, cudaStream_t stream) {
    if (!reduce) {
        RT_REQUIRE((n_rows + kDgThreads - 1) / kDgThreads < ((int64_t)1 << 31), RT_ERR_INVALID,
                   points ? "%s: batch of %lld points too large for one launch" : "%s: %lld rows too many for one launch",
                   fn, (long long)n_rows);
        rows(n_rows, 0, nullptr);
        RT_CUDA_TRY(cudaGetLastError());
        return RT_OK;
    }
    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    const int64_t win = dg_window(n_rows, l, workspace_bytes);
    RT_REQUIRE(win > 0, RT_ERR_SIZE, "%s: workspace %zu < %zu (one %s)", fn, workspace_bytes,
               carve_dg(nullptr, 1, l).total, points ? "point" : "row");
    const DgWorkspace w = carve_dg(workspace, win, l);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    if (l.acc) {
        acc = w.acc;
        RT_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)l.n_keys * 12u, stream));
    }
    const int passes = dg_sort_passes(l.n_keys);
    for (int64_t base = 0; base < n_rows; base += win) {
        const int64_t nw = n_rows - base < win ? n_rows - base : win;
        const auto contrib = rows(nw, base, &w);
        RT_CUDA_TRY(cudaGetLastError());
        const int rc = dg_reduce(w, l.pairs * nw, l.n_keys, passes, dev.sm_count, contrib, acc, stream);
        if (rc != RT_OK) return rc;
    }
    return finish(acc, dev.sm_count);
}

static int no_finish(const float*, int) { return RT_OK; }

// ------------------------------------------------------------------ scene rows
// The slots a call emits: vertex slots 0..2 and / or transform slots 3..6
static void sg_slots(bool transforms, bool vertices, int* slot0, int* n_slots) {
    *slot0 = vertices ? 0 : 3;
    *n_slots = (vertices ? 3 : 0) + (transforms ? 4 : 0);
}
static DgLayout scene_layout(int n_slots, int64_t n_keys) {
    return DgLayout{{4u * kSgRowFloats, 0u}, n_slots, kSgMaxRows, n_keys, true};
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

// dg_run over scene rows: the row kernel `launch(n, base, out)` emits the pairs of the wanted slots into out; the
// accumulator is copied to grad_vertices and grad_transforms at the end.
template <class Launch>
static int sg_run(const char* fn, bool points, int64_t n_rows, int64_t n_inst, int64_t n_verts, int64_t n_keys,
                  float* grad_transforms, float* grad_vertices, void* workspace, size_t workspace_bytes,
                  const Launch& launch, cudaStream_t stream) {
    int slot0 = 0, n_slots = 0;
    sg_slots(grad_transforms != nullptr, grad_vertices != nullptr, &slot0, &n_slots);
    return dg_run(fn, points, n_rows, n_slots > 0, scene_layout(n_slots, n_keys), workspace, workspace_bytes, nullptr,
                  [&](int64_t n, int64_t base, const DgWorkspace* w) {
                      SgPairsOut out{};
                      out.n_keys = (uint64_t)n_keys;
                      if (w) {
                          out.rec = static_cast<float*>(w->rec[0]); out.keys = w->keys; out.vals = w->vals;
                          out.slot0 = slot0; out.n_slots = n_slots;
                      }
                      launch(n, base, out);
                      return SceneContrib{out.rec, slot0, n_slots};
                  },
                  [&](const float* acc, int sm_count) -> int {
                      const int64_t total = (grad_vertices ? 3 * n_verts : 0) + (grad_transforms ? 12 * n_inst : 0);
                      if (total > 0) {
                          k_sg_outputs<<<grid_for(total, kDgThreads, sm_count, 8), kDgThreads, 0, stream>>>(
                              acc, n_verts, n_inst, grad_vertices, grad_transforms);
                          RT_CUDA_TRY(cudaGetLastError());
                      }
                      return RT_OK;
                  },
                  stream);
}

}  // namespace rt

using namespace rt;

extern "C" int rt_distance_grad_sizes(int64_t n_points, int64_t n_verts, size_t* workspace_bytes) {
    RT_REQUIRE(n_points >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts && workspace_bytes, RT_ERR_INVALID,
               "rt_distance_grad_sizes: bad arguments (at most %lld vertices)", (long long)(kDgMaxVerts - 1));
    *workspace_bytes = carve_dg(nullptr, n_points < kDgMaxPoints ? n_points : kDgMaxPoints,
                                mesh_layout(n_verts, false)).total;
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
    p.b = batch_layout(points);
    p.first = first;
    p.grad_out = grad_out; p.value = value; p.closest = closest; p.tri = tri_idx; p.faces = faces;
    p.n_faces = n_faces; p.n_verts = n_verts;
    p.grad_points = grad_points;
    return dg_run(fn, true, n, grad_vertices != nullptr, mesh_layout(n_verts, false), workspace, workspace_bytes,
                  grad_vertices,
                  [&](int64_t nw, int64_t base, const DgWorkspace* w) {
                      p.n = nw; p.base = base;
                      if (w) { p.q = static_cast<float*>(w->rec[0]); p.keys = w->keys; p.vals = w->vals; }
                      k_dg_points<<<row_blocks(nw), kDgThreads, 0, stream>>>(p);
                      return MeshContrib{p.q, uv + 2 * base};
                  },
                  no_finish, stream);
}

extern "C" int rt_ray_grad_sizes(int64_t n_rows, int64_t n_verts, size_t* workspace_bytes) {
    RT_REQUIRE(n_rows >= 0 && n_verts >= 0 && n_verts < kDgMaxVerts && workspace_bytes, RT_ERR_INVALID,
               "rt_ray_grad_sizes: bad arguments (at most %lld vertices)", (long long)(kDgMaxVerts - 1));
    *workspace_bytes = carve_dg(nullptr, n_rows < kDgMaxPoints ? n_rows : kDgMaxPoints, mesh_layout(n_verts, true)).total;
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
    p.h = HitRows{rays->origins, rays->directions, batch_layout(rays), first, window, n_rows, row_ray, grad_loc, grad_uv,
                  grad_origins, grad_directions};
    p.tri = tri_idx;
    p.mesh = RgMesh{vertices, n_verts, faces, n_faces};
    return dg_run(fn, false, n_rows, grad_vertices != nullptr, mesh_layout(n_verts, true), workspace, workspace_bytes,
                  grad_vertices,
                  [&](int64_t nw, int64_t base, const DgWorkspace* w) {
                      p.n = nw; p.base = base;
                      if (w) {
                          p.q = static_cast<float*>(w->rec[0]); p.w = static_cast<float*>(w->rec[1]);
                          p.keys = w->keys; p.vals = w->vals;
                      }
                      k_rg_rows<<<row_blocks(nw), kDgThreads, 0, stream>>>(p);
                      return MeshContrib{p.q, p.w};
                  },
                  no_finish, stream);
}

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
    *workspace_bytes = carve_dg(nullptr, w > 0 ? w : 1, scene_layout(n_slots, n_verts_total + 4 * n_inst)).total;
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
    p.h = HitRows{rays->origins, rays->directions, batch_layout(rays), first, window, n_rows, row_ray, grad_loc, grad_uv,
                  grad_origins, grad_directions};
    p.inst = inst_idx; p.tri = tri_idx;
    return sg_run(fn, false, n_rows, n_inst, n_verts_total, n_keys, grad_transforms, grad_vertices, workspace,
                  workspace_bytes,
                  [&](int64_t n, int64_t base, const SgPairsOut& out) {
                      p.n = n; p.base = base; p.out = out;
                      k_sg_hit_rows<<<row_blocks(n), kDgThreads, 0, stream>>>(p);
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
    p.b = batch_layout(points);
    p.first = first;
    p.grad_out = grad_out; p.value = value; p.closest = closest; p.inst = inst_idx; p.tri = tri_idx; p.uv = uv;
    p.grad_points = grad_points;
    return sg_run(fn, false, n, n_inst, n_verts_total, n_keys, grad_transforms, grad_vertices, workspace, workspace_bytes,
                  [&](int64_t nw, int64_t base, const SgPairsOut& out) {
                      p.n = nw; p.base = base; p.out = out;
                      k_sg_point_rows<<<row_blocks(nw), kDgThreads, 0, stream>>>(p);
                  }, stream);
}
