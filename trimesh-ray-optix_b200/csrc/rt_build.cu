// rt_build.cu — BVH construction on the GPU (sm_100a), C ABI entry points rt_bvh_* / rt_sort_*.
//
// Replaces OptixAccelStructureWrapperCPP::buildAccelStructure (triro/backend/ray.cpp:27-100):
//   optixAccelComputeMemoryUsage -> rt_bvh_sizes
//   optixAccelBuild + optixAccelCompact -> rt_bvh_build
// Pipeline (all on the caller's stream, no host synchronisation):
//   k_scene_bounds  triangle boxes -> scene box (ordered-uint atomics)
//   k_morton        63-bit Morton code of each triangle's box centre
//   onesweep sort   rt_sort.cuh
//   k_karras        binary radix tree over the sorted codes (Karras 2012)
//   k_refit         bottom-up boxes with one atomic counter per inner node
//   k_collapse      persistent cooperative kernel, one grid-wide level per iteration:
//                   greedy surface-area collapse to 8-wide quantised nodes + triangle records
//   k_finalize      blob header, zeroed alignment gaps of the used prefix
#include <cooperative_groups.h>
#include <string.h>
#include "rt_api.h"
#include "rt_build_core.cuh"
#include "rt_sort.cuh"

namespace cg = cooperative_groups;

namespace rt {

// ------------------------------------------------------------------ error plumbing (shared by all TUs)
char* error_buffer() {
    static thread_local char buf[512] = {0};
    return buf;
}
int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}
int device_info(DeviceInfo* out) {
    static thread_local int cached_dev = -1;
    static thread_local int cached_sms = 0;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); out->device = -1; out->sm_count = 0; return RT_ERR_CUDA; }
    if (dev != cached_dev) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
            cudaGetLastError(); out->device = -1; out->sm_count = 0; return RT_ERR_CUDA;
        }
        cached_dev = dev; cached_sms = sms;
    }
    out->device = cached_dev; out->sm_count = cached_sms;
    return RT_OK;
}

// ------------------------------------------------------------------ build state in the workspace
struct BuildState {
    uint32_t bounds_lo[3];   // ordered-uint encoded floats
    uint32_t bounds_hi[3];
    uint32_t node_count;
    uint32_t tri_count;
    uint32_t depth;
    uint32_t bad_index;      // number of faces with an out-of-range vertex index
    uint32_t pad[6];
};

struct Workspace {
    BuildState* state;
    uint64_t* keys;
    uint32_t* vals;
    void* sort_ws;
    uint32_t *left, *right, *first, *last, *parent, *flags, *wide_src, *wide_parent;
    BBox* box;
    size_t total;
};

static Workspace carve_workspace(void* base, int64_t n, uint32_t node_cap) {
    Workspace w;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { uint8_t* q = p ? p + off : nullptr; off += align_up_sz(bytes, 256); return q; };
    const size_t nn = (size_t)(n > 0 ? n : 0);
    const size_t ni = nn > 0 ? nn - 1 : 0;
    w.state = reinterpret_cast<BuildState*>(take(sizeof(BuildState)));
    w.flags = reinterpret_cast<uint32_t*>(take(ni * 4));          // state + flags are zeroed together
    w.keys = reinterpret_cast<uint64_t*>(take(nn * 8));
    w.vals = reinterpret_cast<uint32_t*>(take(nn * 4));
    w.sort_ws = take(sort::workspace_bytes((int64_t)nn));
    w.left = reinterpret_cast<uint32_t*>(take(ni * 4));
    w.right = reinterpret_cast<uint32_t*>(take(ni * 4));
    w.first = reinterpret_cast<uint32_t*>(take(ni * 4));
    w.last = reinterpret_cast<uint32_t*>(take(ni * 4));
    w.parent = reinterpret_cast<uint32_t*>(take((2 * nn) * 4));
    w.wide_src = reinterpret_cast<uint32_t*>(take((size_t)node_cap * 4));
    w.wide_parent = reinterpret_cast<uint32_t*>(take((size_t)node_cap * 4));
    w.box = reinterpret_cast<BBox*>(take((2 * nn) * sizeof(BBox)));
    w.total = off;
    return w;
}

// ------------------------------------------------------------------ kernels
__device__ __forceinline__ bool load_tri(const float* __restrict__ verts, int64_t nv, const int32_t* __restrict__ faces,
                                         int64_t prim, float v[9]) {
    const int32_t r0 = faces[3 * prim], r1 = faces[3 * prim + 1], r2 = faces[3 * prim + 2];
    const bool ok = r0 >= 0 && r0 < nv && r1 >= 0 && r1 < nv && r2 >= 0 && r2 < nv;
    const int32_t i0 = clamp_index(r0, nv), i1 = clamp_index(r1, nv), i2 = clamp_index(r2, nv);
    v[0] = verts[3 * (size_t)i0]; v[1] = verts[3 * (size_t)i0 + 1]; v[2] = verts[3 * (size_t)i0 + 2];
    v[3] = verts[3 * (size_t)i1]; v[4] = verts[3 * (size_t)i1 + 1]; v[5] = verts[3 * (size_t)i1 + 2];
    v[6] = verts[3 * (size_t)i2]; v[7] = verts[3 * (size_t)i2 + 1]; v[8] = verts[3 * (size_t)i2 + 2];
    return ok;
}

__global__ void __launch_bounds__(256) k_init_state(BuildState* st) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        for (int a = 0; a < 3; ++a) { st->bounds_lo[a] = kOrdPosInf; st->bounds_hi[a] = kOrdNegInf; }
        st->node_count = 1u;
    }
}

__global__ void __launch_bounds__(256) k_scene_bounds(const float* __restrict__ verts, int64_t nv,
                                                      const int32_t* __restrict__ faces, int64_t n, BuildState* st) {
    // ordered-uint encoding throughout (rt_build_core.cuh): the box does not depend on the order of the reduction
    uint32_t lo[3] = {kOrdPosInf, kOrdPosInf, kOrdPosInf}, hi[3] = {kOrdNegInf, kOrdNegInf, kOrdNegInf};
    uint32_t bad = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v[9];
        if (!load_tri(verts, nv, faces, i, v)) ++bad;
        const BBox b = tri_bbox(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
        lo[0] = min(lo[0], ord_lo(b.lx)); lo[1] = min(lo[1], ord_lo(b.ly)); lo[2] = min(lo[2], ord_lo(b.lz));
        hi[0] = max(hi[0], ord_hi(b.hx)); hi[1] = max(hi[1], ord_hi(b.hy)); hi[2] = max(hi[2], ord_hi(b.hz));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = min(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = max(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
    }
    // block-level reduction first: one set of atomics per CTA instead of per warp
    __shared__ uint32_t s_lo[8][3], s_hi[8][3];
    __shared__ uint32_t s_bad[8];
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { s_lo[warp][a] = lo[a]; s_hi[warp][a] = hi[a]; }
        s_bad[warp] = bad;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
#pragma unroll
            for (int a = 0; a < 3; ++a) { lo[a] = min(lo[a], s_lo[w][a]); hi[a] = max(hi[a], s_hi[w][a]); }
            bad += s_bad[w];
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (lo[a] != kOrdPosInf) atomicMin(&st->bounds_lo[a], lo[a]);
            if (hi[a] != kOrdNegInf) atomicMax(&st->bounds_hi[a], hi[a]);
        }
        if (bad) atomicAdd(&st->bad_index, bad);
    }
}

__global__ void __launch_bounds__(256) k_morton(const float* __restrict__ verts, int64_t nv,
                                                const int32_t* __restrict__ faces, int64_t n,
                                                const BuildState* __restrict__ st, uint64_t* __restrict__ keys,
                                                uint32_t* __restrict__ vals) {
    float lo[3], hi[3], inv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { lo[a] = ord2f(st->bounds_lo[a]); hi[a] = ord2f(st->bounds_hi[a]); }
    morton_scale(lo, hi, inv);
    const int drop = 3 * (21 - morton_axis_bits(n));      // low bits that do not take part in the ordering
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v[9];
        load_tri(verts, nv, faces, i, v);
        const BBox b = tri_bbox(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
        keys[i] = morton63(0.5f * (b.lx + b.hx), 0.5f * (b.ly + b.hy), 0.5f * (b.lz + b.hz), lo, inv) >> drop;
        vals[i] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(256) k_karras(const uint64_t* __restrict__ keys, int64_t n,
                                                uint32_t* __restrict__ left, uint32_t* __restrict__ right,
                                                uint32_t* __restrict__ first, uint32_t* __restrict__ last,
                                                uint32_t* __restrict__ parent) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n - 1; i += stride) {
        const KarrasNode k = karras_node(keys, n, i);
        left[i] = k.left; right[i] = k.right; first[i] = k.first; last[i] = k.last;
        parent[k.left] = (uint32_t)i;
        parent[k.right] = (uint32_t)i;
        if (i == 0) parent[0] = 0xffffffffu;
    }
}

__device__ __forceinline__ BBox load_box_cg(const BBox* p) {
    const float4 a = __ldcg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldcg(reinterpret_cast<const float4*>(p) + 1);
    BBox r; r.lx = a.x; r.ly = a.y; r.lz = a.z; r.pad0 = 0.f; r.hx = b.x; r.hy = b.y; r.hz = b.z; r.pad1 = 0.f;
    return r;
}
__device__ __forceinline__ void store_box_cg(BBox* p, const BBox& b, uint32_t left = 0u, uint32_t right = 0u) {
    // the pad words of an inner node's record carry its child references (used by the collapse)
    __stcg(reinterpret_cast<float4*>(p), make_float4(b.lx, b.ly, b.lz, __uint_as_float(left)));
    __stcg(reinterpret_cast<float4*>(p) + 1, make_float4(b.hx, b.hy, b.hz, __uint_as_float(right)));
}

// Bottom-up boxes.  One CTA owns a TILE of kRefitTile consecutive leaves (sorted order), one thread per leaf climbs:
// the second thread to arrive at an inner node merges the two child boxes and goes on (Karras 2012).  In sorted Morton
// order every Karras subtree is a contiguous leaf range [first, last] and an inner node's index is one end of its
// range, so for all inner nodes whose range lies inside the tile - all but O(log) per tile - the arrival counter lives
// in SHARED memory and the hand-over between the two children needs only a block-scope fence; only the nodes above a
// tile boundary use the global counters and a device-scope fence.  (Round 1 used global atomics + __threadfence for
// every node: 4.8 ms at 16.8 M triangles.)
constexpr int kRefitTile = 1024;
__global__ void __launch_bounds__(256) k_refit(const float* __restrict__ verts, int64_t nv,
                                               const int32_t* __restrict__ faces, int64_t n,
                                               const uint32_t* __restrict__ sorted_prim,
                                               const uint32_t* __restrict__ left, const uint32_t* __restrict__ right,
                                               const uint32_t* __restrict__ first, const uint32_t* __restrict__ last,
                                               const uint32_t* __restrict__ parent, uint32_t* __restrict__ flags,
                                               BBox* __restrict__ box, uint32_t leaf_max) {
    __shared__ uint32_t s_flags[kRefitTile];
    {
        const int64_t tile = blockIdx.x;                                      // one tile per CTA: no barrier at a tile's end,
        const int64_t a = tile * kRefitTile;                                  // the block scheduler balances uneven climbs
        const int64_t b = (a + kRefitTile < n ? a + kRefitTile : n) - 1;      // leaves [a, b]
        for (int i = threadIdx.x; i < kRefitTile; i += blockDim.x) s_flags[i] = 0u;
        __syncthreads();
        for (int64_t k = a + threadIdx.x; k <= b; k += blockDim.x) {
            float v[9];
            load_tri(verts, nv, faces, (int64_t)sorted_prim[k], v);
            const BBox lb = leaf_bbox(tri_bbox(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]));
            store_box_cg(&box[(n - 1) + k], lb);
            if (n == 1) continue;
            uint32_t me = (uint32_t)((n - 1) + k);
            uint32_t cur = parent[me];
            BBox mine = lb;                                    // box of the subtree this thread has completed ...
            uint32_t mine_count = 1u;                          // ... and its number of triangles
            for (;;) {
                const uint32_t f = first[cur], e = last[cur];
                const bool local = (int64_t)f >= a && (int64_t)e <= b;
                uint32_t arrived;
                if (local) {
                    __threadfence_block();                     // publish box[me] to the CTA before announcing it
                    arrived = atomicAdd(&s_flags[cur - (uint32_t)a], 1u);
                } else {
                    __threadfence();                           // ... to the device
                    arrived = atomicAdd(&flags[cur], 1u);
                }
                if (arrived == 0u) break;                      // first arrival: sibling not ready
                const uint32_t l = left[cur], rr = right[cur];
                const uint32_t sibling = l == me ? rr : l;
                mine = bbox_union(mine, load_box_cg(&box[sibling]));   // L1-bypassing load, ordered after the atomic
                // child references ride in the pad words; bit 31 = "covers more than leaf_max triangles" (the collapse
                // then needs no first/last loads to decide whether a child can be expanded)
                const uint32_t total = e - f + 1u, sib_count = total - mine_count;
                const uint32_t me_bit = mine_count > leaf_max ? 0x80000000u : 0u, sib_bit = sib_count > leaf_max ? 0x80000000u : 0u;
                store_box_cg(&box[cur], mine, l | (l == me ? me_bit : sib_bit), rr | (l == me ? sib_bit : me_bit));
                mine_count = total;
                if (cur == 0u) break;
                me = cur;
                cur = parent[cur];
            }
        }
    }
}

__global__ void __launch_bounds__(128) k_collapse(BinaryTree t, CollapseOut o, const float* __restrict__ verts,
                                                  int64_t nv, const int32_t* __restrict__ faces, BuildState* st) {
    cg::grid_group grid = cg::this_grid();
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t gsize = gridDim.x * blockDim.x;
    uint32_t begin = 0, end = 1, depth = 0;
    while (begin < end) {
        for (uint32_t w = begin + gtid; w < end; w += gsize) collapse_node(t, o, w, verts, nv, faces);
        ++depth;
        __threadfence();
        grid.sync();
        uint32_t new_end = *reinterpret_cast<volatile uint32_t*>(o.node_count);
        if (new_end > o.node_cap) new_end = o.node_cap;
        grid.sync();   // everybody has sampled node_count before the next level allocates
        begin = end;
        end = new_end;
    }
    if (gtid == 0) st->depth = depth;
}

__global__ void __launch_bounds__(256) k_fill_tris(const float* __restrict__ verts, int64_t nv,
                                                   const int32_t* __restrict__ faces, int64_t n,
                                                   const uint32_t* __restrict__ tri_pos,
                                                   const uint32_t* __restrict__ sorted_prim, uint8_t* tris) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        fill_tri_record(tris, (uint32_t)i, tri_pos, sorted_prim, verts, nv, faces);
}

// The (parent << 3 | slot) array of the wide nodes (only rt_bvh_refit reads it) is built in the workspace and placed
// right behind the nodes actually in use (parents_offset_for), so that the used prefix of the blob - what travels over
// NCCL or to disk - is complete: a blob received by broadcast or load can be re-fitted like the original.

__global__ void __launch_bounds__(256) k_place_parents(uint8_t* blob, const BuildState* st, BlobLayout lay,
                                                       const uint32_t* __restrict__ wide_parent) {
    const uint32_t n_nodes = st->node_count < lay.node_cap ? st->node_count : lay.node_cap;
    uint32_t* dst = reinterpret_cast<uint32_t*>(blob + parents_offset_for(lay.nodes_offset, n_nodes));
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes; i += stride) dst[i] = wide_parent[i];
}

// One warp: lane 0 writes the header (and the root of an empty mesh), all lanes zero the alignment gaps inside the
// used prefix, so that the prefix a save() or a broadcast carries depends on the mesh alone (the blob itself comes
// uninitialised from the caller's allocator).
__global__ void k_finalize(rt_blob_header* hdr, const BuildState* st, int64_t n, BlobLayout lay) {
    if (blockIdx.x != 0) return;
    uint8_t* blob = reinterpret_cast<uint8_t*>(hdr);
    const uint32_t n_nodes = n > 0 ? (st->node_count < lay.node_cap ? st->node_count : lay.node_cap) : 1u;
    const uint64_t parents_offset = parents_offset_for(lay.nodes_offset, n_nodes);
    const uint64_t used = used_bytes_for(parents_offset, n_nodes);
    const uint64_t gap[4][2] = {{sizeof(rt_blob_header), lay.tris_offset},
                                {lay.tris_offset + (uint64_t)n * 48u, lay.nodes_offset},
                                {lay.nodes_offset + (uint64_t)n_nodes * 80u, parents_offset},
                                {parents_offset + (uint64_t)n_nodes * 4u, used}};
    for (int g = 0; g < 4; ++g)
        for (uint64_t b = gap[g][0] + threadIdx.x; b < gap[g][1]; b += blockDim.x) blob[b] = 0;
    if (threadIdx.x != 0) return;
    rt_blob_header h;
    memset(&h, 0, sizeof(h));
    h.magic = RT_BLOB_MAGIC;
    h.abi_version = RT_ABI_VERSION;
    h.n_tris = (uint32_t)n;
    h.n_nodes = n_nodes;
    h.depth = n > 0 ? st->depth : 1u;
    h.n_nodes_cap = lay.node_cap;
    h.tris_offset = lay.tris_offset;
    h.nodes_offset = lay.nodes_offset;
    h.parents_offset = parents_offset;
    h.used_bytes = used;
    // an empty mesh has the zero box; a mesh whose triangle boxes are all NaN has the empty box (+inf, -inf)
    for (int a = 0; a < 3; ++a) {
        h.aabb_lo[a] = n > 0 ? ord2f(st->bounds_lo[a]) : 0.0f;
        h.aabb_hi[a] = n > 0 ? ord2f(st->bounds_hi[a]) : 0.0f;
    }
    h.bad_index_faces = n > 0 ? st->bad_index : 0u;
    h.node_overflow = n > 0 ? (st->node_count > lay.node_cap ? 1u : 0u) : 0u;   // must not happen
    *hdr = h;
    if (n == 0) {
        // empty mesh: a root without children, every ray misses
        Node8 nd;
        memset(&nd, 0, sizeof(nd));
        nd.ex = nd.ey = nd.ez = 1;   // imask = trimask = 0: no slot is ever reported
        *reinterpret_cast<Node8*>(blob + lay.nodes_offset) = nd;
        *reinterpret_cast<uint32_t*>(blob + h.parents_offset) = 0xffffffffu;
    }
}

}  // namespace rt

using namespace rt;

extern "C" const char* rt_last_error(void) { return error_buffer(); }
extern "C" int rt_abi_version(void) { return RT_ABI_VERSION; }
extern "C" int rt_device_sm_count(void) {
    DeviceInfo d;
    if (device_info(&d) != RT_OK) return 0;
    return d.sm_count;
}

extern "C" int rt_bvh_sizes(int64_t n_verts, int64_t n_faces, size_t* workspace_bytes, size_t* blob_bytes) {
    RT_REQUIRE(n_verts >= 0 && n_faces >= 0, RT_ERR_INVALID, "rt_bvh_sizes: negative size");
    RT_REQUIRE(n_faces <= (int64_t)1 << 30, RT_ERR_INVALID, "rt_bvh_sizes: more than 2^30 faces");
    RT_REQUIRE(workspace_bytes && blob_bytes, RT_ERR_INVALID, "rt_bvh_sizes: null output pointer");
    const BlobLayout lay = blob_layout(n_faces);
    const Workspace w = carve_workspace(nullptr, n_faces, lay.node_cap);
    *workspace_bytes = w.total;
    *blob_bytes = lay.total_bytes;
    return RT_OK;
}

extern "C" int rt_bvh_build(const float* vertices, int64_t n_verts, const int32_t* faces, int64_t n_faces,
                            void* workspace, size_t workspace_bytes, void* blob, size_t blob_bytes, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    RT_REQUIRE(n_verts >= 0 && n_faces >= 0 && n_faces <= (int64_t)1 << 30, RT_ERR_INVALID,
               "rt_bvh_build: bad sizes (n_verts=%lld n_faces=%lld)", (long long)n_verts, (long long)n_faces);
    RT_REQUIRE(blob && workspace, RT_ERR_INVALID, "rt_bvh_build: null blob/workspace");
    RT_REQUIRE(((uintptr_t)blob & 255) == 0 && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "rt_bvh_build: blob and workspace must be 256-byte aligned");
    RT_REQUIRE(n_faces == 0 || (vertices && faces && n_verts > 0), RT_ERR_INVALID,
               "rt_bvh_build: faces given but vertices/faces pointer null or n_verts == 0");
    const BlobLayout lay = blob_layout(n_faces);
    Workspace w = carve_workspace(workspace, n_faces, lay.node_cap);
    RT_REQUIRE(workspace_bytes >= w.total, RT_ERR_SIZE, "rt_bvh_build: workspace %zu < %zu", workspace_bytes, w.total);
    RT_REQUIRE(blob_bytes >= lay.total_bytes, RT_ERR_SIZE, "rt_bvh_build: blob %zu < %zu", blob_bytes, lay.total_bytes);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "rt_bvh_build: no CUDA device");
    const int64_t n = n_faces;
    uint8_t* blob8 = reinterpret_cast<uint8_t*>(blob);
    rt_blob_header* hdr = reinterpret_cast<rt_blob_header*>(blob8);

    if (n > 0) {
        // state + refit flags
        const size_t zero = align_up_sz(sizeof(BuildState), 256) + align_up_sz((size_t)(n - 1) * 4, 256);
        RT_CUDA_TRY(cudaMemsetAsync(w.state, 0, zero, stream));
        k_init_state<<<1, 32, 0, stream>>>(w.state);
        RT_CUDA_TRY(cudaMemsetAsync(w.wide_src, 0, 4, stream));   // wide node 0 expands binary node 0
        const int g = grid_for(n, 256, dev.sm_count, 8);
        k_scene_bounds<<<g, 256, 0, stream>>>(vertices, n_verts, faces, n, w.state);
        k_morton<<<g, 256, 0, stream>>>(vertices, n_verts, faces, n, w.state, w.keys, w.vals);
        // an odd number of passes leaves the sorted keys / triangle ids in the sort's alternate buffers: use them where they are
        uint64_t* skeys = w.keys; uint32_t* svals = w.vals;
        RT_CUDA_TRY(sort::sort_pairs(w.keys, w.vals, n, w.sort_ws, dev.sm_count, stream, morton_sort_passes(n), &skeys, &svals));
        if (n > 1) k_karras<<<g, 256, 0, stream>>>(skeys, n, w.left, w.right, w.first, w.last, w.parent);
        k_refit<<<(unsigned)((n + kRefitTile - 1) / kRefitTile), 256, 0, stream>>>(
            vertices, n_verts, faces, n, svals, w.left, w.right, w.first, w.last, w.parent, w.flags, w.box,
            (uint32_t)leaf_tris_setting());

        BinaryTree t;
        t.n = n; t.left = w.left; t.right = w.right; t.first = w.first; t.last = w.last; t.box = w.box;
        t.sorted_prim = svals; t.leaf_max = leaf_tris_setting(); t.flagged = 1;
        CollapseOut o;
        o.nodes = blob8 + lay.nodes_offset; o.tris = blob8 + lay.tris_offset; o.wide_src = w.wide_src;
        o.tri_pos = reinterpret_cast<uint32_t*>(skeys);       // the sorted keys are dead once the hierarchy exists (8n bytes, n words needed)
        o.parent = w.wide_parent;
        o.node_count = &w.state->node_count; o.tri_count = &w.state->tri_count; o.node_cap = lay.node_cap;
        int per_sm = 0;
        RT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_collapse, 128, 0));
        RT_REQUIRE(per_sm > 0, RT_ERR_CUDA, "rt_bvh_build: collapse kernel does not fit an SM");
        int cgrid = dev.sm_count * per_sm;
        const int64_t want = (n / 4 + 127) / 128 + 1;     // never more threads than first-level work can use
        if ((int64_t)cgrid > want) cgrid = (int)want;
        BuildState* stp = w.state;
        void* args[] = {&t, &o, (void*)&vertices, (void*)&n_verts, (void*)&faces, &stp};
        RT_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_collapse, dim3(cgrid), dim3(128), args, 0, stream));
        k_fill_tris<<<g, 256, 0, stream>>>(vertices, n_verts, faces, n, o.tri_pos, svals, blob8 + lay.tris_offset);
        k_place_parents<<<grid_for(lay.node_cap, 256, dev.sm_count, 4), 256, 0, stream>>>(blob8, w.state, lay, w.wide_parent);
    }
    k_finalize<<<1, 32, 0, stream>>>(hdr, w.state, n, lay);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

// ------------------------------------------------------------------ refit (same topology, new vertices)
namespace rt {
struct RefitWorkspace {
    BBox* node_box;        // [node_cap]
    uint32_t* counters;    // [node_cap] children that have reported
    size_t total;
};
static RefitWorkspace carve_refit(void* base, uint32_t node_cap) {
    RefitWorkspace w;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    const size_t cb = align_up_sz((size_t)node_cap * 4u, 256);
    w.counters = reinterpret_cast<uint32_t*>(p);
    w.node_box = reinterpret_cast<BBox*>(p ? p + cb : nullptr);
    w.total = cb + align_up_sz((size_t)node_cap * sizeof(BBox), 256);
    return w;
}

__global__ void __launch_bounds__(256) k_refit_tris(const float* __restrict__ verts, int64_t nv,
                                                    const int32_t* __restrict__ faces, int64_t n, uint8_t* tris) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int32_t prim = *reinterpret_cast<const int32_t*>(tris + (size_t)i * 48u + 12);
        write_tri_record(tris, (uint32_t)i, (uint32_t)prim, verts, nv, faces);
    }
}

// one thread per node without inner children starts; the last child to report climbs to the parent
__global__ void __launch_bounds__(128) k_refit_nodes(rt_blob_header* hdr, BBox* node_box, uint32_t* counters) {
    uint8_t* blob = reinterpret_cast<uint8_t*>(hdr);
    uint8_t* nodes = blob + hdr->nodes_offset;
    const uint8_t* tris = blob + hdr->tris_offset;
    const uint32_t* parent = reinterpret_cast<const uint32_t*>(blob + hdr->parents_offset);
    const uint32_t n_nodes = hdr->n_nodes;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t w0 = blockIdx.x * blockDim.x + threadIdx.x; w0 < n_nodes; w0 += stride) {
        if (nodes[(size_t)w0 * 80u + 15] != 0) continue;   // imask != 0: an inner child will take care of it
        uint32_t w = w0;
        for (;;) {
            const BBox nb = refit_node(nodes, tris, w, node_box);
            __stcg(reinterpret_cast<float4*>(&node_box[w]), make_float4(nb.lx, nb.ly, nb.lz, 0.f));
            __stcg(reinterpret_cast<float4*>(&node_box[w]) + 1, make_float4(nb.hx, nb.hy, nb.hz, 0.f));
            if (w == 0u) {
                hdr->aabb_lo[0] = nb.lx; hdr->aabb_lo[1] = nb.ly; hdr->aabb_lo[2] = nb.lz;
                hdr->aabb_hi[0] = nb.hx; hdr->aabb_hi[1] = nb.hy; hdr->aabb_hi[2] = nb.hz;
                break;
            }
            const uint32_t pw = parent[w] >> 3;
            const uint32_t need = (uint32_t)__popc((uint32_t)nodes[(size_t)pw * 80u + 15]);
            __threadfence();
            if (atomicAdd(&counters[pw], 1u) + 1u != need) break;
            w = pw;
        }
    }
}
}  // namespace rt

extern "C" int rt_bvh_refit_sizes(int64_t n_faces, size_t* workspace_bytes) {
    RT_REQUIRE(n_faces >= 0 && n_faces <= (int64_t)1 << 30 && workspace_bytes, RT_ERR_INVALID, "rt_bvh_refit_sizes: bad arguments");
    // bound for any leaf size the blob may have been built with (the node count itself is only known on the device)
    *workspace_bytes = carve_refit(nullptr, wide_node_cap(n_faces, 1)).total;
    return RT_OK;
}

extern "C" int rt_bvh_refit(const float* vertices, int64_t n_verts, const int32_t* faces, int64_t n_faces, void* workspace,
                            size_t workspace_bytes, void* blob, size_t blob_bytes, void* stream_) {
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    RT_REQUIRE(n_verts >= 0 && n_faces >= 0 && n_faces <= (int64_t)1 << 30, RT_ERR_INVALID, "rt_bvh_refit: bad sizes");
    RT_REQUIRE(blob && workspace, RT_ERR_INVALID, "rt_bvh_refit: null blob/workspace");
    RT_REQUIRE(((uintptr_t)blob & 255) == 0 && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "rt_bvh_refit: blob and workspace must be 256-byte aligned");
    // The kernels take every offset and count from the blob's own header (so a blob that arrived by NCCL broadcast or
    // from disk - just its used prefix - re-fits like the original, whatever leaf size it was built with); the host
    // can only bound the sizes: header + triangle records + one node + its parent word.
    const uint32_t node_cap = wide_node_cap(n_faces, 1);
    RT_REQUIRE(blob_bytes >= RT_BLOB_HEADER_BYTES + (size_t)n_faces * 48u + 84u, RT_ERR_SIZE,
               "rt_bvh_refit: blob of %zu bytes cannot hold %lld triangles", blob_bytes, (long long)n_faces);
    RefitWorkspace w = carve_refit(workspace, node_cap);
    RT_REQUIRE(workspace_bytes >= w.total, RT_ERR_SIZE, "rt_bvh_refit: workspace %zu < %zu", workspace_bytes, w.total);
    if (n_faces == 0) return RT_OK;
    RT_REQUIRE(vertices && faces && n_verts > 0, RT_ERR_INVALID, "rt_bvh_refit: null vertices/faces");
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "rt_bvh_refit: no CUDA device");
    uint8_t* blob8 = reinterpret_cast<uint8_t*>(blob);
    RT_CUDA_TRY(cudaMemsetAsync(w.counters, 0, align_up_sz((size_t)node_cap * 4u, 256), stream));
    k_refit_tris<<<grid_for(n_faces, 256, dev.sm_count, 8), 256, 0, stream>>>(vertices, n_verts, faces, n_faces,
                                                                              blob8 + RT_BLOB_HEADER_BYTES);
    k_refit_nodes<<<grid_for(node_cap, 128, dev.sm_count, 8), 128, 0, stream>>>(reinterpret_cast<rt_blob_header*>(blob8),
                                                                                    w.node_box, w.counters);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

namespace rt {
// The onesweep sort on the low 8 * passes key bits for other units (the caller guarantees the rest is zero); the
// sorted pairs are at *keys_out / *vals_out (the workspace's alternate buffers after an odd number of passes).
int sort_pairs_low(uint64_t* keys, uint32_t* vals, int64_t n, void* workspace, int passes, uint64_t** keys_out,
                   uint32_t** vals_out, cudaStream_t stream) {
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "sort: no CUDA device");
    RT_CUDA_TRY(sort::sort_pairs(keys, vals, n, workspace, dev.sm_count, stream, passes, keys_out, vals_out));
    return RT_OK;
}
}  // namespace rt

extern "C" int rt_sort_sizes(int64_t n, size_t* workspace_bytes) {
    RT_REQUIRE(n >= 0 && n <= (int64_t)1 << 30 && workspace_bytes, RT_ERR_INVALID, "rt_sort_sizes: bad arguments");
    *workspace_bytes = sort::workspace_bytes(n);
    return RT_OK;
}

extern "C" int rt_sort_pairs_u64(uint64_t* keys, uint32_t* vals, int64_t n, void* workspace, size_t workspace_bytes,
                                 void* stream_) {
    RT_REQUIRE(n >= 0 && n <= (int64_t)1 << 30, RT_ERR_INVALID, "rt_sort_pairs_u64: bad n");
    if (n <= 1) return RT_OK;
    RT_REQUIRE(keys && vals && workspace, RT_ERR_INVALID, "rt_sort_pairs_u64: null pointer");
    RT_REQUIRE(workspace_bytes >= sort::workspace_bytes(n), RT_ERR_SIZE, "rt_sort_pairs_u64: workspace too small");
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "rt_sort_pairs_u64: no CUDA device");
    RT_CUDA_TRY(sort::sort_pairs(keys, vals, n, workspace, dev.sm_count, reinterpret_cast<cudaStream_t>(stream_)));
    return RT_OK;
}
