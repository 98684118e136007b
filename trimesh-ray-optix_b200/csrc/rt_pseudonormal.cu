// rt_pseudonormal.cu — the pseudo-normal side array of a BVH8 blob (rt_pseudonormals): per triangle record the
// angle-weighted vertex normals and the edge normals the signed-distance kernel (rt_closest.cu) reads, plus the counts
// of boundary, non-manifold and inconsistently oriented edges.
//
// From the blob alone (header and triangle records), in three stable sorts with the builder's onesweep radix sort:
//   1. corners (3 per record) by z bits, then by (x bits << 32 | y bits): runs of equal coordinates are welded
//      vertices; one thread per run head sums the run in order (weld_run) and writes every member's normal and id;
//   2. half-edges by (min id << 32 | max id): one thread per run head sums the unit face normals, writes every
//      member's normal and classifies the edge (edge_run).
// A run is walked serially, so a vertex of valence k costs O(k) on one thread.  Buffers are sized by their capacity in
// triangles; a blob with more triangles than they hold gets nothing written (and zero counts).
#include "rt_api.h"
#include "rt_pseudonormal.cuh"

namespace rt {

__global__ void __launch_bounds__(256) k_pn_corner_keys(const uint8_t* blob, uint32_t cap, uint64_t* keys, uint32_t* vals,
                                                        int xy) {
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(blob);
    const uint8_t* tris = blob + hdr->tris_offset;
    const uint32_t n = hdr->n_tris;
    if (n > cap) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 3u * cap; j += stride) {
        // pass 1 keys corner j; pass 2 keys the corner the first sort put at position j
        const uint32_t c = xy ? vals[j] : j;
        uint64_t key = kPnNoKey;
        if (c < 3u * n) {
            float v[9];
            load_tri(tris, c / 3u, v);
            if (tri_finite(v)) key = xy ? corner_key_xy(v, c % 3u) : corner_key_z(v, c % 3u);
        }
        keys[j] = key;
        if (!xy) vals[j] = c;
    }
}

__global__ void __launch_bounds__(256) k_pn_weld(const uint8_t* blob, uint32_t cap, const uint32_t* sorted, uint32_t* vid,
                                                 uint8_t* normals) {
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(blob);
    const uint32_t n = hdr->n_tris;
    if (n > cap) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 3u * n; j += stride)
        weld_run(blob + hdr->tris_offset, sorted, 3u * n, j, vid, normals);
}

__global__ void __launch_bounds__(256) k_pn_edge_keys(const uint8_t* blob, uint32_t cap, const uint32_t* vid, uint64_t* keys,
                                                      uint32_t* vals) {
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(blob);
    const uint32_t n = hdr->n_tris;
    if (n > cap) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t h = blockIdx.x * blockDim.x + threadIdx.x; h < 3u * cap; h += stride) {
        keys[h] = h < 3u * n ? half_edge_key(vid, h) : kPnNoKey;
        vals[h] = h;
    }
}

__global__ void __launch_bounds__(256) k_pn_edges(const uint8_t* blob, uint32_t cap, const uint32_t* sorted,
                                                  const uint64_t* keys, const uint32_t* vid, uint8_t* normals,
                                                  unsigned long long* counts) {
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(blob);
    const uint32_t n = hdr->n_tris;
    if (n > cap) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 3u * n; j += stride) {
        if (keys[j] == kPnNoKey) {   // a half-edge of a non-finite triangle
            store_row_slot(normals, sorted[j] / 3u, half_edge_slot(sorted[j] % 3u), 0.0f, 0.0f, 0.0f);
            continue;
        }
        if (!edge_head(keys, j)) continue;
        const uint32_t cls = edge_class(edge_run(blob + hdr->tris_offset, sorted, keys, 3u * n, j, vid, normals));
        if (cls < 3u) atomicAdd(&counts[cls], 1ull);
    }
}

struct PnWorkspace {
    uint64_t* keys;    // [3 cap]
    uint32_t* vals;    // [3 cap]
    uint32_t* vid;     // [3 cap] vertex id of every corner
    void* sort_ws;     // rt_sort_sizes(3 cap)
    size_t sort_bytes, total;
};
static PnWorkspace carve_pn(void* base, uint32_t cap) {
    PnWorkspace w;
    const size_t m = (size_t)3u * cap;
    const size_t kb = align_up_sz(m * 8u, 256), vb = align_up_sz(m * 4u, 256);
    size_t sb = 0;
    rt_sort_sizes((int64_t)m, &sb);
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    w.keys = reinterpret_cast<uint64_t*>(p);
    w.vals = reinterpret_cast<uint32_t*>(p ? p + kb : nullptr);
    w.vid = reinterpret_cast<uint32_t*>(p ? p + kb + vb : nullptr);
    w.sort_ws = p ? p + kb + 2 * vb : nullptr;
    w.sort_bytes = align_up_sz(sb, 256);
    w.total = kb + 2 * vb + w.sort_bytes;
    return w;
}

constexpr int64_t kPnMaxFaces = ((int64_t)1 << 30) / 3;   // 3 n corners must fit one rt_sort_pairs_u64 call

}  // namespace rt

using namespace rt;

extern "C" int rt_pseudonormals_sizes(int64_t n_faces, size_t* normals_bytes, size_t* workspace_bytes) {
    RT_REQUIRE(n_faces >= 0 && n_faces <= kPnMaxFaces && normals_bytes && workspace_bytes, RT_ERR_INVALID,
               "rt_pseudonormals_sizes: bad arguments (at most %lld triangles)", (long long)kPnMaxFaces);
    *normals_bytes = align_up_sz((size_t)n_faces * kPnRowBytes, 256);
    *workspace_bytes = carve_pn(nullptr, (uint32_t)n_faces).total;
    return RT_OK;
}

extern "C" int rt_pseudonormals(const void* blob, void* normals, size_t normals_bytes, void* workspace,
                                size_t workspace_bytes, uint64_t* edge_counts_dev, void* stream_) {
    const char* fn = "rt_pseudonormals";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    RT_REQUIRE(blob != nullptr && ((uintptr_t)blob & 15) == 0, RT_ERR_INVALID, "%s: blob null or not 16-byte aligned", fn);
    RT_REQUIRE(edge_counts_dev != nullptr, RT_ERR_INVALID, "%s: null edge counts", fn);
    RT_CUDA_TRY(cudaMemsetAsync(edge_counts_dev, 0, 3 * sizeof(uint64_t), stream));
    // The triangle count lives in the blob's header on the device: the capacity of the buffers is passed to the
    // kernels, which write nothing when the blob holds more triangles.
    const int64_t cap64 = (int64_t)(normals_bytes / kPnRowBytes);
    RT_REQUIRE(cap64 <= kPnMaxFaces, RT_ERR_INVALID, "%s: normals for %lld triangles: at most %lld", fn, (long long)cap64,
               (long long)kPnMaxFaces);
    const uint32_t cap = (uint32_t)cap64;
    if (cap == 0) return RT_OK;
    RT_REQUIRE(normals != nullptr && ((uintptr_t)normals & 15) == 0, RT_ERR_INVALID,
               "%s: normals null or not 16-byte aligned", fn);
    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    PnWorkspace w = carve_pn(workspace, cap);
    RT_REQUIRE(workspace_bytes >= w.total, RT_ERR_SIZE, "%s: workspace %zu < %zu", fn, workspace_bytes, w.total);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    const uint8_t* b = reinterpret_cast<const uint8_t*>(blob);
    uint8_t* nrm = reinterpret_cast<uint8_t*>(normals);
    unsigned long long* counts = reinterpret_cast<unsigned long long*>(edge_counts_dev);
    const int64_t m = 3 * (int64_t)cap;
    const int grid = grid_for(m, 256, dev.sm_count, 8);
    k_pn_corner_keys<<<grid, 256, 0, stream>>>(b, cap, w.keys, w.vals, 0);
    RT_CUDA_TRY(cudaGetLastError());
    int rc = rt_sort_pairs_u64(w.keys, w.vals, m, w.sort_ws, w.sort_bytes, stream);
    if (rc != RT_OK) return rc;
    k_pn_corner_keys<<<grid, 256, 0, stream>>>(b, cap, w.keys, w.vals, 1);
    RT_CUDA_TRY(cudaGetLastError());
    rc = rt_sort_pairs_u64(w.keys, w.vals, m, w.sort_ws, w.sort_bytes, stream);
    if (rc != RT_OK) return rc;
    k_pn_weld<<<grid, 256, 0, stream>>>(b, cap, w.vals, w.vid, nrm);
    k_pn_edge_keys<<<grid, 256, 0, stream>>>(b, cap, w.vid, w.keys, w.vals);
    RT_CUDA_TRY(cudaGetLastError());
    rc = rt_sort_pairs_u64(w.keys, w.vals, m, w.sort_ws, w.sort_bytes, stream);
    if (rc != RT_OK) return rc;
    k_pn_edges<<<grid, 256, 0, stream>>>(b, cap, w.vals, w.keys, w.vid, nrm, counts);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
