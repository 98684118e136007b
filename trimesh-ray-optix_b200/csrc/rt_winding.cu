// rt_winding.cu — generalized winding numbers for a batch of query points (rt_winding_number) and the per-node
// moments they use (rt_winding_moments), on the BVH8 blob the ray queries use.
//
// Moments: a side array of one 64-byte WindMoment per node, computed bottom-up from the blob alone (its header, triangle
// records, nodes and parent links), with the climbing pattern of k_refit_nodes: one thread per node without inner
// children starts, the last child to report computes its parent.  node_moment() reads a node's triangle records in
// record order and its children in slot order, so the records do not depend on which thread climbs.
//
// Winding numbers: one thread per point, wind_step (rt_winding.cuh) from the root; leaf triangles exactly, far inner
// children by their expansion, near ones visited in slot order.  The host simulator under tests/winding/ gives the
// same bits.
#include <type_traits>
#include "rt_api.h"
#include "rt_winding.cuh"

namespace rt {

constexpr int kWindThreads = 128;

// one thread per node without inner children starts; the last child to report climbs to the parent
__global__ void __launch_bounds__(128) k_winding_moments(const uint8_t* blob, uint8_t* moments, float* weights,
                                                         uint32_t* counters, uint32_t cap) {
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(blob);
    const uint8_t* nodes = blob + hdr->nodes_offset;
    const uint8_t* tris = blob + hdr->tris_offset;
    const uint32_t* parent = reinterpret_cast<const uint32_t*>(blob + hdr->parents_offset);
    const uint32_t n_nodes = hdr->n_nodes;
    if (n_nodes > cap) return;   // buffers sized for fewer triangles than the blob holds: write nothing out of bounds
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t w0 = blockIdx.x * blockDim.x + threadIdx.x; w0 < n_nodes; w0 += stride) {
        if (nodes[(size_t)w0 * 80u + 15] != 0) continue;   // imask != 0: an inner child will take care of it
        uint32_t w = w0;
        for (;;) {
            const WindNodeOut o = node_moment(nodes, tris, w, moments, weights);
            store_moment(moments, w, o.mo, weights, o.weight);
            if (w == 0u) break;
            const uint32_t pw = parent[w] >> 3;
            const uint32_t need = (uint32_t)__popc((uint32_t)nodes[(size_t)pw * 80u + 15]);
            __threadfence();
            if (atomicAdd(&counters[pw], 1u) + 1u != need) break;
            __threadfence();
            w = pw;
        }
    }
}

struct WindParams {
    const uint8_t* blob;
    const uint8_t* moments;
    const float* origins;
    int64_t shape[4], stride[4];
    int packed;                  // row-major contiguous [.., 3]: offset 3 * r
    int64_t first, n;            // window [first, first + n) of the batch; outputs indexed by (r - first)
    float beta;
    float* winding;
    unsigned long long* counters;
};

template <bool STATS>
__global__ void __launch_bounds__(kWindThreads) k_winding_number(const __grid_constant__ WindParams p) {
    using S = typename std::conditional<STATS, WindStats, WindNoStats>::type;
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(p.blob);
    const uint8_t* tris = p.blob + hdr->tris_offset;
    const uint8_t* nodes = p.blob + hdr->nodes_offset;
    const int64_t i = (int64_t)blockIdx.x * kWindThreads + threadIdx.x;
    S st;
    if (i < p.n) {
        const int64_t o = batch_offset(p.shape, p.stride, p.packed, p.first + i);
        const int64_t os = p.stride[3];
        WindTrav t;
        wind_init(t, p.origins[o], p.origins[o + os], p.origins[o + 2 * os]);
        ArrayStack<WindStackEntry> stack;
        while (!wind_step(nodes, tris, p.moments, p.beta, t, st, stack)) {}
        p.winding[i] = wind_result(t);
    }
    if (STATS) {
        unsigned long long c0 = st.n_nodes(), c1 = st.n_tris(), c2 = i < p.n ? 1ull : 0ull, c3 = st.n_fars();
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

struct WindWorkspace {
    uint32_t* counters;    // [cap] children that have reported
    float* weights;        // [cap] total area of each node's subtree
    size_t total;
};
static WindWorkspace carve_wind(void* base, uint32_t cap) {
    WindWorkspace w;
    uint8_t* p = reinterpret_cast<uint8_t*>(base);
    const size_t cb = align_up_sz((size_t)cap * 4u, 256);
    w.counters = reinterpret_cast<uint32_t*>(p);
    w.weights = reinterpret_cast<float*>(p ? p + cb : nullptr);
    w.total = 2 * cb;
    return w;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_winding_moments_sizes(int64_t n_faces, size_t* moments_bytes, size_t* workspace_bytes) {
    RT_REQUIRE(n_faces >= 0 && n_faces <= (int64_t)1 << 30 && moments_bytes && workspace_bytes, RT_ERR_INVALID,
               "rt_winding_moments_sizes: bad arguments");
    // bound for any leaf size the blob may have been built with (the node count itself is only known on the device)
    const uint32_t cap = wide_node_cap(n_faces, 1);
    *moments_bytes = align_up_sz((size_t)cap * 64u, 256);
    *workspace_bytes = carve_wind(nullptr, cap).total;
    return RT_OK;
}

extern "C" int rt_winding_moments(const void* blob, void* moments, size_t moments_bytes, void* workspace,
                                  size_t workspace_bytes, void* stream_) {
    const char* fn = "rt_winding_moments";
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    RT_REQUIRE(blob != nullptr && ((uintptr_t)blob & 15) == 0, RT_ERR_INVALID, "%s: blob null or not 16-byte aligned", fn);
    RT_REQUIRE(moments != nullptr && ((uintptr_t)moments & 15) == 0, RT_ERR_INVALID,
               "%s: moments null or not 16-byte aligned", fn);
    RT_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 255) == 0, RT_ERR_INVALID,
               "%s: workspace null or not 256-byte aligned", fn);
    // The node count lives in the blob's header on the device: the host can only bound it.  The buffers' capacity is
    // passed to the kernel, which writes nothing when the blob has more nodes than they hold.
    const size_t cap_m = moments_bytes / 64u, cap_w = workspace_bytes / 512u * 64u;   // carve_wind(cap_w) fits
    size_t cap_sz = cap_m < cap_w ? cap_m : cap_w;
    if (cap_sz > 0xffffffffu) cap_sz = 0xffffffffu;
    const uint32_t cap = (uint32_t)cap_sz;
    RT_REQUIRE(cap >= 1, RT_ERR_SIZE, "%s: moments (%zu bytes) or workspace (%zu bytes) too small for one node", fn,
               moments_bytes, workspace_bytes);
    WindWorkspace w = carve_wind(workspace, cap);
    RT_REQUIRE(workspace_bytes >= w.total, RT_ERR_SIZE, "%s: workspace %zu < %zu", fn, workspace_bytes, w.total);
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    RT_CUDA_TRY(cudaMemsetAsync(w.counters, 0, (size_t)cap * 4u, stream));
    k_winding_moments<<<grid_for(cap, 128, dev.sm_count, 8), 128, 0, stream>>>(
        reinterpret_cast<const uint8_t*>(blob), reinterpret_cast<uint8_t*>(moments), w.weights, w.counters, cap);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

extern "C" int rt_winding_number(const void* blob, const void* moments, const rt_ray_desc* points, const rt_trace_opts* opts,
                                 float beta, float* winding, uint64_t* counters_dev, void* scratch, void* stream) {
    (void)scratch;   // one thread per point: no work counter, the scratch is left as it was
    const char* fn = "rt_winding_number";
    RT_REQUIRE(blob != nullptr && ((uintptr_t)blob & 15) == 0, RT_ERR_INVALID, "%s: blob null or not 16-byte aligned", fn);
    RT_REQUIRE(moments != nullptr && ((uintptr_t)moments & 15) == 0, RT_ERR_INVALID,
               "%s: moments null or not 16-byte aligned", fn);
    RT_REQUIRE(beta >= 1.0f, RT_ERR_INVALID, "%s: beta must be >= 1 or +inf (got %g)", fn, (double)beta);
    int64_t first = 0, count = 0;
    const int rc = batch_window(fn, points, opts, &first, &count);
    if (rc != RT_OK) return rc;
    if (counters_dev) RT_CUDA_TRY(cudaMemsetAsync(counters_dev, 0, 4 * sizeof(uint64_t), (cudaStream_t)stream));
    if (count == 0) return RT_OK;
    RT_REQUIRE(points->origins != nullptr, RT_ERR_INVALID, "%s: null points", fn);
    RT_REQUIRE(winding != nullptr, RT_ERR_INVALID, "%s: null output", fn);
    WindParams p = {};
    p.blob = reinterpret_cast<const uint8_t*>(blob);
    p.moments = reinterpret_cast<const uint8_t*>(moments);
    p.origins = points->origins;
    for (int a = 0; a < 4; ++a) { p.shape[a] = points->shape[a]; p.stride[a] = points->o_stride[a]; }
    p.packed = batch_packed(points->shape, points->o_stride) ? 1 : 0;
    p.first = first;
    p.n = count;
    p.beta = beta;
    p.winding = winding;
    p.counters = reinterpret_cast<unsigned long long*>(counters_dev);
    const int64_t grid = (count + kWindThreads - 1) / kWindThreads;
    RT_REQUIRE(grid < ((int64_t)1 << 31), RT_ERR_INVALID, "%s: batch of %lld points too large for one launch", fn,
               (long long)count);
    if (counters_dev)
        k_winding_number<true><<<(unsigned)grid, kWindThreads, 0, (cudaStream_t)stream>>>(p);
    else
        k_winding_number<false><<<(unsigned)grid, kWindThreads, 0, (cudaStream_t)stream>>>(p);
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
