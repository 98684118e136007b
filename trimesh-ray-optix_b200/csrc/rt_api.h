// rt_api.h — shared plumbing of the C ABI translation units: error reporting, blob header
// access, launch geometry.  Nothing here is exported.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include "../../include/raymesh_b200.h"
#include "rt_core.cuh"

namespace rt {

// thread-local message returned by rt_last_error()
char* error_buffer();
int set_error(int code, const char* fmt, ...);

#define RT_CUDA_TRY(expr)                                                                         \
    do {                                                                                          \
        cudaError_t e__ = (expr);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return ::rt::set_error(RT_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                                   __FILE__, __LINE__);                                           \
    } while (0)

#define RT_REQUIRE(cond, code, ...)                                \
    do {                                                           \
        if (!(cond)) return ::rt::set_error((code), __VA_ARGS__);  \
    } while (0)

struct DeviceInfo { int device; int sm_count; };
// cached per device; sm_count == 0 when there is no usable device
int device_info(DeviceInfo* out);

// rt_build.cu: the builder's onesweep sort on the low 8 * passes key bits (sorted pairs at *keys_out / *vals_out)
int sort_pairs_low(uint64_t* keys, uint32_t* vals, int64_t n, void* workspace, int passes, uint64_t** keys_out,
                   uint32_t** vals_out, cudaStream_t stream);

inline size_t align_up_sz(size_t x, size_t a) { return (x + a - 1) / a * a; }

// blocks for a grid-stride loop over n items: enough to cover them, at most per_sm blocks per SM
inline int grid_for(int64_t n, int threads, int sm_count, int per_sm) {
    int64_t b = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count * per_sm;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

// a batch (rt_ray_desc origins or directions) that is row-major contiguous [s0, s1, s2, 3]: row r starts at element
// 3 r (batch_offset); dimensions of extent 1 may carry any stride
inline bool batch_packed(const int64_t shape[4], const int64_t stride[4]) {
    if (stride[3] != 1) return false;
    int64_t expect = 3;
    for (int i = 2; i >= 0; --i) {
        if (shape[i] != 1 && stride[i] != expect) return false;
        expect *= shape[i];
    }
    return true;
}

// Checks the descriptor of a [*b, 3] batch and resolves the window [*first, *first + *n) that opts selects: all of
// the batch when opts is NULL, to its end when ray_count <= 0.  The data pointers are left to the caller: which ones a
// query reads, and whether it reads them for an empty window, differ between entry points.
inline int batch_window(const char* fn, const rt_ray_desc* d, const rt_trace_opts* opts, int64_t* first, int64_t* n) {
    RT_REQUIRE(d != nullptr, RT_ERR_INVALID, "%s: null batch descriptor", fn);
    RT_REQUIRE(d->nray >= 0 && d->shape[3] == 3, RT_ERR_INVALID, "%s: batch must be [*b, 3] (nray %lld, last dimension %lld)",
               fn, (long long)d->nray, (long long)d->shape[3]);
    RT_REQUIRE(d->shape[0] >= 0 && d->shape[1] >= 0 && d->shape[2] >= 0 && d->shape[0] * d->shape[1] * d->shape[2] == d->nray,
               RT_ERR_INVALID, "%s: nray %lld does not match shape", fn, (long long)d->nray);
    const int64_t f = opts ? opts->ray_first : 0, c = opts ? opts->ray_count : 0;
    RT_REQUIRE(f >= 0 && f <= d->nray, RT_ERR_INVALID, "%s: ray_first %lld outside [0, %lld]", fn, (long long)f,
               (long long)d->nray);
    const int64_t m = c <= 0 ? d->nray - f : c;
    RT_REQUIRE(m <= d->nray - f, RT_ERR_INVALID, "%s: window [%lld, +%lld) exceeds the batch of %lld", fn, (long long)f,
               (long long)m, (long long)d->nray);
    *first = f;
    *n = m;
    return RT_OK;
}

// Triangles per leaf slot used by the builder: kLeafTrisDefault, or TRIRO_LEAF_TRIS=1..3 (read once per process;
// sizes, build and refit of one process always agree).
inline int leaf_tris_setting() {
    static const int v = [] {
        const char* e = getenv("TRIRO_LEAF_TRIS");
        const int x = e ? atoi(e) : kLeafTrisDefault;
        return x < 1 ? 1 : (x > kLeafMaxTris ? kLeafMaxTris : x);
    }();
    return v;
}

// Blob geometry derived from the triangle count alone (host side, no device read needed).
struct BlobLayout {
    size_t tris_offset, nodes_offset, parents_offset, total_bytes;
    uint32_t node_cap;
};
inline BlobLayout blob_layout(int64_t n_faces) {
    BlobLayout l;
    l.tris_offset = RT_BLOB_HEADER_BYTES;
    l.nodes_offset = align_up_sz(l.tris_offset + (size_t)(n_faces > 0 ? n_faces : 0) * 48u, 256);
    l.node_cap = wide_node_cap(n_faces, leaf_tris_setting());
    l.parents_offset = align_up_sz(l.nodes_offset + (size_t)l.node_cap * 80u, 256);
    l.total_bytes = l.parents_offset + align_up_sz((size_t)l.node_cap * 4u, 256);
    return l;
}

}  // namespace rt
