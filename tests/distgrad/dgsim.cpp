// dgsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the distance gradient of rt_distgrad.cu on the CPU with its own RT_HD
// functions (rt_distgrad.cuh), window by window, with the host reduction of dgreduce.h.  Never linked into
// libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC dgsim.cpp -o libdgsim.so
#include <algorithm>
#include <vector>
#include "dgreduce.h"

using namespace rt;

// Dense [n,3] points; windows of `window` points (<= 0: one window).  grad_points / grad_vertices may be null.
extern "C" int dg_grad(int64_t n, const float* pts, const float* g, const float* value, const float* closest,
                       const int32_t* tri, const float* uv, const int32_t* faces, int64_t n_faces, int64_t n_verts,
                       int64_t window, float* grad_points, float* grad_vertices) {
    if (window <= 0 || window > n) window = n > 0 ? n : 1;
    if (grad_vertices) std::fill(grad_vertices, grad_vertices + 3 * n_verts, 0.0f);
    for (int64_t base = 0; base < n; base += window) {
        const int64_t nw = std::min(window, n - base);
        const int64_t m = 3 * nw;
        std::vector<float> q(3 * nw);
        std::vector<uint64_t> key(m);
        for (int64_t i = 0; i < nw; ++i) {
            const int64_t w = base + i;
            const bool live = dg_point_q(pts[3 * w], pts[3 * w + 1], pts[3 * w + 2], g[w], value[w], closest[3 * w],
                                         closest[3 * w + 1], closest[3 * w + 2], tri[w], n_faces, &q[3 * i]);
            if (grad_points) for (int c = 0; c < 3; ++c) grad_points[3 * w + c] = q[3 * i + c];
            for (uint32_t k = 0; k < 3; ++k) key[3 * i + k] = dg_key(live, faces, tri[w], k, n_verts);
        }
        if (grad_vertices)
            dg_reduce_host(key, n_verts, [&](uint32_t e, float out[3]) { dg_contrib(q.data(), uv + 2 * base, e, out); },
                           grad_vertices);
    }
    return 0;
}
