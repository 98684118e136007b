// dgsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the distance gradient of rt_distgrad.cu on the CPU with its own RT_HD
// functions (rt_distgrad.cuh), window by window, with std::stable_sort in place of the onesweep sort: a stable sort
// of the same keys yields the same permutation.  Never linked into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC dgsim.cpp -o libdgsim.so
#include <algorithm>
#include <numeric>
#include <vector>
#include "../../trimesh-ray-optix_b200/csrc/rt_distgrad.cuh"

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
        if (!grad_vertices) continue;
        std::vector<uint32_t> vals(m);
        std::iota(vals.begin(), vals.end(), 0u);
        std::stable_sort(vals.begin(), vals.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
        std::vector<uint64_t> keys(m);
        for (int64_t j = 0; j < m; ++j) keys[j] = key[vals[j]];
        std::vector<uint32_t> start(n_verts);
        for (int64_t j = 0; j < m; ++j) dg_run_start(j, keys.data(), n_verts, start.data());
        const uint64_t slots = dg_next_size(m);
        std::vector<uint32_t> lk[2], li[2];
        std::vector<float> lv[2];
        for (int b = 0; b < 2; ++b) { lk[b].assign(slots, kDgEmpty); li[b].assign(slots, 0); lv[b].assign(3 * slots, 0.0f); }
        DgLevel lev[2] = {{lk[0].data(), li[0].data(), lv[0].data()}, {lk[1].data(), li[1].data(), lv[1].data()}};
        for (int64_t j = 0; j < m; ++j)
            dg_level0_at(j, m, keys.data(), vals.data(), start.data(), n_verts, q.data(), uv + 2 * base, grad_vertices,
                         lev[0]);
        uint64_t size = m, len = m;
        int cur = 0;
        while (len > kDgGroup) {
            size = dg_next_size(size);
            len = (len + kDgGroup - 1) / kDgGroup;
            std::fill(lk[cur ^ 1].begin(), lk[cur ^ 1].end(), kDgEmpty);
            for (uint64_t j = 0; j < size; ++j) dg_level_at(j, size, lev[cur], grad_vertices, lev[cur ^ 1]);
            cur ^= 1;
        }
    }
    return 0;
}
