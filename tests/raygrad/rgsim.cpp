// rgsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the hit gradient of rt_ray_grad (rt_distgrad.cu) on the CPU with its own
// RT_HD functions (rt_raygrad.cuh, rt_distgrad.cuh), row window by row window, with the host reduction of
// tests/distgrad/dgreduce.h.  Never linked into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC rgsim.cpp -o librgsim.so
#include <algorithm>
#include <vector>
#include "../../trimesh-ray-optix_b200/csrc/rt_raygrad.cuh"
#include "../distgrad/dgreduce.h"

using namespace rt;

// Dense [n_rays,3] origins and directions; n_rows rows (row_ray null: row i is ray i); windows of `window` rows (<= 0:
// one window).  grad_loc / grad_uv may be null (0); grad_origins, grad_directions, grad_vertices may be null.
static bool eval_row(int64_t n_rays, const float* o, const float* d, const int32_t* row_ray, const int32_t* tri,
                     const float* grad_loc, const float* grad_uv, const RgMesh& mesh, int64_t j, RgRow& r) {
    const int64_t ray = row_ray ? (int64_t)row_ray[j] : j;
    const float zero[3] = {0.0f, 0.0f, 0.0f};
    if (ray < 0 || ray >= n_rays) return rg_row(zero, zero, zero, 0.0f, 0.0f, -1, mesh, r);
    return rg_row(o + 3 * ray, d + 3 * ray, grad_loc ? grad_loc + 3 * j : zero, grad_uv ? grad_uv[2 * j] : 0.0f,
                  grad_uv ? grad_uv[2 * j + 1] : 0.0f, tri[j], mesh, r);
}

// Per row: lambda, t lambda, q, w [n_rows, 3 / 3 / 3 / 2] and whether the row is live.
extern "C" int rg_row_values(int64_t n_rays, const float* o, const float* d, int64_t n_rows, const int32_t* row_ray,
                             const int32_t* tri, const float* grad_loc, const float* grad_uv, const float* vertices,
                             int64_t n_verts, const int32_t* faces, int64_t n_faces, float* lam, float* tlam, float* q,
                             float* w, uint8_t* live) {
    const RgMesh mesh{vertices, n_verts, faces, n_faces};
    for (int64_t j = 0; j < n_rows; ++j) {
        RgRow r;
        live[j] = eval_row(n_rays, o, d, row_ray, tri, grad_loc, grad_uv, mesh, j, r) ? 1 : 0;
        for (int c = 0; c < 3; ++c) { lam[3 * j + c] = r.lam[c]; tlam[3 * j + c] = r.tlam[c]; q[3 * j + c] = r.q[c]; }
        w[2 * j] = r.w[0]; w[2 * j + 1] = r.w[1];
    }
    return 0;
}

extern "C" int rg_grad(int64_t n_rays, const float* o, const float* d, int64_t n_rows, const int32_t* row_ray,
                       const int32_t* tri, const float* grad_loc, const float* grad_uv, const float* vertices,
                       int64_t n_verts, const int32_t* faces, int64_t n_faces, int64_t window, float* grad_origins,
                       float* grad_directions, float* grad_vertices) {
    const RgMesh mesh{vertices, n_verts, faces, n_faces};
    auto ray_of = [&](int64_t j) -> int64_t {
        const int64_t ray = row_ray ? (int64_t)row_ray[j] : j;
        return ray >= 0 && ray < n_rays ? ray : -1;
    };
    auto eval = [&](int64_t j, RgRow& r) { return eval_row(n_rays, o, d, row_ray, tri, grad_loc, grad_uv, mesh, j, r); };
    if (grad_origins) std::fill(grad_origins, grad_origins + 3 * n_rays, 0.0f);
    if (grad_directions) std::fill(grad_directions, grad_directions + 3 * n_rays, 0.0f);
    if (grad_vertices) std::fill(grad_vertices, grad_vertices + 3 * n_verts, 0.0f);
    for (int64_t j = 0; j < n_rows; ++j) {
        if (!rg_head(j, row_ray) || ray_of(j) < 0) continue;
        float go[3], gd[3];
        rg_ray_sums(j, n_rows, row_ray, [&](int64_t k, RgRow& r) { eval(k, r); }, go, gd);
        const int64_t ray = ray_of(j);
        for (int c = 0; c < 3; ++c) {
            if (grad_origins) grad_origins[3 * ray + c] = go[c];
            if (grad_directions) grad_directions[3 * ray + c] = gd[c];
        }
    }
    if (!grad_vertices) return 0;
    if (window <= 0 || window > n_rows) window = n_rows > 0 ? n_rows : 1;
    for (int64_t base = 0; base < n_rows; base += window) {
        const int64_t nw = std::min(window, n_rows - base);
        const int64_t m = 3 * nw;
        std::vector<float> q(3 * nw), w(2 * nw);
        std::vector<uint64_t> key(m);
        for (int64_t i = 0; i < nw; ++i) {
            RgRow r;
            const bool live = eval(base + i, r);
            for (int c = 0; c < 3; ++c) q[3 * i + c] = r.q[c];
            w[2 * i] = r.w[0]; w[2 * i + 1] = r.w[1];
            for (uint32_t k = 0; k < 3; ++k) key[3 * i + k] = dg_key(live, faces, tri[base + i], k, n_verts);
        }
        dg_reduce_host(key, n_verts, [&](uint32_t e, float out[3]) { dg_contrib(q.data(), w.data(), e, out); },
                       grad_vertices);
    }
    return 0;
}
