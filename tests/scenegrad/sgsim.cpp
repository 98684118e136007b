// sgsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the instanced-scene gradients of rt_scene_grad.cu on the CPU with their
// own RT_HD functions (rt_scenegrad.cuh, rt_raygrad.cuh, rt_distgrad.cuh), row window by row window, with
// std::stable_sort in place of the onesweep sort: a stable sort of the same keys yields the same permutation.  The scene
// table comes from tests/scene (ss_prepare) and the member table holds host addresses.  Never linked into
// libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC sgsim.cpp -o libsgsim.so
#include <algorithm>
#include <functional>
#include <numeric>
#include <vector>
#include "../../trimesh-ray-optix_b200/csrc/rt_scenegrad.cuh"

using namespace rt;

namespace {
// one row of a window: writes its factors and keys; returns nothing (dead rows write +0 and sentinel keys)
using RowFn = std::function<void(int64_t row, SgRow& r, bool& live, uint64_t key[3], int32_t& inst)>;

// steps 1 (pairs), 2 and 3 of every window, then the outputs, as sg_run does
void reduce(int64_t n_rows, int64_t n_inst, int64_t n_verts, int outputs, int64_t window, const RowFn& row,
            float* grad_transforms, float* grad_vertices) {
    const bool want_t = (outputs & 1) != 0, want_v = (outputs & 2) != 0;
    if (!want_t && !want_v) return;
    const int slot0 = want_v ? 0 : 3, n_slots = (want_v ? 3 : 0) + (want_t ? 4 : 0);
    const uint64_t n_keys = (uint64_t)(n_verts + 4 * n_inst);
    std::vector<float> acc(3 * n_keys, 0.0f);
    if (window <= 0 || window > n_rows) window = n_rows > 0 ? n_rows : 1;
    for (int64_t base = 0; base < n_rows; base += window) {
        const int64_t nw = std::min(window, n_rows - base);
        const int64_t m = n_slots * nw;
        std::vector<float> rec(kSgRowFloats * nw);
        std::vector<uint64_t> key(m);
        for (int64_t i = 0; i < nw; ++i) {
            SgRow r;
            bool live;
            uint64_t vk[3];
            int32_t inst;
            row(base + i, r, live, vk, inst);
            sg_store(r, rec.data() + kSgRowFloats * i);
            for (int s = 0; s < n_slots; ++s) key[n_slots * i + s] = sg_key(live, vk, inst, slot0 + s, n_verts, n_keys);
        }
        std::vector<uint32_t> vals(m);
        std::iota(vals.begin(), vals.end(), 0u);
        std::stable_sort(vals.begin(), vals.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
        std::vector<uint64_t> keys(m);
        for (int64_t j = 0; j < m; ++j) keys[j] = key[vals[j]];
        std::vector<uint32_t> start(n_keys);
        for (int64_t j = 0; j < m; ++j) dg_run_start(j, keys.data(), n_keys, start.data());
        const uint64_t slots = dg_next_size(m);
        std::vector<uint32_t> lk[2], li[2];
        std::vector<float> lv[2];
        for (int b = 0; b < 2; ++b) { lk[b].assign(slots, kDgEmpty); li[b].assign(slots, 0); lv[b].assign(3 * slots, 0.0f); }
        DgLevel lev[2] = {{lk[0].data(), li[0].data(), lv[0].data()}, {lk[1].data(), li[1].data(), lv[1].data()}};
        for (int64_t j = 0; j < m; ++j)
            dg_level0_with(j, m, keys.data(), vals.data(), start.data(), n_keys,
                           [&](uint32_t e, float out[3]) { sg_contrib(rec.data(), slot0, n_slots, e, out); }, acc.data(),
                           lev[0]);
        uint64_t size = m, len = m;
        int cur = 0;
        while (len > kDgGroup) {
            size = dg_next_size(size);
            len = (len + kDgGroup - 1) / kDgGroup;
            std::fill(lk[cur ^ 1].begin(), lk[cur ^ 1].end(), kDgEmpty);
            for (uint64_t j = 0; j < size; ++j) dg_level_at(j, size, lev[cur], acc.data(), lev[cur ^ 1]);
            cur ^= 1;
        }
    }
    if (grad_vertices) std::copy(acc.begin(), acc.begin() + 3 * n_verts, grad_vertices);
    if (grad_transforms)
        for (int64_t e = 0; e < 12 * n_inst; ++e) sg_transform_out(acc.data(), n_verts, e, grad_transforms);
}

struct HitRows {
    SgScene sc;
    int64_t n_rays;
    const float *o, *d, *grad_loc, *grad_uv;
    const int32_t *row_ray, *inst, *tri;
    int64_t ray_of(int64_t j) const {
        const int64_t ray = row_ray ? (int64_t)row_ray[j] : j;
        return ray >= 0 && ray < n_rays ? ray : -1;
    }
    bool eval(int64_t j, RgRow& rr, SgRow& r, uint64_t key[3]) const {
        const float z[3] = {0.0f, 0.0f, 0.0f};
        const int64_t ray = ray_of(j);
        if (ray < 0) return sg_hit_row(sc, -1, -1, z, z, z, 0.0f, 0.0f, rr, r, key);
        return sg_hit_row(sc, inst[j], tri[j], o + 3 * ray, d + 3 * ray, grad_loc ? grad_loc + 3 * j : z,
                          grad_uv ? grad_uv[2 * j] : 0.0f, grad_uv ? grad_uv[2 * j + 1] : 0.0f, rr, r, key);
    }
};
}  // namespace

// Hit rows over dense [n_rays,3] origins / directions; window <= 0: one window.  Outputs may be null.
extern "C" int sg_ray_grad(const uint8_t* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                           int64_t n_verts, int64_t n_rays, const float* o, const float* d, int64_t n_rows,
                           const int32_t* row_ray, const int32_t* inst, const int32_t* tri, const float* grad_loc,
                           const float* grad_uv, int64_t window, int outputs, float* grad_origins,
                           float* grad_directions, float* grad_transforms, float* grad_vertices) {
    const HitRows h{sg_scene(table, n_inst, members, n_meshes, n_verts), n_rays, o, d, grad_loc, grad_uv, row_ray, inst, tri};
    if (grad_origins) std::fill(grad_origins, grad_origins + 3 * n_rays, 0.0f);
    if (grad_directions) std::fill(grad_directions, grad_directions + 3 * n_rays, 0.0f);
    for (int64_t j = 0; j < n_rows; ++j) {
        if (!rg_head(j, row_ray) || h.ray_of(j) < 0) continue;
        float go[3], gd[3];
        rg_ray_sums(j, n_rows, row_ray, [&](int64_t k, RgRow& rr) { SgRow r; uint64_t key[3]; h.eval(k, rr, r, key); },
                    go, gd);
        const int64_t ray = h.ray_of(j);
        for (int c = 0; c < 3; ++c) {
            if (grad_origins) grad_origins[3 * ray + c] = go[c];
            if (grad_directions) grad_directions[3 * ray + c] = gd[c];
        }
    }
    reduce(n_rows, n_inst, n_verts, outputs, window, [&](int64_t j, SgRow& r, bool& live, uint64_t key[3], int32_t& in) {
        RgRow rr;
        live = h.eval(j, rr, r, key);
        in = live ? inst[j] : -1;
    }, grad_transforms, grad_vertices);
    return 0;
}

// Point rows over dense [n,3] points and the forward's outputs.
extern "C" int sg_point_grad(const uint8_t* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                             int64_t n_verts, int64_t n, const float* p, const float* grad_out, const float* value,
                             const float* closest, const int32_t* inst, const int32_t* tri, const float* uv,
                             int64_t window, int outputs, float* grad_points, float* grad_transforms,
                             float* grad_vertices) {
    const SgScene sc = sg_scene(table, n_inst, members, n_meshes, n_verts);
    auto eval = [&](int64_t i, float q[3], SgRow& r, uint64_t key[3]) {
        return sg_point_row(sc, inst[i], tri[i], p[3 * i], p[3 * i + 1], p[3 * i + 2], grad_out[i], value[i],
                            closest[3 * i], closest[3 * i + 1], closest[3 * i + 2], uv[2 * i], uv[2 * i + 1], q, r, key);
    };
    for (int64_t i = 0; i < n && grad_points; ++i) {
        SgRow r;
        uint64_t key[3];
        eval(i, grad_points + 3 * i, r, key);
    }
    reduce(n, n_inst, n_verts, outputs, window, [&](int64_t i, SgRow& r, bool& live, uint64_t key[3], int32_t& in) {
        float q[3];
        live = eval(i, q, r, key);
        in = inst[i];
    }, grad_transforms, grad_vertices);
    return 0;
}

// Per hit row: lambda, t lambda, q, q_obj, x [3 each], w [2], live.
extern "C" int sg_hit_rows(const uint8_t* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                           int64_t n_verts, int64_t n_rays, const float* o, const float* d, int64_t n_rows,
                           const int32_t* row_ray, const int32_t* inst, const int32_t* tri, const float* grad_loc,
                           const float* grad_uv, float* lam, float* tlam, float* q, float* qo, float* x, float* w,
                           uint8_t* live) {
    const HitRows h{sg_scene(table, n_inst, members, n_meshes, n_verts), n_rays, o, d, grad_loc, grad_uv, row_ray, inst, tri};
    for (int64_t j = 0; j < n_rows; ++j) {
        RgRow rr;
        SgRow r;
        uint64_t key[3];
        live[j] = h.eval(j, rr, r, key) ? 1 : 0;
        for (int c = 0; c < 3; ++c) {
            lam[3 * j + c] = rr.lam[c]; tlam[3 * j + c] = rr.tlam[c]; q[3 * j + c] = r.q[c];
            qo[3 * j + c] = r.qo[c]; x[3 * j + c] = r.x[c];
        }
        w[2 * j] = r.w[0]; w[2 * j + 1] = r.w[1];
    }
    return 0;
}
