// rt_distgrad.cuh — the arithmetic of the distance gradient (rt_distgrad.cu, DESIGN.md §4.9): the per-point factor q,
// the vertex contributions and one step of the deterministic per-vertex reduction.  Everything here is RT_HD, like
// rt_point.cuh, so that tests/distgrad/ runs exactly the code the kernels run.
//
// For a point p with forward outputs (value, c, t, w0, w1) and incoming gradient g:
//   q = g * s * (p - c) / |value|, s = -1 when value's sign bit is set else +1   (= grad_points)
//   contribution of corner k of triangle t to vertex faces[t][k]: -w_k * q, w2 = 1 - w0 - w1
// Reduction order of one vertex (per point window): its contributions sorted stably by vertex, so in ascending
// (point, corner) order, are summed in groups of kDgGroup consecutive ones, left to right starting from the first;
// the group sums are summed the same way, level after level, until one value remains.  That order depends on the
// vertex's own list only, not on where its run lies in the sorted array.
#pragma once
#include "rt_core.cuh"

namespace rt {

constexpr uint32_t kDgGroup = 32;                     // contributions per group of the reduction tree
constexpr uint32_t kDgEmpty = 0xffffffffu;            // key of an unused slot of a level buffer (levels >= 1)
constexpr int64_t kDgMaxPoints = ((int64_t)1 << 30) / 3;   // 3 pairs per point must fit one sort call
constexpr int64_t kDgMaxVerts = 0xffffffffll;              // vertex ids and the sentinel n_verts fit 32 bits

// q of one point; false (and q = +0) when the point contributes nothing: value +-0, +-inf or NaN, or no triangle
RT_HD bool dg_point_q(float px, float py, float pz, float g, float value, float cx, float cy, float cz, int32_t tri,
                      int64_t n_faces, float q[3]) {
    q[0] = q[1] = q[2] = 0.0f;
    const float a = fabsf(value);
    if (!(a > 0.0f) || !(a < as_float(0x7f800000u)) || tri < 0 || (int64_t)tri >= n_faces) return false;
    const float gs = value < 0.0f ? -g : g;
    q[0] = fmul(gs, fdiv(fsub(px, cx), a));
    q[1] = fmul(gs, fdiv(fsub(py, cy), a));
    q[2] = fmul(gs, fdiv(fsub(pz, cz), a));
    return true;
}

// sort key of corner k of a live point: its vertex, or n_verts (sorted last, never summed) for an index out of range
RT_HD uint64_t dg_key(bool live, const int32_t* faces, int32_t tri, uint32_t k, int64_t n_verts) {
    if (!live) return (uint64_t)n_verts;
    const int64_t v = faces[3 * (int64_t)tri + k];
    return v >= 0 && v < n_verts ? (uint64_t)v : (uint64_t)n_verts;
}

// contribution -w_k * q_i of pair e = 3 i + k (q and uv of the window)
RT_HD void dg_contrib(const float* q, const float* uv, uint32_t e, float out[3]) {
    const uint32_t i = e / 3u, k = e % 3u;
    const float u0 = uv[2 * (size_t)i], u1 = uv[2 * (size_t)i + 1];
    const float w = k == 0u ? u0 : (k == 1u ? u1 : fsub(fsub(1.0f, u0), u1));
    out[0] = fmul(-w, q[3 * (size_t)i]);
    out[1] = fmul(-w, q[3 * (size_t)i + 1]);
    out[2] = fmul(-w, q[3 * (size_t)i + 2]);
}

// A level of the tree: slots of (key, index of the value in its vertex's list at this level, value).
struct DgLevel { uint32_t* key; uint32_t* idx; float* val; };

// Ends the group whose first member sits at slot j of a level, index g in its vertex's list, sum s: the vertex's
// total when the group is its whole list (added to grad_vertices), else one member of the next level at slot
// 2 * floor((j - g) / kDgGroup) + g / kDgGroup.  A list longer than kDgGroup starting at slot a of a level
// occupies [2 floor(a / kDgGroup), + ceil(len / kDgGroup)) of the next, which ends before the next such list's slots
// start, and within 2 ceil(slots / kDgGroup) slots.
RT_HD void dg_group_end(uint32_t v, uint64_t j, uint32_t g, bool more, const float s[3], float* grad_vertices,
                        DgLevel next) {
    if (!more) {
        grad_vertices[3 * (size_t)v] = fadd(grad_vertices[3 * (size_t)v], s[0]);
        grad_vertices[3 * (size_t)v + 1] = fadd(grad_vertices[3 * (size_t)v + 1], s[1]);
        grad_vertices[3 * (size_t)v + 2] = fadd(grad_vertices[3 * (size_t)v + 2], s[2]);
        return;
    }
    const uint64_t o = 2 * ((j - g) / kDgGroup) + g / kDgGroup;
    next.key[o] = v;
    next.idx[o] = g / kDgGroup;
    next.val[3 * o] = s[0]; next.val[3 * o + 1] = s[1]; next.val[3 * o + 2] = s[2];
}

// Level 0 at sorted position j of m pairs: start[v] = first position of vertex v (written by dg_run_start);
// contrib(e, out) is the contribution of pair e.
template <class Contrib>
RT_HD void dg_level0_with(uint64_t j, uint64_t m, const uint64_t* keys, const uint32_t* vals, const uint32_t* start,
                          uint64_t n_verts, const Contrib& contrib, float* grad_vertices, DgLevel next) {
    const uint64_t key = keys[j];
    if (key >= n_verts) return;
    const uint32_t v = (uint32_t)key;
    const uint32_t g = (uint32_t)(j - start[v]);
    if (g % kDgGroup != 0u) return;
    float s[3], c[3];
    contrib(vals[j], s);
    for (uint64_t t = 1; t < kDgGroup && j + t < m && keys[j + t] == key; ++t) {
        contrib(vals[j + t], c);
        s[0] = fadd(s[0], c[0]); s[1] = fadd(s[1], c[1]); s[2] = fadd(s[2], c[2]);
    }
    const bool more = g > 0u || (j + kDgGroup < m && keys[j + kDgGroup] == key);
    dg_group_end(v, j, g, more, s, grad_vertices, next);
}

// Level 0 of the point and hit-row sums: pair e = 3 i + k contributes -w_k q_i (dg_contrib)
RT_HD void dg_level0_at(uint64_t j, uint64_t m, const uint64_t* keys, const uint32_t* vals, const uint32_t* start,
                        uint64_t n_verts, const float* q, const float* uv, float* grad_vertices, DgLevel next) {
    dg_level0_with(j, m, keys, vals, start, n_verts, [&](uint32_t e, float out[3]) { dg_contrib(q, uv, e, out); },
                   grad_vertices, next);
}

RT_HD void dg_run_start(uint64_t j, const uint64_t* keys, uint64_t n_verts, uint32_t* start) {
    const uint64_t key = keys[j];
    if (key < n_verts && (j == 0 || keys[j - 1] != key)) start[key] = (uint32_t)j;
}

// Level >= 1 at slot j of `size` slots
RT_HD void dg_level_at(uint64_t j, uint64_t size, DgLevel cur, float* grad_vertices, DgLevel next) {
    const uint32_t v = cur.key[j];
    if (v == kDgEmpty) return;
    const uint32_t g = cur.idx[j];
    if (g % kDgGroup != 0u) return;
    float s[3] = {cur.val[3 * j], cur.val[3 * j + 1], cur.val[3 * j + 2]};
    for (uint64_t t = 1; t < kDgGroup && j + t < size && cur.key[j + t] == v; ++t) {
        s[0] = fadd(s[0], cur.val[3 * (j + t)]);
        s[1] = fadd(s[1], cur.val[3 * (j + t) + 1]);
        s[2] = fadd(s[2], cur.val[3 * (j + t) + 2]);
    }
    const bool more = g > 0u || (j + kDgGroup < size && cur.key[j + kDgGroup] == v);
    dg_group_end(v, j, g, more, s, grad_vertices, next);
}

// slots of the level after one of `size` slots
RT_HD uint64_t dg_next_size(uint64_t size) { return 2 * ((size + kDgGroup - 1) / kDgGroup); }

// radix-sort passes (8 bits each) that order keys 0..n_verts
RT_HD int dg_sort_passes(int64_t n_verts) {
    int bits = 0;
    while (bits < 64 && ((uint64_t)n_verts >> bits) != 0) ++bits;
    return bits == 0 ? 1 : (bits + 7) / 8;
}

}  // namespace rt
