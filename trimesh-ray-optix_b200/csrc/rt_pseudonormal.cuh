// rt_pseudonormal.cuh — angle-weighted pseudo-normals (Bærentzen & Aanæs 2005) of the triangles of a BVH8 blob: the
// corner weld, the per-vertex and per-edge sums and the row layout the signed-distance kernel reads.  Everything here
// is RT_HD, like rt_point.cuh and rt_winding.cuh, so that tests/pseudonormal/ runs exactly the code of
// rt_pseudonormal.cu on the CPU (with std::stable_sort in place of the onesweep sort: a stable sort of the same keys
// gives the same permutation).
//
// Contract (DESIGN.md §4.8): corners are welded by exact equality of their coordinates (-0 counted as +0), from the
// blob alone; a triangle with a non-finite vertex takes part in nothing.  Each sum runs over its group in ascending
// corner / half-edge index, so the rows are a function of the blob alone.
#pragma once
#include "rt_winding.cuh"

namespace rt {

// One row of 6 x 16 bytes per triangle RECORD (the slot the closest-point walk ends on, not the prim): the
// pseudo-normals of vertex a, b, c and of edge ab, ac, bc, i.e. the row slot of region r (rt_point.cuh) is r - 1.  The
// face region needs no entry: its normal is recomputed from the record.
constexpr uint32_t kPnRowBytes = 96;
constexpr uint64_t kPnNoKey = ~0ull;        // corners and half-edges of non-finite triangles: sorted last, never welded

// half-edge k of a record runs from corner k to corner (k + 1) % 3: ab, bc, ca; their row slots
RT_HD uint32_t half_edge_slot(uint32_t k) { return k == 0u ? 3u : (k == 1u ? 5u : 4u); }

RT_HD bool tri_finite(const float v[9]) {
    return finite3(v[0], v[1], v[2]) && finite3(v[3], v[4], v[5]) && finite3(v[6], v[7], v[8]);
}

// coordinate bits with -0 taken as +0, so that the two zeros weld
RT_HD uint32_t weld_bits(float x) { return x == 0.0f ? 0u : as_uint(x); }

// the two sort keys of a corner: z first (LSD), then (x << 32 | y); the stable second sort orders by (x, y, z)
RT_HD uint64_t corner_key_z(const float v[9], uint32_t k) { return (uint64_t)weld_bits(v[3 * k + 2]); }
RT_HD uint64_t corner_key_xy(const float v[9], uint32_t k) {
    return ((uint64_t)weld_bits(v[3 * k]) << 32) | (uint64_t)weld_bits(v[3 * k + 1]);
}
RT_HD bool same_corner(const float a[9], uint32_t ka, const float b[9], uint32_t kb) {
    return weld_bits(a[3 * ka]) == weld_bits(b[3 * kb]) && weld_bits(a[3 * ka + 1]) == weld_bits(b[3 * kb + 1]) &&
           weld_bits(a[3 * ka + 2]) == weld_bits(b[3 * kb + 2]);
}

// unit face normal (v1 - v0) x (v2 - v0) / |.|; the zero vector when the computed cross product has zero length
RT_HD void face_unit_normal(const float v[9], float& x, float& y, float& z) {
    const float e1x = fsub(v[3], v[0]), e1y = fsub(v[4], v[1]), e1z = fsub(v[5], v[2]);
    const float e2x = fsub(v[6], v[0]), e2y = fsub(v[7], v[1]), e2z = fsub(v[8], v[2]);
    x = fsub(fmul(e1y, e2z), fmul(e1z, e2y));
    y = fsub(fmul(e1z, e2x), fmul(e1x, e2z));
    z = fsub(fmul(e1x, e2y), fmul(e1y, e2x));
    unit3(x, y, z);
}

// interior angle at corner k: atan2(|e1 x e2|, e1 . e2) of the unit edge vectors leaving the corner (unit vectors keep
// the products in range at any scale); 0 when an edge has zero length
RT_HD float corner_angle(const float v[9], uint32_t k) {
    const uint32_t i = k, j = (k + 1u) % 3u, l = (k + 2u) % 3u;
    float e1x = fsub(v[3 * j], v[3 * i]), e1y = fsub(v[3 * j + 1], v[3 * i + 1]), e1z = fsub(v[3 * j + 2], v[3 * i + 2]);
    float e2x = fsub(v[3 * l], v[3 * i]), e2y = fsub(v[3 * l + 1], v[3 * i + 1]), e2z = fsub(v[3 * l + 2], v[3 * i + 2]);
    if (!(unit3(e1x, e1y, e1z) > 0.0f && unit3(e2x, e2y, e2z) > 0.0f)) return 0.0f;
    const float cx = fsub(fmul(e1y, e2z), fmul(e1z, e2y));
    const float cy = fsub(fmul(e1z, e2x), fmul(e1x, e2z));
    const float cz = fsub(fmul(e1x, e2y), fmul(e1y, e2x));
    return atan2_rn(fsqrt(dot3f(cx, cy, cz, cx, cy, cz)), dot3f(e1x, e1y, e1z, e2x, e2y, e2z));
}

RT_HD void store_row_slot(uint8_t* normals, uint32_t rec, uint32_t slot, float x, float y, float z) {
    float* q = reinterpret_cast<float*>(normals + (size_t)rec * kPnRowBytes + (size_t)slot * 16u);
    q[0] = x; q[1] = y; q[2] = z; q[3] = 0.0f;
}

// ------------------------------------------------------------------ corner weld
// `sorted` = the 3n corner indices (3 * record + slot) ordered by (x, y, z) with non-finite triangles last.  Called for
// sorted position j: a non-finite triangle's corner zeroes its own row slot; the head of a run of equal coordinates
// sums sum_i alpha_i n^_i over the run in order, then writes the vertex normal and the vertex id (= j) of every member.
// Positions that are neither return at once.
RT_HD void weld_run(const uint8_t* tris, const uint32_t* sorted, uint32_t n_corners, uint32_t j, uint32_t* vid,
                    uint8_t* normals) {
    const uint32_t c = sorted[j];
    float v[9];
    load_tri(tris, c / 3u, v);
    if (!tri_finite(v)) {
        vid[c] = 0xffffffffu;
        store_row_slot(normals, c / 3u, c % 3u, 0.0f, 0.0f, 0.0f);
        return;
    }
    if (j > 0u) {
        const uint32_t cp = sorted[j - 1u];
        float w[9];
        load_tri(tris, cp / 3u, w);
        if (same_corner(v, c % 3u, w, cp % 3u)) return;   // a finite predecessor with the same coordinates: not a head
    }
    float sx = 0.0f, sy = 0.0f, sz = 0.0f;
    uint32_t end = j;
    for (; end < n_corners; ++end) {
        const uint32_t m = sorted[end];
        float w[9];
        load_tri(tris, m / 3u, w);
        if (!tri_finite(w) || !same_corner(v, c % 3u, w, m % 3u)) break;
        float nx, ny, nz;
        face_unit_normal(w, nx, ny, nz);
        const float a = corner_angle(w, m % 3u);
        sx = fadd(sx, fmul(a, nx)); sy = fadd(sy, fmul(a, ny)); sz = fadd(sz, fmul(a, nz));
    }
    for (uint32_t m = j; m < end; ++m) {
        const uint32_t cm = sorted[m];
        vid[cm] = j;
        store_row_slot(normals, cm / 3u, cm % 3u, sx, sy, sz);
    }
}

// ------------------------------------------------------------------ edges
// key of half-edge h = 3 * record + k (corner k to corner k + 1): (min id << 32 | max id) of its two vertex ids
RT_HD uint64_t half_edge_key(const uint32_t* vid, uint32_t h) {
    const uint32_t r = h / 3u, k = h % 3u;
    const uint32_t a = vid[3u * r + k], b = vid[3u * r + (k + 1u) % 3u];
    if (a == 0xffffffffu || b == 0xffffffffu) return kPnNoKey;
    return a < b ? ((uint64_t)a << 32) | b : ((uint64_t)b << 32) | a;
}

// `sorted` / `keys` = the 3n half-edges ordered by key.  Called for sorted position j: a half-edge of a non-finite
// triangle zeroes its row slot; the head of a run of equal keys sums the unit face normals of the run in order,
// writes the edge normal into every member's row and classifies the edge: one face = boundary (counts[0]), more than
// two = non-manifold (counts[1]), two that run the same way = inconsistent (counts[2]).
struct EdgeRun { uint32_t faces, forward; float x, y, z; };

RT_HD bool edge_head(const uint64_t* keys, uint32_t j) { return keys[j] != kPnNoKey && (j == 0u || keys[j - 1u] != keys[j]); }

RT_HD EdgeRun edge_run(const uint8_t* tris, const uint32_t* sorted, const uint64_t* keys, uint32_t n_half, uint32_t j,
                       const uint32_t* vid, uint8_t* normals) {
    EdgeRun e = {0u, 0u, 0.0f, 0.0f, 0.0f};
    uint32_t end = j;
    for (; end < n_half && keys[end] == keys[j]; ++end) {
        const uint32_t h = sorted[end];
        float w[9];
        load_tri(tris, h / 3u, w);
        float nx, ny, nz;
        face_unit_normal(w, nx, ny, nz);
        e.x = fadd(e.x, nx); e.y = fadd(e.y, ny); e.z = fadd(e.z, nz);
        ++e.faces;
        const uint32_t r = h / 3u, k = h % 3u;
        if (vid[3u * r + k] <= vid[3u * r + (k + 1u) % 3u]) ++e.forward;
    }
    for (uint32_t m = j; m < end; ++m) {
        const uint32_t h = sorted[m];
        store_row_slot(normals, h / 3u, half_edge_slot(h % 3u), e.x, e.y, e.z);
    }
    return e;
}

RT_HD uint32_t edge_class(const EdgeRun& e) {   // 0 boundary, 1 non-manifold, 2 inconsistent, 3 fine
    if (e.faces == 1u) return 0u;
    if (e.faces > 2u) return 1u;
    return e.forward == 1u ? 3u : 2u;
}

// ------------------------------------------------------------------ the sign
// +d when (p - c) . n < 0 (inside), -d otherwise; an exact d = 0 gives +0.  n is the pseudo-normal of the region of c:
// the unit face normal for the face, the record's row for a vertex or an edge.
RT_HD void region_normal(const uint8_t* normals, uint32_t rec, uint32_t region, const float v[9], float& nx, float& ny,
                         float& nz) {
    if (region == kRegionFace) {
        face_unit_normal(v, nx, ny, nz);
    } else {
        const U4 q = ldg128(normals + (size_t)rec * kPnRowBytes + (size_t)(region - 1u) * 16u);
        nx = as_float(q.x); ny = as_float(q.y); nz = as_float(q.z);
    }
}

RT_HD float pseudonormal_sign(const uint8_t* normals, uint32_t rec, const PointHit& h, float px, float py, float pz,
                              const float v[9], float d) {
    float nx, ny, nz;
    region_normal(normals, rec, h.region, v, nx, ny, nz);
    const float s = dot3f(fsub(px, h.cx), fsub(py, h.cy), fsub(pz, h.cz), nx, ny, nz);
    return (s < 0.0f || d == 0.0f) ? d : -d;
}

}  // namespace rt
