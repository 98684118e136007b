// rt_scenegrad.cuh — the arithmetic of the instanced-scene gradients (rt_distgrad.cu, DESIGN.md §4.13): the per-row
// factors of hit rows and point rows, the pairs of the joint key space and their level-0 contributions.  Everything
// here is RT_HD, like rt_raygrad.cuh, so that tests/scenegrad/ runs exactly the code the kernels run.
//
// A row of instance i (transform A | b from the table) and triangle t of its member (object vertices v_k) ends on the
// world triangle W_k = affine_row(A row, b (0 as -0), v_k).  Hit rows recompute the hit with rg_row on that world
// triangle; point rows take q from dg_point_q and w from the forward's uv.  Then, in binary32:
//   w2 = (1 - w0) - w1,  x_c = (w0 v0_c + w1 v1_c) + w2 v2_c,  q_obj_j = affine_row(A column j, -0, q)
// and the row's pairs are (key, pair index) with the keys
//   slot k < 3:  vertex_base + faces[t][k]              contribution -w_k q_obj
//   slot 3 + j:  n_verts + 4 i + j   (column j of A|b)  contribution -x_j q (j < 3), -q (j = 3)
// q_obj uses the stored fwd columns with offset -0 and zero coefficients skipped, as scene_pseudonormal_sign forms
// A^-T n: an identity instance gives q_obj = q bit for bit, so its vertex sums are those of rt_ray_grad /
// rt_distance_grad.
#pragma once
#include "rt_raygrad.cuh"
#include "rt_scene.cuh"

namespace rt {

constexpr int kSgRowFloats = 11;                               // q, q_obj, x, w0, w1
constexpr int64_t kSgMaxRows = ((int64_t)1 << 30) / 7;         // 7 pairs per row must fit one sort call

// The scene as the backward sees it: the table, the bounds of what a row may index, the member table and the size
// n_verts of the member-vertex part of the key space.
struct SgScene {
    SceneView sv;
    int64_t n_inst, n_meshes;
    const rt_scene_member* members;
    int64_t n_verts;
};

RT_HD SgScene sg_scene(const uint8_t* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                       int64_t n_verts) {
    const SceneHeader* h = reinterpret_cast<const SceneHeader*>(table);
    SgScene s;
    s.sv = scene_view(table);
    s.n_inst = (int64_t)h->n_inst < n_inst ? (int64_t)h->n_inst : n_inst;
    s.n_meshes = (int64_t)h->n_meshes < n_meshes ? (int64_t)h->n_meshes : n_meshes;
    s.members = members;
    s.n_verts = n_verts;
    return s;
}

// Per-row factors of a live row (all +0 for a dead one).
struct SgRow { float q[3], qo[3], x[3], w[2]; };

// The record and object vertices of row (inst, tri), and the keys of its three vertices; false when the row
// contributes nothing: inst or its mesh out of range, tri outside the member's faces, a vertex index outside its
// vertices or its key outside [0, n_verts).
RT_HD bool sg_triangle(const SgScene& sc, int32_t inst, int32_t tri, const SceneInst*& s, float v[9], uint64_t key[3]) {
    if (inst < 0 || (int64_t)inst >= sc.n_inst) return false;
    s = &sc.sv.inst[inst];
    if (s->mesh < 0 || (int64_t)s->mesh >= sc.n_meshes) return false;
    const rt_scene_member& m = sc.members[s->mesh];
    if (tri < 0 || (int64_t)tri >= m.n_faces) return false;
    for (int k = 0; k < 3; ++k) {
        const int64_t vi = m.faces[3 * (int64_t)tri + k];
        if (vi < 0 || vi >= m.n_verts) return false;
        const int64_t g = m.vertex_base + vi;
        if (g < 0 || g >= sc.n_verts) return false;
        key[k] = (uint64_t)g;
        for (int c = 0; c < 3; ++c) v[3 * k + c] = m.vertices[3 * vi + c];
    }
    return true;
}

// w2, x and q_obj of a row with q and (w0, w1); false (r all +0) when any of q, w, x, q_obj is not finite.
RT_HD bool sg_finish(const float fwd[12], const float v[9], const float q[3], float w0, float w1, SgRow& r) {
    const float w2 = fsub(fsub(1.0f, w0), w1);
    const float nz = as_float(0x80000000u);
    float x[3], qo[3];
    bool ok = rg_finite(w0) && rg_finite(w1) && rg_finite(w2);
    for (int c = 0; c < 3; ++c) {
        x[c] = fadd(fadd(fmul(w0, v[c]), fmul(w1, v[3 + c])), fmul(w2, v[6 + c]));
        qo[c] = affine_row(fwd[c], fwd[4 + c], fwd[8 + c], nz, q[0], q[1], q[2]);
        ok = ok && rg_finite(q[c]) && rg_finite(x[c]) && rg_finite(qo[c]);
    }
    for (int c = 0; c < 3; ++c) r.q[c] = r.qo[c] = r.x[c] = 0.0f;
    r.w[0] = r.w[1] = 0.0f;
    if (!ok) return false;
    for (int c = 0; c < 3; ++c) { r.q[c] = q[c]; r.qo[c] = qo[c]; r.x[c] = x[c]; }
    r.w[0] = w0; r.w[1] = w1;
    return true;
}

// A hit row: rg_row on the world triangle (rr: lambda, t lambda, q, w), then sg_finish; false (rr and r all +0) when
// the row contributes nothing.
RT_HD bool sg_hit_row(const SgScene& sc, int32_t inst, int32_t tri, const float o[3], const float d[3], const float gl[3],
                      float gu0, float gu1, RgRow& rr, SgRow& r, uint64_t key[3]) {
    const SceneInst* s = nullptr;
    float v[9], wv[9];
    const int32_t f[3] = {0, 1, 2};
    const bool found = sg_triangle(sc, inst, tri, s, v, key);
    if (found) {
        for (int c = 0; c < 3; ++c) {
            const float* m = s->fwd + 4 * c;
            const float bc = zero_as_negative(m[3]);
            for (int k = 0; k < 3; ++k) wv[3 * k + c] = affine_row(m[0], m[1], m[2], bc, v[3 * k], v[3 * k + 1], v[3 * k + 2]);
        }
    }
    const RgMesh world{wv, 3, f, 1};
    bool live = rg_row(o, d, gl, gu0, gu1, found ? 0 : -1, world, rr);
    live = live && sg_finish(s->fwd, v, rr.q, rr.w[0], rr.w[1], r);
    if (!live) {
        for (int c = 0; c < 3; ++c) rr.lam[c] = rr.tlam[c] = rr.q[c] = r.q[c] = r.qo[c] = r.x[c] = 0.0f;
        rr.w[0] = rr.w[1] = r.w[0] = r.w[1] = 0.0f;
    }
    return live;
}

// A point row: q of dg_point_q (over the member's faces), w = (uv0, uv1), then sg_finish; false (q and r all +0) when
// the row contributes nothing.
RT_HD bool sg_point_row(const SgScene& sc, int32_t inst, int32_t tri, float px, float py, float pz, float g, float value,
                        float cx, float cy, float cz, float u0, float u1, float q[3], SgRow& r, uint64_t key[3]) {
    const SceneInst* s = nullptr;
    float v[9];
    bool live = sg_triangle(sc, inst, tri, s, v, key);
    live = live && dg_point_q(px, py, pz, g, value, cx, cy, cz, 0, 1, q);
    live = live && sg_finish(s->fwd, v, q, u0, u1, r);
    if (!live) {
        for (int c = 0; c < 3; ++c) q[c] = r.q[c] = r.qo[c] = r.x[c] = 0.0f;
        r.w[0] = r.w[1] = 0.0f;
    }
    return live;
}

// Key of slot s (0..6) of a row of instance inst; n_keys (sorted last, never summed) for a dead row.
RT_HD uint64_t sg_key(bool live, const uint64_t vkey[3], int32_t inst, int s, uint64_t n_verts, uint64_t n_keys) {
    if (!live) return n_keys;
    return s < 3 ? vkey[s] : n_verts + 4u * (uint64_t)inst + (uint64_t)(s - 3);
}

// Contribution of pair e = n_slots i + (s - slot0) of a window whose rows' factors are rec[kSgRowFloats i ...]
RT_HD void sg_contrib(const float* rec, int slot0, int n_slots, uint32_t e, float out[3]) {
    const uint32_t i = e / (uint32_t)n_slots;
    const int s = (int)(e % (uint32_t)n_slots) + slot0;
    const float* r = rec + (size_t)kSgRowFloats * i;     // q 0..2, q_obj 3..5, x 6..8, w 9..10
    if (s < 3) {
        const float w = s == 0 ? r[9] : (s == 1 ? r[10] : fsub(fsub(1.0f, r[9]), r[10]));
        for (int c = 0; c < 3; ++c) out[c] = fmul(-w, r[3 + c]);
    } else if (s < 6) {
        for (int c = 0; c < 3; ++c) out[c] = fmul(-r[6 + s - 3], r[c]);
    } else {
        for (int c = 0; c < 3; ++c) out[c] = -r[c];
    }
}

RT_HD void sg_store(const SgRow& r, float* rec) {
    for (int c = 0; c < 3; ++c) { rec[c] = r.q[c]; rec[3 + c] = r.qo[c]; rec[6 + c] = r.x[c]; }
    rec[9] = r.w[0]; rec[10] = r.w[1];
}

// grad_transforms[i][r][j] from the sum of key n_verts + 4 i + j
RT_HD void sg_transform_out(const float* acc, uint64_t n_verts, uint64_t e, float* grad_transforms) {
    const uint64_t i = e / 12u, r = (e % 12u) / 4u, j = e % 4u;
    grad_transforms[e] = acc[3 * (n_verts + 4u * i + j) + r];
}

}  // namespace rt
