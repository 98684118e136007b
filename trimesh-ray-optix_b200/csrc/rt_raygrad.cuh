// rt_raygrad.cuh — the arithmetic of the hit gradient (rt_ray_grad in rt_distgrad.cu, DESIGN.md §4.10): the per-row
// factor lambda, the barycentric weights, the zero rules and the per-ray row sums.  Everything here is RT_HD, like
// rt_distgrad.cuh, so that tests/raygrad/ runs exactly the code the kernels run.  The vertex sums are those of
// rt_distgrad.cuh, with q = lambda - g_L and uv = w.
//
// For a row with ray (o, d), triangle t = (v0, v1, v2), e1 = v1 - v0, e2 = v2 - v0 and incoming gradients g_L (of
// loc) and g_U (of uv), the hit is recomputed with one fixed Moeller-Trumbore sequence in binary32:
//   s = o - v0, p = d x e2, det = e1.p, b1 = s.p / det, r = s x e1, b2 = d.r / det, t = e2.r / det
// and then
//   gb1 = g_L.e1 - g_U0 + g_U1, gb2 = g_L.e2 - g_U0, lambda = (gb1 p + gb2 (e1 x d)) / det
//   grad_o += lambda, grad_d += t lambda, corner k of t gets -w_k q with q = lambda - g_L, w = (1 - b1 - b2, b1)
// (the weight of corner 2 is 1 - w0 - w1, as in rt_distgrad.cuh).
#pragma once
#include "rt_distgrad.cuh"

namespace rt {

struct RgMesh {
    const float* vertices;       // [n_verts, 3]
    int64_t n_verts;
    const int32_t* faces;        // [n_faces, 3]
    int64_t n_faces;
};

// What one row writes: lambda (its grad_o term), t lambda (its grad_d term), q and w.  All +0 for a dead row.
struct RgRow { float lam[3], tlam[3], q[3], w[2]; };

RT_HD float rg_dot(const float a[3], const float b[3]) {
    return fadd(fadd(fmul(a[0], b[0]), fmul(a[1], b[1])), fmul(a[2], b[2]));
}

RT_HD void rg_cross(const float a[3], const float b[3], float out[3]) {
    out[0] = fsub(fmul(a[1], b[2]), fmul(a[2], b[1]));
    out[1] = fsub(fmul(a[2], b[0]), fmul(a[0], b[2]));
    out[2] = fsub(fmul(a[0], b[1]), fmul(a[1], b[0]));
}

RT_HD bool rg_finite(float x) { return fabsf(x) < as_float(0x7f800000u); }

// One row; false (and r all +0) when it contributes nothing: triangle outside [0, n_faces), a vertex index outside
// [0, n_verts), det = 0, or any value it would write (lambda, t lambda, q, w and the weight of corner 2) not finite.
RT_HD bool rg_row(const float o[3], const float d[3], const float gl[3], float gu0, float gu1, int32_t tri,
                  const RgMesh& m, RgRow& r) {
    for (int c = 0; c < 3; ++c) r.lam[c] = r.tlam[c] = r.q[c] = 0.0f;
    r.w[0] = r.w[1] = 0.0f;
    if (tri < 0 || (int64_t)tri >= m.n_faces) return false;
    float v[3][3];
    for (int k = 0; k < 3; ++k) {
        const int64_t vi = m.faces[3 * (int64_t)tri + k];
        if (vi < 0 || vi >= m.n_verts) return false;
        for (int c = 0; c < 3; ++c) v[k][c] = m.vertices[3 * vi + c];
    }
    float e1[3], e2[3], s[3], p[3], rr[3], ed[3], lam[3], tlam[3], q[3];
    for (int c = 0; c < 3; ++c) {
        e1[c] = fsub(v[1][c], v[0][c]);
        e2[c] = fsub(v[2][c], v[0][c]);
        s[c] = fsub(o[c], v[0][c]);
    }
    rg_cross(d, e2, p);
    const float det = rg_dot(e1, p);
    if (det == 0.0f) return false;
    const float b1 = fdiv(rg_dot(s, p), det);
    rg_cross(s, e1, rr);
    const float b2 = fdiv(rg_dot(d, rr), det);
    const float t = fdiv(rg_dot(e2, rr), det);
    const float gb1 = fadd(fsub(rg_dot(gl, e1), gu0), gu1);
    const float gb2 = fsub(rg_dot(gl, e2), gu0);
    rg_cross(e1, d, ed);
    bool ok = true;
    for (int c = 0; c < 3; ++c) {
        lam[c] = fdiv(fadd(fmul(gb1, p[c]), fmul(gb2, ed[c])), det);
        tlam[c] = fmul(t, lam[c]);
        q[c] = fsub(lam[c], gl[c]);
        ok = ok && rg_finite(lam[c]) && rg_finite(tlam[c]) && rg_finite(q[c]);
    }
    const float w0 = fsub(fsub(1.0f, b1), b2);
    ok = ok && rg_finite(w0) && rg_finite(b1) && rg_finite(fsub(fsub(1.0f, w0), b1));
    if (!ok) return false;
    for (int c = 0; c < 3; ++c) { r.lam[c] = lam[c]; r.tlam[c] = tlam[c]; r.q[c] = q[c]; }
    r.w[0] = w0; r.w[1] = b1;
    return true;
}

// Row j heads its ray's run of rows (row_ray null: every row is its own run).
RT_HD bool rg_head(int64_t j, const int32_t* row_ray) { return row_ray == nullptr || j == 0 || row_ray[j - 1] != row_ray[j]; }

// grad_o and grad_d of the ray whose run starts at row j: the rows' lambda and t lambda summed left to right in row
// order, from +0.  `row(k, r)` evaluates row k.
template <class RowFn>
RT_HD void rg_ray_sums(int64_t j, int64_t n_rows, const int32_t* row_ray, const RowFn& row, float go[3], float gd[3]) {
    go[0] = go[1] = go[2] = gd[0] = gd[1] = gd[2] = 0.0f;
    int64_t k = j;
    do {
        RgRow r;
        row(k, r);
        for (int c = 0; c < 3; ++c) { go[c] = fadd(go[c], r.lam[c]); gd[c] = fadd(gd[c], r.tlam[c]); }
        ++k;
    } while (row_ray != nullptr && k < n_rows && row_ray[k] == row_ray[j]);
}

}  // namespace rt
