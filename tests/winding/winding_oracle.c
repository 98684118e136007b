/* winding_oracle.c — TEST INFRASTRUCTURE ONLY.  The truth oracle of the generalized winding number: a brute-force sum
 * over every triangle in binary64 (OpenMP over the points), with the edge-case contract of rt_winding.cuh:
 *   - a triangle with a non-finite vertex contributes 0;
 *   - a triangle whose det = a . ((v1 - v0) x (v2 - v0)) (= det[a b c]) is exactly 0 contributes 0 (q in its plane,
 *     on it, zero area), and so does one with q at a vertex;
 *   - a non-finite point gives NaN; an empty mesh gives +0.
 * Omega = 2 atan2(det, |a||b||c| + (a.b)|c| + (b.c)|a| + (c.a)|b|) (van Oosterom & Strackee), w = sum Omega / 4 pi.
 *
 * Build: gcc -O2 -fopenmp -ffp-contract=off -fPIC -shared winding_oracle.c -o libwindoracle.so -lm
 */
#include <math.h>
#include <stdint.h>

static int finite3(const double* v) { return isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2]); }

static double solid_angle64(const double* q, const double* v0, const double* v1, const double* v2) {
    if (!finite3(v0) || !finite3(v1) || !finite3(v2)) return 0.0;
    const double a[3] = {v0[0] - q[0], v0[1] - q[1], v0[2] - q[2]};
    const double b[3] = {v1[0] - q[0], v1[1] - q[1], v1[2] - q[2]};
    const double c[3] = {v2[0] - q[0], v2[1] - q[1], v2[2] - q[2]};
    const double la = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    const double lb = sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]);
    const double lc = sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
    if (la == 0.0 || lb == 0.0 || lc == 0.0) return 0.0;          /* q at a vertex */
    /* det[a b c] = a . ((v1 - v0) x (v2 - v0)): exactly 0 for a repeated vertex or exactly collinear vertices */
    const double e1[3] = {v1[0] - v0[0], v1[1] - v0[1], v1[2] - v0[2]};
    const double e2[3] = {v2[0] - v0[0], v2[1] - v0[1], v2[2] - v0[2]};
    const double n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
    const double det = a[0] * n[0] + a[1] * n[1] + a[2] * n[2];
    if (det == 0.0) return 0.0;
    const double ab = a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
    const double bc = b[0] * c[0] + b[1] * c[1] + b[2] * c[2];
    const double ca = c[0] * a[0] + c[1] * a[1] + c[2] * a[2];
    return 2.0 * atan2(det, la * lb * lc + ab * lc + bc * la + ca * lb);
}

/* w[i] for n points; vertices float32 [nv, 3] (widened exactly), faces int32 [nf, 3] (indices assumed valid) */
int wo_winding(const float* verts, int64_t nv, const int32_t* faces, int64_t nf, int64_t n, const float* pts, double* w) {
    (void)nv;
    const double inv4pi = 1.0 / (4.0 * 3.14159265358979323846);
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < n; ++i) {
        const double q[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
        if (!finite3(q)) { w[i] = NAN; continue; }
        double s = 0.0;
        for (int64_t t = 0; t < nf; ++t) {
            double v[3][3];
            for (int k = 0; k < 3; ++k)
                for (int j = 0; j < 3; ++j) v[k][j] = verts[3 * (int64_t)faces[3 * t + k] + j];
            s += solid_angle64(q, v[0], v[1], v[2]);
        }
        w[i] = s * inv4pi;
    }
    return 0;
}

/* atan2 and the solid angle of one triangle in binary64, for the known-answer tests */
double wo_solid_angle(const double* q, const double* tri) { return solid_angle64(q, tri, tri + 3, tri + 6); }
