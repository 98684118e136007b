/*
 * point_oracle.c — CPU ORACLE of the closest-point query (rt_closest_point).  TEST INFRASTRUCTURE, never linked into
 * the product.  Compile with -ffp-contract=off.
 *
 * Contract checked: for each point, the triangle minimising the key (d2, prim) over all triangles with
 * d2 <= max_d2, where d2 is the squared distance of the closest point point_tri() computes.
 *   MIRROR (mode 1): binary32, point_tri in the operation sequence of the product (point_tri.inc with REAL = float),
 *                    max_d2 = fl(m * m): results must equal the GPU's bit for bit.
 *   TRUTH  (mode 0): the same algorithm in binary64, max_d2 = m * m in binary64.
 * Candidates are all triangles (brute force, bvh = NULL) or those a median-split BVH2 cannot exclude: a subtree is
 * skipped only when its box, widened by 1e-5 of the coordinates' magnitude (more than the rounding of a binary32
 * closest point), is farther than the best d2 so far (with a relative slack of 1e-6 for the rounding of d2).
 * Points are processed in parallel with OpenMP.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define REAL float
#define PT_NAME(x) f_##x
#include "point_tri.inc"
#undef REAL
#undef PT_NAME
#define REAL double
#define PT_NAME(x) d_##x
#include "point_tri.inc"
#undef REAL
#undef PT_NAME

typedef struct {
    const float* verts;
    const int32_t* faces;
    int64_t nv, nf;
} PMesh;

static const float* pvert(const PMesh* m, int64_t tri, int c) {
    int32_t i = m->faces[3 * tri + c];
    if (i < 0) i = 0;
    if (i >= m->nv) i = (int32_t)(m->nv - 1);
    return m->verts + 3 * (size_t)i;
}

typedef struct { double lo[3], hi[3]; int32_t left, right, first, count; } PNode;
typedef struct { PMesh mesh; PNode* nodes; int32_t* order; int32_t n_nodes; } PBvh;

static void tri_box(const PMesh* m, int32_t t, double lo[3], double hi[3], double c[3]) {
    for (int a = 0; a < 3; ++a) { lo[a] = INFINITY; hi[a] = -INFINITY; }
    for (int k = 0; k < 3; ++k) {
        const float* v = pvert(m, t, k);
        for (int a = 0; a < 3; ++a) { if (v[a] < lo[a]) lo[a] = v[a]; if (v[a] > hi[a]) hi[a] = v[a]; }
    }
    for (int a = 0; a < 3; ++a) c[a] = lo[a] <= hi[a] ? 0.5 * (lo[a] + hi[a]) : 0.0;
}

static double* g_cent;   /* centroids during the build (single-threaded) */
static int g_axis;
static int cmp_cent(const void* x, const void* y) {
    const double a = g_cent[3 * (size_t)*(const int32_t*)x + g_axis], b = g_cent[3 * (size_t)*(const int32_t*)y + g_axis];
    return a < b ? -1 : (a > b ? 1 : 0);
}

static int32_t pbuild(PBvh* b, const double* lo, const double* hi, int32_t first, int32_t count) {
    const int32_t id = b->n_nodes++;
    PNode* n = &b->nodes[id];
    double clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int a = 0; a < 3; ++a) { n->lo[a] = INFINITY; n->hi[a] = -INFINITY; }
    for (int32_t i = first; i < first + count; ++i) {
        const int32_t t = b->order[i];
        for (int a = 0; a < 3; ++a) {
            if (lo[3 * (size_t)t + a] < n->lo[a]) n->lo[a] = lo[3 * (size_t)t + a];
            if (hi[3 * (size_t)t + a] > n->hi[a]) n->hi[a] = hi[3 * (size_t)t + a];
            const double c = g_cent[3 * (size_t)t + a];
            if (c < clo[a]) clo[a] = c;
            if (c > chi[a]) chi[a] = c;
        }
    }
    n->left = n->right = -1; n->first = first; n->count = count;
    if (count <= 4) return id;
    int axis = 0;
    for (int a = 1; a < 3; ++a) if (chi[a] - clo[a] > chi[axis] - clo[axis]) axis = a;
    g_axis = axis;
    qsort(b->order + first, (size_t)count, sizeof(int32_t), cmp_cent);
    const int32_t half = count / 2;
    const int32_t l = pbuild(b, lo, hi, first, half);
    const int32_t r = pbuild(b, lo, hi, first + half, count - half);
    b->nodes[id].left = l; b->nodes[id].right = r;
    return id;
}

void* point_bvh_build(const float* verts, int64_t nv, const int32_t* faces, int64_t nf) {
    PBvh* b = (PBvh*)calloc(1, sizeof(PBvh));
    b->mesh.verts = verts; b->mesh.faces = faces; b->mesh.nv = nv; b->mesh.nf = nf;
    if (nf == 0) return b;
    b->nodes = (PNode*)malloc(sizeof(PNode) * (size_t)(2 * nf));
    b->order = (int32_t*)malloc(sizeof(int32_t) * (size_t)nf);
    double* lo = (double*)malloc(sizeof(double) * 3 * (size_t)nf);
    double* hi = (double*)malloc(sizeof(double) * 3 * (size_t)nf);
    g_cent = (double*)malloc(sizeof(double) * 3 * (size_t)nf);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < nf; ++i) { tri_box(&b->mesh, (int32_t)i, lo + 3 * i, hi + 3 * i, g_cent + 3 * i); b->order[i] = (int32_t)i; }
    pbuild(b, lo, hi, 0, (int32_t)nf);
    free(lo); free(hi); free(g_cent); g_cent = NULL;
    return b;
}

void point_bvh_free(void* p) {
    PBvh* b = (PBvh*)p;
    if (!b) return;
    free(b->nodes); free(b->order); free(b);
}

/* squared distance from p to the node box widened by 1e-5 of the magnitude of box and point, times (1 - 1e-6) */
static double box_lb(const PNode* n, const double p[3]) {
    double s = 0.0;
    for (int a = 0; a < 3; ++a) {
        const double mag = fabs(n->lo[a]) + fabs(n->hi[a]) + fabs(p[a]);
        const double pad = 1e-5 * mag + 1e-37;
        double g = 0.0;
        if (p[a] < n->lo[a] - pad) g = n->lo[a] - pad - p[a];
        else if (p[a] > n->hi[a] + pad) g = p[a] - n->hi[a] - pad;
        s += g * g;
    }
    return s * (1.0 - 1e-6);
}

typedef struct { double best; int32_t prim; } Best;

static void visit(const PMesh* m, int mode, const double pd[3], const float pf[3], int32_t t, Best* b) {
    const float *v0 = pvert(m, t, 0), *v1 = pvert(m, t, 1), *v2 = pvert(m, t, 2);
    double d2;
    if (mode == 1) {
        float out[6];
        f_point_tri(pf, v0, v1, v2, out);
        d2 = (double)out[3];
    } else {
        const double a[3] = {v0[0], v0[1], v0[2]}, bb[3] = {v1[0], v1[1], v1[2]}, c[3] = {v2[0], v2[1], v2[2]};
        double out[6];
        d_point_tri(pd, a, bb, c, out);
        d2 = out[3];
    }
    if (d2 < b->best || (d2 == b->best && t < b->prim)) { b->best = d2; b->prim = t; }
}

/* mode 0 truth / 1 mirror; bvh from point_bvh_build or NULL (brute force).  Outputs per point (any may be NULL):
 * closest[3], distance, tri (-1 = none), uv[2], d2 (+inf = none); double arrays hold binary32 values exactly in mode 1. */
int point_query(const float* verts, int64_t nv, const int32_t* faces, int64_t nf, void* bvh_handle, int mode, int64_t n,
                const float* points, double max_distance, double* closest, double* distance, int32_t* tri, double* uv,
                double* d2_out) {
    PMesh mesh; mesh.verts = verts; mesh.faces = faces; mesh.nv = nv; mesh.nf = nf;
    const PBvh* bvh = (const PBvh*)bvh_handle;
    const float mf = (float)max_distance;
    const double max_d2 = mode == 1 ? (double)(mf * mf) : max_distance * max_distance;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < n; ++i) {
        const float pf[3] = {points[3 * i], points[3 * i + 1], points[3 * i + 2]};
        const double pd[3] = {pf[0], pf[1], pf[2]};
        Best b; b.best = max_d2; b.prim = INT32_MAX;
        const int finite = isfinite(pf[0]) && isfinite(pf[1]) && isfinite(pf[2]);
        if (finite && nf > 0) {
            if (!bvh) {
                for (int64_t t = 0; t < nf; ++t) visit(&mesh, mode, pd, pf, (int32_t)t, &b);
            } else {
                int32_t stack[256];
                int sp = 0;
                stack[sp++] = 0;
                while (sp > 0) {
                    const PNode* nd = &bvh->nodes[stack[--sp]];
                    if (box_lb(nd, pd) > b.best) continue;
                    if (nd->left < 0) {
                        for (int32_t k = 0; k < nd->count; ++k) visit(&mesh, mode, pd, pf, bvh->order[nd->first + k], &b);
                        continue;
                    }
                    const double ll = box_lb(&bvh->nodes[nd->left], pd), lr = box_lb(&bvh->nodes[nd->right], pd);
                    if (ll <= lr) { stack[sp++] = nd->right; stack[sp++] = nd->left; }
                    else { stack[sp++] = nd->left; stack[sp++] = nd->right; }
                }
            }
        }
        const int found = b.prim != INT32_MAX;
        double q[6] = {0, 0, 0, INFINITY, 0, 0};
        double dist = INFINITY;
        if (found) {
            const float *v0 = pvert(&mesh, b.prim, 0), *v1 = pvert(&mesh, b.prim, 1), *v2 = pvert(&mesh, b.prim, 2);
            if (mode == 1) {
                float out[6];
                f_point_tri(pf, v0, v1, v2, out);
                for (int k = 0; k < 6; ++k) q[k] = out[k];
                dist = (double)sqrtf(out[3]);
            } else {
                const double a[3] = {v0[0], v0[1], v0[2]}, bb[3] = {v1[0], v1[1], v1[2]}, c[3] = {v2[0], v2[1], v2[2]};
                d_point_tri(pd, a, bb, c, q);
                dist = sqrt(q[3]);
            }
        }
        if (closest) { closest[3 * i] = q[0]; closest[3 * i + 1] = q[1]; closest[3 * i + 2] = q[2]; }
        if (distance) distance[i] = dist;
        if (tri) tri[i] = found ? b.prim : -1;
        if (uv) { uv[2 * i] = q[4]; uv[2 * i + 1] = q[5]; }
        if (d2_out) d2_out[i] = q[3];
    }
    return 0;
}

/* d2 of every (point, triangle) pair, binary32 mirror or binary64 truth: [n, nf] row-major */
void point_all_d2(const float* verts, int64_t nv, const int32_t* faces, int64_t nf, int mode, int64_t n, const float* points,
                  double* out) {
    PMesh mesh; mesh.verts = verts; mesh.faces = faces; mesh.nv = nv; mesh.nf = nf;
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        const float pf[3] = {points[3 * i], points[3 * i + 1], points[3 * i + 2]};
        const double pd[3] = {pf[0], pf[1], pf[2]};
        for (int64_t t = 0; t < nf; ++t) {
            const float *v0 = pvert(&mesh, t, 0), *v1 = pvert(&mesh, t, 1), *v2 = pvert(&mesh, t, 2);
            if (mode == 1) {
                float o[6];
                f_point_tri(pf, v0, v1, v2, o);
                out[i * nf + t] = o[3];
            } else {
                const double a[3] = {v0[0], v0[1], v0[2]}, bb[3] = {v1[0], v1[1], v1[2]}, c[3] = {v2[0], v2[1], v2[2]};
                double o[6];
                d_point_tri(pd, a, bb, c, o);
                out[i * nf + t] = o[3];
            }
        }
    }
}

int point_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
