// rt_scene.cuh — arithmetic of instanced scenes (rt_scene.cu): the per-instance preparation (binary64 inverse, world
// box, padding) and the two-level walk (a top-level BVH8 over instance boxes, each instance's own BVH8 below it).
//
// Everything here is RT_HD and a pure function of its arguments, so the host simulator under tests/scene/ runs the
// same code (DESIGN.md §4.11).  The top-level tree is an ordinary blob from rt_bvh_build: instance i is the "triangle"
// (lo_i, hi_i, lo_i) whose box is exactly the padded world box [lo_i, hi_i], and its record's prim is i.
#pragma once
#include "../../include/raymesh_b200.h"
#include "rt_pseudonormal.cuh"

namespace rt {

#if defined(__CUDA_ARCH__)
RT_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
RT_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
RT_HD double dsqrt(double a) { return __dsqrt_rn(a); }
#else
RT_HD double dadd(double a, double b) { return a + b; }
RT_HD double ddiv(double a, double b) { return a / b; }
RT_HD double dsqrt(double a) { return sqrt(a); }
#endif

// Scene table (one device buffer): [SceneHeader][instance records, 128 B each][BLAS blob addresses, 8 B each].
struct alignas(16) SceneHeader {
    uint64_t n_meshes, n_inst, inst_offset, blobs_offset;
    uint64_t reserved[4];
};
static_assert(sizeof(SceneHeader) == 64, "SceneHeader must be 64 bytes");

constexpr uint32_t kInstMirrored = 1u;   // det(A) < 0: facing flips
constexpr uint32_t kInstEmpty = 2u;      // the mesh has no triangle with a finite box: never visited

// Instance record.  fwd = (A | b) row-major 3x4 as given; inv = (A^-1 | c), c = -A^-1 b, both computed in binary64
// and rounded to binary32 once; zero offsets are stored as -0, the identity of binary32 addition (affine_row).
struct alignas(16) SceneInst {
    float fwd[12];
    float inv[12];
    int32_t mesh;
    uint32_t flags;
    float lo[3], hi[3];          // the padded world box, as the top-level record holds it
};
static_assert(sizeof(SceneInst) == 128, "SceneInst must be 128 bytes");

// Row k of an affine map applied to (x, y, z): ffma(m0, x, ffma(m1, y, ffma(m2, z, c))) with every term of a zero
// coefficient left out.  With the identity (1, 0, 0, -0) the result is x itself, bit for bit, including -0, infinities
// and NaN: one identity instance reproduces the single-mesh traversal exactly (ray_inverse reads the sign of -0).
RT_HD float affine_row(float m0, float m1, float m2, float c, float x, float y, float z) {
    float acc = c;
    acc = m2 != 0.0f ? ffma(m2, z, acc) : acc;
    acc = m1 != 0.0f ? ffma(m1, y, acc) : acc;
    acc = m0 != 0.0f ? ffma(m0, x, acc) : acc;
    return acc;
}

// World ray -> object ray of an instance (the ray parameter t is the same in both spaces).
RT_HD void object_ray(const SceneInst& s, float ox, float oy, float oz, float dx, float dy, float dz, float o[3],
                      float d[3]) {
    const float nz = as_float(0x80000000u);
    for (int k = 0; k < 3; ++k) {
        const float* m = s.inv + 4 * k;
        o[k] = affine_row(m[0], m[1], m[2], m[3], ox, oy, oz);
        d[k] = affine_row(m[0], m[1], m[2], nz, dx, dy, dz);
    }
}

// ---------------------------------------------------------------- preparation (binary64)
RT_HD double det3(const double a[9]) {
    const double c0 = dsub(dmul(a[4], a[8]), dmul(a[5], a[7]));
    const double c1 = dsub(dmul(a[3], a[8]), dmul(a[5], a[6]));
    const double c2 = dsub(dmul(a[3], a[7]), dmul(a[4], a[6]));
    return dadd(dsub(dmul(a[0], c0), dmul(a[1], c1)), dmul(a[2], c2));
}

RT_HD float round_down(double x) { const float f = (float)x; return (double)f > x ? nextafterf(f, -INFINITY) : f; }
RT_HD float round_up(double x) { const float f = (float)x; return (double)f < x ? nextafterf(f, INFINITY) : f; }
RT_HD float zero_as_negative(float x) { return x == 0.0f ? as_float(0x80000000u) : x; }
RT_HD bool finite_f(float x) { return x == x && fabsf(x) <= 3.4028235e38f; }

// Inverse (A^-1 | -A^-1 b) of a binary32 3x4 transform in binary64, rounded to binary32; *kappa = ||A||inf ||A^-1||inf
// in binary64.  false: the transform is not finite, det(A) is 0, or the rounded inverse is not finite.
RT_HD bool invert_transform(const float fwd[12], float inv[12], double* det_out, double* kappa) {
    double a[9], b[3];
    bool ok = true;
    for (int k = 0; k < 3; ++k) {
        for (int j = 0; j < 3; ++j) { a[3 * k + j] = (double)fwd[4 * k + j]; ok = ok && finite_f(fwd[4 * k + j]); }
        b[k] = (double)fwd[4 * k + 3];
        ok = ok && finite_f(fwd[4 * k + 3]);
    }
    const double det = det3(a);
    *det_out = det;
    if (!ok || !(det != 0.0)) return false;
    double m[9];
    m[0] = ddiv(dsub(dmul(a[4], a[8]), dmul(a[5], a[7])), det);
    m[1] = ddiv(dsub(dmul(a[2], a[7]), dmul(a[1], a[8])), det);
    m[2] = ddiv(dsub(dmul(a[1], a[5]), dmul(a[2], a[4])), det);
    m[3] = ddiv(dsub(dmul(a[5], a[6]), dmul(a[3], a[8])), det);
    m[4] = ddiv(dsub(dmul(a[0], a[8]), dmul(a[2], a[6])), det);
    m[5] = ddiv(dsub(dmul(a[2], a[3]), dmul(a[0], a[5])), det);
    m[6] = ddiv(dsub(dmul(a[3], a[7]), dmul(a[4], a[6])), det);
    m[7] = ddiv(dsub(dmul(a[1], a[6]), dmul(a[0], a[7])), det);
    m[8] = ddiv(dsub(dmul(a[0], a[4]), dmul(a[1], a[3])), det);
    double na = 0.0, nm = 0.0;
    for (int k = 0; k < 3; ++k) {
        const double c = dsub(0.0, dadd(dadd(dmul(m[3 * k], b[0]), dmul(m[3 * k + 1], b[1])), dmul(m[3 * k + 2], b[2])));
        for (int j = 0; j < 3; ++j) inv[4 * k + j] = (float)m[3 * k + j];
        inv[4 * k + 3] = zero_as_negative((float)c);
        const double ra = dadd(dadd(fabs(a[3 * k]), fabs(a[3 * k + 1])), fabs(a[3 * k + 2]));
        const double rm = dadd(dadd(fabs(m[3 * k]), fabs(m[3 * k + 1])), fabs(m[3 * k + 2]));
        na = ra > na ? ra : na;
        nm = rm > nm ? rm : nm;
        for (int j = 0; j < 4; ++j) ok = ok && finite_f(inv[4 * k + j]);
    }
    *kappa = dmul(na, nm);
    return ok;
}

// Padding of the world boxes relative to kappa * S, S = ||b||inf + ||A||inf * R (R = largest |coordinate| of the
// mesh's box): DESIGN.md §4.11 derives it and the condition ||o||inf <= 32 S under which no hit is culled.
constexpr double kScenePad = 1.0 / 16384.0;

// Fills everything of one instance record but fwd and mesh (which the caller sets) from the mesh blob's header, and
// writes its top-level vertices v[6] = (lo, hi) and face f[3] = (2i, 2i+1, 2i).  The transform must have passed
// invert_transform (the entry point checks it on the host before the launch).
RT_HD void prepare_instance(const uint8_t* blob, SceneInst& s, uint32_t i, float* v, int32_t* f) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    double det = 0.0, kappa = 0.0;
    invert_transform(s.fwd, s.inv, &det, &kappa);
    const float* blo = h->aabb_lo;
    const float* bhi = h->aabb_hi;
    bool empty = h->n_tris == 0u;
    double R = 0.0;
    for (int a = 0; a < 3; ++a) {
        empty = empty || !(blo[a] <= bhi[a]) || !finite_f(blo[a]) || !finite_f(bhi[a]);
        const double m = fabs((double)blo[a]) > fabs((double)bhi[a]) ? fabs((double)blo[a]) : fabs((double)bhi[a]);
        R = m > R ? m : R;
    }
    s.flags = (det < 0.0 ? kInstMirrored : 0u) | (empty ? kInstEmpty : 0u);
    if (empty) {   // a point box at the instance's origin: the record exists, the walk never enters it
        for (int a = 0; a < 3; ++a) { s.lo[a] = s.fwd[4 * a + 3]; s.hi[a] = s.fwd[4 * a + 3]; }
    } else {
        double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        double na = 0.0, nb = 0.0;
        for (int k = 0; k < 3; ++k) {
            const double ra = dadd(dadd(fabs((double)s.fwd[4 * k]), fabs((double)s.fwd[4 * k + 1])), fabs((double)s.fwd[4 * k + 2]));
            na = ra > na ? ra : na;
            const double bk = fabs((double)s.fwd[4 * k + 3]);
            nb = bk > nb ? bk : nb;
        }
        for (int c = 0; c < 8; ++c) {
            const double p[3] = {(double)((c & 1) ? bhi[0] : blo[0]), (double)((c & 2) ? bhi[1] : blo[1]),
                                 (double)((c & 4) ? bhi[2] : blo[2])};
            for (int k = 0; k < 3; ++k) {
                const double w = dadd(dadd(dadd(dmul((double)s.fwd[4 * k], p[0]), dmul((double)s.fwd[4 * k + 1], p[1])),
                                           dmul((double)s.fwd[4 * k + 2], p[2])), (double)s.fwd[4 * k + 3]);
                lo[k] = w < lo[k] ? w : lo[k];
                hi[k] = w > hi[k] ? w : hi[k];
            }
        }
        const double pad = dmul(dmul(kScenePad, kappa), dadd(nb, dmul(na, R)));
        for (int k = 0; k < 3; ++k) { s.lo[k] = round_down(dsub(lo[k], pad)); s.hi[k] = round_up(dadd(hi[k], pad)); }
    }
    for (int a = 0; a < 3; ++a) { v[a] = s.lo[a]; v[3 + a] = s.hi[a]; }
    f[0] = (int32_t)(2u * i); f[1] = (int32_t)(2u * i + 1u); f[2] = (int32_t)(2u * i);
}

// ---------------------------------------------------------------- trace
// Slab test of a record's exact box [lo, hi] against (0, tmax), widened by 2^-20 relative per plane (the two roundings
// of (p - o) * idir are below 2^-23 relative), inclusive at both ends.  Infinite plane distances stay infinite; a NaN
// drops out of fminf/fmaxf, which only widens.
RT_HD bool box_hit(const Ray& r, const float lo[3], const float hi[3], float tmax) {
    const float kn = 1.0f - 9.5367432e-7f, kf = 1.0f + 9.5367432e-7f;
    float tn = 0.0f, tf = tmax;
    const float o[3] = {r.ox, r.oy, r.oz}, id[3] = {r.idx, r.idy, r.idz};
    for (int a = 0; a < 3; ++a) {
        const float t0 = fmul(fsub(lo[a], o[a]), id[a]), t1 = fmul(fsub(hi[a], o[a]), id[a]);
        float n = fminf(t0, t1), f = fmaxf(t0, t1);
        n = fmul(n, n > 0.0f ? kn : kf);
        f = fmul(f, f > 0.0f ? kf : kn);
        tn = fmaxf(tn, n);
        tf = fminf(tf, f);
    }
    return tn <= tf;
}

// Element offset of row r of a [*b, 3] batch flattened to shape[0..2] with element strides stride[0..2].
RT_HD int64_t scene_offset(const int64_t shape[4], const int64_t stride[4], int64_t r) {
    const int64_t i2 = r % shape[2];
    const int64_t q = r / shape[2];
    const int64_t i1 = q % shape[1];
    const int64_t i0 = q / shape[1];
    return i0 * stride[0] + i1 * stride[1] + i2 * stride[2];
}

struct SceneView {
    const SceneInst* inst;
    const uint64_t* blobs;      // BLAS blob address of each mesh
};
RT_HD SceneView scene_view(const uint8_t* table) {
    const SceneHeader* h = reinterpret_cast<const SceneHeader*>(table);
    SceneView v;
    v.inst = reinterpret_cast<const SceneInst*>(table + h->inst_offset);
    v.blobs = reinterpret_cast<const uint64_t*>(table + h->blobs_offset);
    return v;
}

// The object ray of instance i and its mesh's node and record arrays; false for an instance of an empty mesh.
RT_HD bool instance_ray(const SceneView& sv, int32_t i, const float w[6], Ray& r, const uint8_t*& nodes,
                        const uint8_t*& tris) {
    const SceneInst& s = sv.inst[i];
    if (s.flags & kInstEmpty) return false;
    const uint8_t* blob = reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]);
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    nodes = blob + h->nodes_offset;
    tris = blob + h->tris_offset;
    float o[3], d[3];
    object_ray(s, w[0], w[1], w[2], w[3], w[4], w[5], o, d);
    ray_setup(r, o[0], o[1], o[2], d[0], d[1], d[2]);
    return true;
}

// Closest hit over the instances: the minimum of the key (t, inst, prim) in (0, tmax).  Instance i's walk starts with
// the best t so far and a tie rule that extends ClosestVisitor's: when i precedes the best instance an equal t wins
// (seed prim INT32_MAX), otherwise it loses (seed -1), so the answer does not depend on the visiting order.
template <class StackT>
struct SceneClosest {
    SceneView sv;
    float w[6];
    float tmax;
    int32_t inst = -1, prim = -1;
    uint32_t slot = 0;
    StackT* stack;
    RT_HD bool visit(int32_t i) {
        Ray r;
        const uint8_t *nodes, *tris;
        if (!instance_ray(sv, i, w, r, nodes, tris)) return false;
        const int32_t seed = (inst >= 0 && i < inst) ? 0x7fffffff : -1;
        ClosestVisitor<NoStats> vis(tmax);
        vis.prim = seed;
        traverse(nodes, tris, r, vis, *stack);
        if (vis.prim != seed) { tmax = vis.tmax; inst = i; prim = vis.prim; slot = vis.slot; }
        return false;
    }
};

template <class StackT>
struct SceneAny {
    SceneView sv;
    float w[6];
    float tmax;
    bool found = false;
    StackT* stack;
    RT_HD bool visit(int32_t i) {
        Ray r;
        const uint8_t *nodes, *tris;
        if (!instance_ray(sv, i, w, r, nodes, tris)) return false;
        AnyVisitor<NoStats> vis(tmax);
        traverse(nodes, tris, r, vis, *stack);
        found = vis.found;
        return found;
    }
};

template <class StackT>
struct SceneCount {
    SceneView sv;
    float w[6];
    float tmax;
    int32_t count = 0;
    StackT* stack;
    RT_HD bool visit(int32_t i) {
        Ray r;
        const uint8_t *nodes, *tris;
        if (!instance_ray(sv, i, w, r, nodes, tris)) return false;
        CountVisitor<NoStats> vis(tmax);
        traverse(nodes, tris, r, vis, *stack);
        count += vis.count;
        return false;
    }
};

// One step of the top-level walk: trav_step's node handling, but a leaf record is an instance.  Its exact box is
// tested first (box_hit), then `vis.visit(inst)` walks the instance's own tree.  Returns true when the ray is finished.
template <class Visitor, class StackT>
RT_HD bool scene_step(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ recs, const Ray& r, Visitor& vis,
                      StackT& stack, Trav& t) {
    if (t.gy & 0xff000000u) {
        const uint32_t hits = t.gy;
        const int bit = 31 - clz32(hits);
        t.gy &= ~(1u << bit);
        if (t.gy & 0xff000000u) { stack.push(t.sp, t.gx, t.gy); ++t.sp; }
        const uint32_t slot = (uint32_t)(bit - 24) ^ r.octinv;
        const uint32_t rel = (uint32_t)popc32(hits & ~(0xffffffffu << slot));
        const uint8_t* np = nodes + (size_t)(t.gx + rel) * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48), n4 = ldg128(np + 64);
        const uint32_t hm = node_test(r, n0, n1, n2, n3, n4, 0.0f, vis.tmax);
        t.gx = n1.x;
        t.gy = (hm & 0xff000000u) | (n0.w >> 24);
        uint32_t ty = hm & 0x00ffffffu;
        const uint32_t tx = n1.y, tmask = n1.z;
        while (ty) {
            const int b = ffs32(ty) - 1;
            ty &= ty - 1u;
            const uint32_t slot_t = tx + (uint32_t)popc32(tmask & ~(0xffffffffu << b));
            const uint8_t* tp = recs + (size_t)slot_t * 48u;
            const U4 a = ldg128(tp), bb = ldg128(tp + 16);
            const float lo[3] = {as_float(a.x), as_float(a.y), as_float(a.z)};
            const float hi[3] = {as_float(bb.x), as_float(bb.y), as_float(bb.z)};
            if (box_hit(r, lo, hi, vis.tmax) && vis.visit((int32_t)a.w)) return true;
        }
    }
    if (!(t.gy & 0xff000000u)) {
        if (t.sp == 0) return true;
        --t.sp;
        stack.pop(t.sp, t.gx, t.gy);
    }
    return false;
}

// Closest-hit outputs of instance `inst`, triangle record `slot`: uv in object space, loc = A loc_obj + b (affine_row
// with b, zero offsets as -0), front = object-space front XOR mirrored.
struct SceneHitOut { bool front; float loc[3]; float uv[2]; };
RT_HD SceneHitOut scene_hit_attr(const SceneView& sv, int32_t inst, uint32_t slot, const float w[6]) {
    Ray r;
    const uint8_t *nodes, *tris;
    instance_ray(sv, inst, w, r, nodes, tris);
    const SceneInst& s = sv.inst[inst];
    const uint8_t* tp = tris + (size_t)slot * 48u;
    const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
    const float v0x = as_float(a.x), v0y = as_float(a.y), v0z = as_float(a.z);
    const float v1x = as_float(b.x), v1y = as_float(b.y), v1z = as_float(b.z);
    const float v2x = as_float(c.x), v2y = as_float(c.y), v2z = as_float(c.z);
    TriHit h;
    tri_test(r, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z, h);
    const HitAttr at = tri_attr(h, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z);
    SceneHitOut out;
    out.front = tri_front(r, h) != ((s.flags & kInstMirrored) != 0u);
    for (int k = 0; k < 3; ++k) {
        const float* m = s.fwd + 4 * k;
        out.loc[k] = affine_row(m[0], m[1], m[2], zero_as_negative(m[3]), at.lx, at.ly, at.lz);
    }
    out.uv[0] = at.uv0;
    out.uv[1] = at.uv1;
    return out;
}

// ---------------------------------------------------------------- point queries (DESIGN.md §4.12)
// Closest point and pseudo-normal signed distance over the instances: the minimum of the key (d2, inst, prim) over
// every non-empty instance and triangle with d2 <= max_d2, d2 = point_tri(p, W0, W1, W2).d2 of the WORLD triangle
// Wk = affine_row(fwd row, zero_as_negative(b), vk).  That is exactly the key (d2, f) of the mesh flattened with the
// same affine_row, faces concatenated in instance order, so the answer equals rt_closest_point on that mesh.

// Side array of the point queries, one entry per instance (rt_scene_point_prepare): sigma <= the smallest singular
// value of A, and the world margin mu(p) = alpha + beta |p|inf of the instance walk's bound (scene_world_bound).
struct alignas(16) ScenePointSide { float sigma, alpha, beta, reserved; };
static_assert(sizeof(ScenePointSide) == 16, "ScenePointSide must be 16 bytes");

// A rigorous lower bound on the smallest eigenvalue of the symmetric 3x3 matrix g (binary64, row-major): eight cyclic
// Jacobi sweeps, then Gershgorin's lower end on the rotated matrix, less a Weyl margin of 2^-40 * `scale` for the
// rounding of the rotations (backward stable: each is an exact orthogonal similarity of a matrix within a few
// 2^-53 ||g|| of the computed one).  `scale` >= ||g||F.  Every operation is fixed, so the host repeats the bits.
RT_HD double sym3_min_eig_lower(const double g_in[9], double scale) {
    double g[9];
    for (int k = 0; k < 9; ++k) g[k] = g_in[k];
    for (int sweep = 0; sweep < 8; ++sweep) {
        for (int pr = 0; pr < 3; ++pr) {
            const int p = pr == 2 ? 1 : 0, q = pr == 0 ? 1 : 2, r = 3 - p - q;
            const double apq = g[3 * p + q];
            if (apq == 0.0) continue;
            const double theta = ddiv(dsub(g[3 * q + q], g[3 * p + p]), dmul(2.0, apq));
            const double t0 = ddiv(1.0, dadd(fabs(theta), dsqrt(dadd(dmul(theta, theta), 1.0))));
            const double t = theta < 0.0 ? -t0 : t0;
            const double c = ddiv(1.0, dsqrt(dadd(dmul(t, t), 1.0)));
            const double sn = dmul(t, c);
            const double arp = g[3 * r + p], arq = g[3 * r + q];
            g[3 * p + p] = dsub(g[3 * p + p], dmul(t, apq));
            g[3 * q + q] = dadd(g[3 * q + q], dmul(t, apq));
            g[3 * p + q] = g[3 * q + p] = 0.0;
            g[3 * r + p] = g[3 * p + r] = dsub(dmul(c, arp), dmul(sn, arq));
            g[3 * r + q] = g[3 * q + r] = dadd(dmul(sn, arp), dmul(c, arq));
        }
    }
    double lo = INFINITY;
    for (int k = 0; k < 3; ++k) {
        const double off = dadd(fabs(g[3 * k + (k + 1) % 3]), fabs(g[3 * k + (k + 2) % 3]));
        const double e = dsub(g[4 * k], off);
        lo = e < lo ? e : lo;
    }
    return dsub(lo, dmul(9.094947017729282e-13, scale));   // 2^-40
}

// The side entry of one instance, from its record and its mesh's header box (binary64, rounded once).  With u = 2^-24,
// M | c the stored inverse, E = A M - I and g = A c + b (both from binary32 values, so their binary64 residuals are
// bounded below), S = ||b||inf + ||A||inf R as in prepare_instance:
//   alpha = sigma 2^-21 ||c||inf + 1.75 ||g||inf + 2^-18 S,   beta = sigma 2^-21 ||M||inf + 1.75 ||E||inf,
// each inflated by 2^-16 and rounded up; DESIGN.md §4.12 derives them.  An empty instance gets zeros (never read).
RT_HD ScenePointSide prepare_point_side(const uint8_t* blob, const SceneInst& s) {
    ScenePointSide out = {0.0f, 0.0f, 0.0f, 0.0f};
    if (s.flags & kInstEmpty) return out;
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    double R = 0.0;
    for (int a = 0; a < 3; ++a) {
        const double lo = fabs((double)h->aabb_lo[a]), hi = fabs((double)h->aabb_hi[a]);
        const double m = lo > hi ? lo : hi;
        R = m > R ? m : R;
    }
    double g[9], fro = 0.0, na = 0.0, nb = 0.0, nm = 0.0, nc = 0.0, ne = 0.0, ng = 0.0;
    const double ulp53 = 1.1102230246251565e-16;   // 2^-53
    for (int k = 0; k < 3; ++k) {
        double ra = 0.0, rm = 0.0, re = 0.0;
        for (int j = 0; j < 3; ++j) {
            double gkj = 0.0, ekj = 0.0, abs_e = 0.0;
            for (int l = 0; l < 3; ++l) {
                gkj = dadd(gkj, dmul((double)s.fwd[4 * l + k], (double)s.fwd[4 * l + j]));
                ekj = dadd(ekj, dmul((double)s.fwd[4 * k + l], (double)s.inv[4 * l + j]));
                abs_e = dadd(abs_e, fabs(dmul((double)s.fwd[4 * k + l], (double)s.inv[4 * l + j])));
            }
            g[3 * k + j] = gkj;
            ekj = dsub(ekj, k == j ? 1.0 : 0.0);
            re = dadd(re, dadd(fabs(ekj), dmul(4.0 * ulp53, dadd(abs_e, 1.0))));
            ra = dadd(ra, fabs((double)s.fwd[4 * k + j]));
            rm = dadd(rm, fabs((double)s.inv[4 * k + j]));
            fro = dadd(fro, dmul((double)s.fwd[4 * k + j], (double)s.fwd[4 * k + j]));
        }
        double gk = (double)s.fwd[4 * k + 3], abs_g = fabs((double)s.fwd[4 * k + 3]);
        for (int l = 0; l < 3; ++l) {
            gk = dadd(gk, dmul((double)s.fwd[4 * k + l], (double)s.inv[4 * l + 3]));
            abs_g = dadd(abs_g, fabs(dmul((double)s.fwd[4 * k + l], (double)s.inv[4 * l + 3])));
        }
        const double gb = dadd(fabs(gk), dmul(4.0 * ulp53, abs_g));
        na = ra > na ? ra : na;
        nm = rm > nm ? rm : nm;
        ne = re > ne ? re : ne;
        ng = gb > ng ? gb : ng;
        const double bk = fabs((double)s.fwd[4 * k + 3]), ck = fabs((double)s.inv[4 * k + 3]);
        nb = bk > nb ? bk : nb;
        nc = ck > nc ? ck : nc;
    }
    const double lam = sym3_min_eig_lower(g, fro);
    const double sigma = lam > 0.0 ? dmul(dsqrt(lam), 1.0 - 3.552713678800501e-15) : 0.0;   // 1 - 2^-48
    out.sigma = round_down(sigma);
    const double sd = (double)out.sigma, k21 = 4.76837158203125e-07, k18 = 3.814697265625e-06, inf16 = 1.0 + 1.52587890625e-05;
    const double S = dadd(nb, dmul(na, R));
    const double alpha = dadd(dadd(dmul(dmul(sd, k21), nc), dmul(1.75, ng)), dmul(k18, S));
    const double beta = dadd(dmul(dmul(sd, k21), nm), dmul(1.75, ne));
    out.alpha = round_up(dmul(alpha, inf16));
    out.beta = round_up(dmul(beta, inf16));
    return out;
}

// Squared distance from (x, y, z) to the box [lo, hi], rounded so that it never exceeds the exact value times 1 - 5u
// (the factor 1 - 2^-20 covers the roundings of the gaps and the sum): the top-level leaf bound.
RT_HD float box_point_lower(float x, float y, float z, const float lo[3], const float hi[3]) {
    const float gx = fmaxf(fmaxf(fsub(lo[0], x), fsub(x, hi[0])), 0.0f);
    const float gy = fmaxf(fmaxf(fsub(lo[1], y), fsub(y, hi[1])), 0.0f);
    const float gz = fmaxf(fmaxf(fsub(lo[2], z), fsub(z, hi[2])), 0.0f);
    return fmul(dot3f(gx, gy, gz, gx, gy, gz), 0.999999046325684f);   // 1 - 2^-20
}

// World vertices of an object-space triangle record: Wk = affine_row(fwd row, zero_as_negative(b), vk).
RT_HD void world_tri(const float fwd[12], const U4& a, const U4& b, const U4& c, float w[9]) {
    const float v[9] = {as_float(a.x), as_float(a.y), as_float(a.z), as_float(b.x), as_float(b.y), as_float(b.z),
                        as_float(c.x), as_float(c.y), as_float(c.z)};
    for (int k = 0; k < 3; ++k) {
        const float* m = fwd + 4 * k;
        const float bk = zero_as_negative(m[3]);
        for (int j = 0; j < 3; ++j) w[3 * j + k] = affine_row(m[0], m[1], m[2], bk, v[3 * j], v[3 * j + 1], v[3 * j + 2]);
    }
}

// World lower bound of an instance-walk slot from its object-space bound lb = slot_lower_bounds(p'):
// (sigma sqrt(lb) - mu)+^2 (1 - 2^-20) <= the d2 point_tri computes for every world triangle below the slot.
RT_HD float scene_world_bound(float lb, float sigma, float mu) {
    const float h = fmaxf(fsub(fmul(sigma, fsqrt(lb)), mu), 0.0f);
    return fmul(fmul(h, h), 0.999999046325684f);
}

// The walk of one instance's own tree: slot bounds from the object point p' mapped to world bounds, leaves tested as
// world triangles against the world point (t.x, t.y, t.z).
struct InstanceSpace {
    float fwd[12];
    float ox, oy, oz;          // p' = affine_row(inv rows, p)
    float sigma, mu;
    RT_HD void bounds(const PointTrav& t, const U4& n0, const U4& n2, const U4& n3, const U4& n4, float lb[8]) const {
        (void)t;
        slot_lower_bounds(ox, oy, oz, n0, n2, n3, n4, lb);
#pragma unroll
        for (int s = 0; s < 8; ++s) lb[s] = scene_world_bound(lb[s], sigma, mu);
    }
    RT_HD void leaf(PointTrav& t, uint32_t rec, const U4& a, const U4& b, const U4& c) const {
        float w[9];
        world_tri(fwd, a, b, c, w);
        const PointHit h = point_tri(t.x, t.y, t.z, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w[8]);
        const int32_t prim = (int32_t)a.w;
        if (h.d2 < t.best || (h.d2 == t.best && prim < t.prim)) { t.best = h.d2; t.prim = prim; t.slot = rec; }
    }
};

// Walks instance i with the world best t.best.  The seed extends the single-mesh tie rule to (d2, inst, prim): when
// no instance has an answer yet or i precedes the best one an equal d2 wins (seed kNoPrim), otherwise it loses
// (seed -1).  Returns the prim found, or the seed when nothing beat the best; lowers t.best and sets *slot on a find.
template <class StackT>
RT_HD int32_t scene_point_instance(const SceneView& sv, const ScenePointSide* side, int32_t i, int32_t best_inst,
                                   PointTrav& t, uint32_t* slot, StackT& stack) {
    const int32_t seed = (best_inst < 0 || i < best_inst) ? kNoPrim : -1;
    const SceneInst& s = sv.inst[i];
    if (s.flags & kInstEmpty) return seed;
    const uint8_t* blob = reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]);
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    InstanceSpace sp;
    for (int k = 0; k < 12; ++k) sp.fwd[k] = s.fwd[k];
    sp.ox = affine_row(s.inv[0], s.inv[1], s.inv[2], s.inv[3], t.x, t.y, t.z);
    sp.oy = affine_row(s.inv[4], s.inv[5], s.inv[6], s.inv[7], t.x, t.y, t.z);
    sp.oz = affine_row(s.inv[8], s.inv[9], s.inv[10], s.inv[11], t.x, t.y, t.z);
    const ScenePointSide e = side[i];
    const float pmax = fmaxf(fmaxf(fabsf(t.x), fabsf(t.y)), fabsf(t.z));
    sp.sigma = e.sigma;
    sp.mu = fadd(e.alpha, fmul(e.beta, pmax));
    PointTrav it;
    it.x = t.x; it.y = t.y; it.z = t.z; it.best = t.best; it.prim = seed; it.slot = 0u; it.node = 0u; it.sp = 0;
    NoStats st;
    while (!point_step(blob + h->nodes_offset, blob + h->tris_offset, it, st, stack, sp)) {}
    if (it.prim != seed) { t.best = it.best; *slot = it.slot; }
    return it.prim;
}

// The top-level walk: world slot bounds (the slot boxes contain the padded instance boxes), and a leaf record is an
// instance, entered when the squared distance to its padded world box is within the best.
template <class StackT>
struct SceneTopSpace {
    SceneView sv;
    const ScenePointSide* side;
    StackT* stack;
    int32_t inst = -1, prim = -1;
    uint32_t slot = 0;
    RT_HD void bounds(const PointTrav& t, const U4& n0, const U4& n2, const U4& n3, const U4& n4, float lb[8]) const {
        slot_lower_bounds(t.x, t.y, t.z, n0, n2, n3, n4, lb);
    }
    RT_HD void leaf(PointTrav& t, uint32_t rec, const U4& a, const U4& b, const U4& c) {
        (void)rec; (void)c;
        const float lo[3] = {as_float(a.x), as_float(a.y), as_float(a.z)};
        const float hi[3] = {as_float(b.x), as_float(b.y), as_float(b.z)};
        if (!(box_point_lower(t.x, t.y, t.z, lo, hi) <= t.best)) return;
        visit(t, (int32_t)a.w);
    }
    RT_HD void visit(PointTrav& t, int32_t i) {
        uint32_t sl = 0u;
        const int32_t seed = (inst < 0 || i < inst) ? kNoPrim : -1;
        const int32_t pr = scene_point_instance(sv, side, i, inst, t, &sl, *stack);
        if (pr != seed) { inst = i; prim = pr; slot = sl; }
    }
};

// Outputs of the answer (inst, slot) for the world point p: point_tri on the world triangle (c, d2, w0, w1, region)
// and the object-space vertices v (for the face normal of the sign).
RT_HD PointHit scene_point_attr(const SceneView& sv, int32_t inst, uint32_t slot, float px, float py, float pz, float v[9]) {
    const SceneInst& s = sv.inst[inst];
    const uint8_t* blob = reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]);
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    const uint8_t* tp = blob + h->tris_offset + (size_t)slot * 48u;
    const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
    v[0] = as_float(a.x); v[1] = as_float(a.y); v[2] = as_float(a.z);
    v[3] = as_float(b.x); v[4] = as_float(b.y); v[5] = as_float(b.z);
    v[6] = as_float(c.x); v[7] = as_float(c.y); v[8] = as_float(c.z);
    float w[9];
    world_tri(s.fwd, a, b, c, w);
    return point_tri(px, py, pz, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w[8]);
}

// Pseudo-normal sign of a scene answer: n = the mesh's row (or object face normal) of the region of c, carried to
// world as n_w = A^-T n (column k of the stored inverse, affine_row with offset -0: the identity keeps n), then
// +d when (p - c) . n_w < 0, else -d; d = 0 gives +0.  A^-T maps outward normals to outward normals for every
// invertible A, mirrors included.
RT_HD float scene_pseudonormal_sign(const SceneInst& s, const uint8_t* normals, uint32_t slot, const PointHit& h, float px,
                                    float py, float pz, const float v[9], float d) {
    float nx, ny, nz;
    region_normal(normals, slot, h.region, v, nx, ny, nz);
    const float nz0 = as_float(0x80000000u);
    const float wx = affine_row(s.inv[0], s.inv[4], s.inv[8], nz0, nx, ny, nz);
    const float wy = affine_row(s.inv[1], s.inv[5], s.inv[9], nz0, nx, ny, nz);
    const float wz = affine_row(s.inv[2], s.inv[6], s.inv[10], nz0, nx, ny, nz);
    const float sg = dot3f(fsub(px, h.cx), fsub(py, h.cy), fsub(pz, h.cz), wx, wy, wz);
    return (sg < 0.0f || d == 0.0f) ? d : -d;
}

}  // namespace rt
