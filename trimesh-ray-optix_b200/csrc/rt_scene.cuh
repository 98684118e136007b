// rt_scene.cuh — arithmetic of instanced scenes (rt_scene.cu): the per-instance preparation (binary64 inverse, world
// box, padding) and the two-level walk (a top-level BVH8 over instance boxes, each instance's own BVH8 below it).
//
// Everything here is RT_HD and a pure function of its arguments, so the host simulator under tests/scene/ runs the
// same code (DESIGN.md §4.11).  The top-level tree is an ordinary blob from rt_bvh_build: instance i is the "triangle"
// (lo_i, hi_i, lo_i) whose box is exactly the padded world box [lo_i, hi_i], and its record's prim is i.
#pragma once
#include "../../include/raymesh_b200.h"
#include "rt_traverse.cuh"

namespace rt {

#if defined(__CUDA_ARCH__)
RT_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
RT_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
#else
RT_HD double dadd(double a, double b) { return a + b; }
RT_HD double ddiv(double a, double b) { return a / b; }
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

}  // namespace rt
