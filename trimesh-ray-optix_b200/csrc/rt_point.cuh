// rt_point.cuh — closest-point queries on the BVH8: point/triangle distance, per-slot lower bounds and one traversal
// step.  Everything here is RT_HD, like rt_core.cuh, so that tests/pointquery/ steps exactly the code the kernel runs
// (rt_closest.cu) on a CPU-built blob.
//
// Result contract (DESIGN.md §4.6): for a point p the answer is the triangle minimising the key (d2, prim) over all
// triangles with d2 <= max_d2, where d2 is what point_tri() returns.  Nothing depends on the traversal order, so the
// kernel, the host simulator and a brute-force loop over point_tri() agree bit for bit.
#pragma once
#include "rt_traverse.cuh"

namespace rt {

#if defined(__CUDA_ARCH__)
RT_HD float fsqrt(float a) { return __fsqrt_rn(a); }
RT_HD uint32_t as_uint(float f) { return __float_as_uint(f); }
#else
RT_HD float fsqrt(float a) { return sqrtf(a); }
RT_HD uint32_t as_uint(float f) { union { float f; uint32_t u; } c; c.f = f; return c.u; }
#endif

// ------------------------------------------------------------------ closest point on one triangle
// Ericson, Real-Time Collision Detection §5.1.5 (Voronoi regions of the vertices, edges and face), as a fixed sequence
// of binary32 operations.  w0, w1 are the weights of v0 and v1, the uv convention of intersects_closest, so
// RayMeshIntersector.interpolate() applies unchanged.  d2 = (p-c).(p-c) of the returned point c.
//   * a triangle whose va + vb + vc (= |ab x ac|^2 in exact arithmetic) is not positive has zero area: its closest
//     point is that of the nearest of its three edges, each taken as a segment; a zero-length segment is a point;
//   * every parameter a division yields lies in [0, 1] (numerator <= denominator by construction, the face weights
//     clamped at 0): the computed c is a convex combination of the vertices up to rounding (the margin of
//     slot_lower_bounds relies on that).  Finite vertices: no division by zero, no NaN;
//   * a NaN coordinate anywhere gives d2 = NaN, which no comparison accepts: such a triangle is never selected.
// `region` is the Voronoi region of the branch that produced c (kRegion*, DESIGN.md §4.8): in the zero-area branch the
// chosen segment's edge, or the vertex at its end when t = 0 or t = 1.  The signed-distance kernel takes the
// pseudo-normal of that feature.
enum : uint32_t { kRegionFace = 0, kRegionA = 1, kRegionB = 2, kRegionC = 3, kRegionAB = 4, kRegionAC = 5, kRegionBC = 6 };
struct PointHit { float cx, cy, cz, d2, w0, w1; uint32_t region; };

// the region of a point at parameter t on the segment from vertex region `v0` to `v1` along edge region `e`
RT_HD uint32_t seg_region(float t, uint32_t v0, uint32_t v1, uint32_t e) { return t == 0.0f ? v0 : (t == 1.0f ? v1 : e); }

RT_HD float dot3f(float ax, float ay, float az, float bx, float by, float bz) {
    return fadd(fadd(fmul(ax, bx), fmul(ay, by)), fmul(az, bz));
}

// closest point of segment a + t*(b - a), t in [0, 1]; returns t
RT_HD float seg_param(float apx, float apy, float apz, float abx, float aby, float abz) {
    const float num = dot3f(apx, apy, apz, abx, aby, abz);
    const float den = dot3f(abx, aby, abz, abx, aby, abz);
    if (!(num > 0.0f) || !(den > 0.0f)) return 0.0f;
    return num < den ? fdiv(num, den) : 1.0f;
}

RT_HD PointHit point_tri(float px, float py, float pz, float ax, float ay, float az, float bx, float by, float bz,
                         float cx, float cy, float cz) {
    PointHit r;
    const bool nan_vertex = ax != ax || ay != ay || az != az || bx != bx || by != by || bz != bz || cx != cx ||
                            cy != cy || cz != cz;
    if (nan_vertex) {
        r.cx = r.cy = r.cz = 0.0f; r.w0 = r.w1 = 0.0f; r.d2 = as_float(0x7fc00000u); r.region = kRegionFace;
        return r;
    }
    const float abx = fsub(bx, ax), aby = fsub(by, ay), abz = fsub(bz, az);
    const float acx = fsub(cx, ax), acy = fsub(cy, ay), acz = fsub(cz, az);
    const float apx = fsub(px, ax), apy = fsub(py, ay), apz = fsub(pz, az);
    const float bpx = fsub(px, bx), bpy = fsub(py, by), bpz = fsub(pz, bz);
    const float cpx = fsub(px, cx), cpy = fsub(py, cy), cpz = fsub(pz, cz);
    const float d1 = dot3f(abx, aby, abz, apx, apy, apz), d2 = dot3f(acx, acy, acz, apx, apy, apz);
    const float d3 = dot3f(abx, aby, abz, bpx, bpy, bpz), d4 = dot3f(acx, acy, acz, bpx, bpy, bpz);
    const float d5 = dot3f(abx, aby, abz, cpx, cpy, cpz), d6 = dot3f(acx, acy, acz, cpx, cpy, cpz);
    const float vc = fsub(fmul(d1, d4), fmul(d3, d2));
    const float vb = fsub(fmul(d5, d2), fmul(d1, d6));
    const float va = fsub(fmul(d3, d6), fmul(d5, d4));
    const float den = fadd(fadd(va, vb), vc);                         // |ab x ac|^2 in exact arithmetic
    if (!(den > 0.0f)) {                                              // zero area: nearest of the three segments
        const float t0 = seg_param(apx, apy, apz, abx, aby, abz);
        const float t1 = seg_param(apx, apy, apz, acx, acy, acz);
        const float bcx = fsub(cx, bx), bcy = fsub(cy, by), bcz = fsub(cz, bz);
        const float t2 = seg_param(bpx, bpy, bpz, bcx, bcy, bcz);
        const float qx0 = fadd(ax, fmul(t0, abx)), qy0 = fadd(ay, fmul(t0, aby)), qz0 = fadd(az, fmul(t0, abz));
        const float qx1 = fadd(ax, fmul(t1, acx)), qy1 = fadd(ay, fmul(t1, acy)), qz1 = fadd(az, fmul(t1, acz));
        const float qx2 = fadd(bx, fmul(t2, bcx)), qy2 = fadd(by, fmul(t2, bcy)), qz2 = fadd(bz, fmul(t2, bcz));
        const float e0 = dot3f(fsub(px, qx0), fsub(py, qy0), fsub(pz, qz0), fsub(px, qx0), fsub(py, qy0), fsub(pz, qz0));
        const float e1 = dot3f(fsub(px, qx1), fsub(py, qy1), fsub(pz, qz1), fsub(px, qx1), fsub(py, qy1), fsub(pz, qz1));
        const float e2 = dot3f(fsub(px, qx2), fsub(py, qy2), fsub(pz, qz2), fsub(px, qx2), fsub(py, qy2), fsub(pz, qz2));
        if (e0 <= e1 && e0 <= e2) {
            r.cx = qx0; r.cy = qy0; r.cz = qz0; r.w0 = fsub(1.0f, t0); r.w1 = t0;
            r.region = seg_region(t0, kRegionA, kRegionB, kRegionAB);
        } else if (e1 <= e2) {
            r.cx = qx1; r.cy = qy1; r.cz = qz1; r.w0 = fsub(1.0f, t1); r.w1 = 0.0f;
            r.region = seg_region(t1, kRegionA, kRegionC, kRegionAC);
        } else {
            r.cx = qx2; r.cy = qy2; r.cz = qz2; r.w0 = 0.0f; r.w1 = fsub(1.0f, t2);
            r.region = seg_region(t2, kRegionB, kRegionC, kRegionBC);
        }
    } else if (d1 <= 0.0f && d2 <= 0.0f) {                            // vertex a
        r.cx = ax; r.cy = ay; r.cz = az; r.w0 = 1.0f; r.w1 = 0.0f; r.region = kRegionA;
    } else if (d3 >= 0.0f && d4 <= d3) {                              // vertex b
        r.cx = bx; r.cy = by; r.cz = bz; r.w0 = 0.0f; r.w1 = 1.0f; r.region = kRegionB;
    } else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f) {              // edge ab
        const float den = fsub(d1, d3);
        const float t = den > 0.0f ? fdiv(d1, den) : 0.0f;
        r.cx = fadd(ax, fmul(t, abx)); r.cy = fadd(ay, fmul(t, aby)); r.cz = fadd(az, fmul(t, abz));
        r.w0 = fsub(1.0f, t); r.w1 = t; r.region = kRegionAB;
    } else if (d6 >= 0.0f && d5 <= d6) {                              // vertex c
        r.cx = cx; r.cy = cy; r.cz = cz; r.w0 = 0.0f; r.w1 = 0.0f; r.region = kRegionC;
    } else if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f) {              // edge ac
        const float den = fsub(d2, d6);
        const float t = den > 0.0f ? fdiv(d2, den) : 0.0f;
        r.cx = fadd(ax, fmul(t, acx)); r.cy = fadd(ay, fmul(t, acy)); r.cz = fadd(az, fmul(t, acz));
        r.w0 = fsub(1.0f, t); r.w1 = 0.0f; r.region = kRegionAC;
    } else if (va <= 0.0f && fsub(d4, d3) >= 0.0f && fsub(d5, d6) >= 0.0f) {   // edge bc
        const float num = fsub(d4, d3);
        const float den = fadd(num, fsub(d5, d6));
        const float t = den > 0.0f ? fdiv(num, den) : 0.0f;
        r.cx = fadd(bx, fmul(t, fsub(cx, bx))); r.cy = fadd(by, fmul(t, fsub(cy, by))); r.cz = fadd(bz, fmul(t, fsub(cz, bz)));
        r.w0 = 0.0f; r.w1 = fsub(1.0f, t); r.region = kRegionBC;
    } else {                                                          // face
        // va, vb, vc >= 0 here in exact arithmetic; v, w >= 0 and v + w <= 1 are enforced so that rounding on a sliver
        // cannot move the point off the triangle
        const float v = fminf(fdiv(fmaxf(vb, 0.0f), den), 1.0f);
        const float w = fminf(fdiv(fmaxf(vc, 0.0f), den), fsub(1.0f, v));
        r.cx = fadd(fadd(ax, fmul(v, abx)), fmul(w, acx));
        r.cy = fadd(fadd(ay, fmul(v, aby)), fmul(w, acy));
        r.cz = fadd(fadd(az, fmul(v, abz)), fmul(w, acz));
        r.w0 = fsub(fsub(1.0f, v), w); r.w1 = v; r.region = kRegionFace;
    }
    const float dx = fsub(px, r.cx), dy = fsub(py, r.cy), dz = fsub(pz, r.cz);
    r.d2 = dot3f(dx, dy, dz, dx, dy, dz);
    return r;
}

// ------------------------------------------------------------------ per-slot lower bounds
// lb[s] <= the d2 point_tri() computes for every triangle below slot s of the node (n0, n2, n3, n4 = words 0, 2, 3, 4),
// read from the same encoding node_test uses: plane = p + q * 2^e, here evaluated relative to the query point as
// fma(q, 2^e, p - x).
//
// Error argument, per axis (u = 2^-24, b = p - x of the node origin, s = 2^e, A = |p| + 256 s bounds every vertex
// coordinate below the node, because the slot boxes contain their triangles in real arithmetic):
//   (1) the plane relative to the point is off by at most u|b| (the subtraction) + u|b + q s| (the fma) <= u(2|b| + 256 s);
//   (2) the closest point c point_tri() returns is a convex combination of the vertices up to rounding, <= 22 u A per
//       axis outside the triangle's box (face branch; vertex 0, edges and segments <= 7 u A), hence outside the slot box;
//   so |x - c| >= gap - m per axis with m = 2^-18 (|b| + |p| + 256 s) = 64 u (...), which covers (1) + (2) with room for
//   the rounding of m itself.  The sum of the squared (gap - m)+ is at most (1 + 5u) times the exact (x-c).(x-c), and
//   point_tri's own d2 is at least (1 - 5u) times it: the final factor 1 - 2^-20 = 1 - 16u (rounded once more) keeps
//   lb <= d2.  Empty slots yield a value that is never used; a NaN point yields NaN, which fails every `<= best`.
RT_HD void slot_lower_bounds(float x, float y, float z, const U4& n0, const U4& n2, const U4& n3, const U4& n4, float lb[8]) {
    const float px = as_float(n0.x), py = as_float(n0.y), pz = as_float(n0.z);
    const float sx = as_float((n0.w & 0xffu) << 23), sy = as_float(((n0.w >> 8) & 0xffu) << 23),
                sz = as_float(((n0.w >> 16) & 0xffu) << 23);
    const float bx = fsub(px, x), by = fsub(py, y), bz = fsub(pz, z);
    const float km = 3.814697265625e-06f;   // 2^-18
    const float mx = fmul(km, fadd(fadd(fabsf(bx), fabsf(px)), fmul(256.0f, sx)));
    const float my = fmul(km, fadd(fadd(fabsf(by), fabsf(py)), fmul(256.0f, sy)));
    const float mz = fmul(km, fadd(fadd(fabsf(bz), fabsf(pz)), fmul(256.0f, sz)));
    const uint32_t qw[12] = {n2.x, n2.y, n2.z, n2.w, n3.x, n3.y, n3.z, n3.w, n4.x, n4.y, n4.z, n4.w};
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const int w = s >> 2, sh = 8 * (s & 3);
        const float qlx = (float)((qw[0 + w] >> sh) & 0xffu), qly = (float)((qw[2 + w] >> sh) & 0xffu);
        const float qlz = (float)((qw[4 + w] >> sh) & 0xffu), qhx = (float)((qw[6 + w] >> sh) & 0xffu);
        const float qhy = (float)((qw[8 + w] >> sh) & 0xffu), qhz = (float)((qw[10 + w] >> sh) & 0xffu);
        // distance to the interval [lo, hi] along each axis: lo - x when positive, x - hi when positive, else 0
        const float gx = fmaxf(fmaxf(ffma(qlx, sx, bx), -ffma(qhx, sx, bx)), 0.0f);
        const float gy = fmaxf(fmaxf(ffma(qly, sy, by), -ffma(qhy, sy, by)), 0.0f);
        const float gz = fmaxf(fmaxf(ffma(qlz, sz, bz), -ffma(qhz, sz, bz)), 0.0f);
        const float hx = fmaxf(fsub(gx, mx), 0.0f), hy = fmaxf(fsub(gy, my), 0.0f), hz = fmaxf(fsub(gz, mz), 0.0f);
        lb[s] = fmul(dot3f(hx, hy, hz, hx, hy, hz), 0.999999046325684f);   // 1 - 2^-20
    }
}

// ------------------------------------------------------------------ traversal
// Group stack after rt_traverse.cuh: one entry per tree level, holding the inner children of a node that are still
// pending, nearest first.  An entry is (child_base, list, bound): list = up to 7 child offsets (3 bits each, the
// order they are visited in) plus their count in bits 29..31, bound = the smallest of their lower bounds when the group
// was pushed (a valid lower bound for all of them).  A popped group whose bound exceeds the current best is dropped
// whole; its children are otherwise visited one by one without a bound of their own (each child's own slots prune).
struct PointStackEntry { uint32_t base, list; float bound; };

struct PointTrav {
    float x, y, z;
    float best;          // d2 of the current answer, initially max_d2
    int32_t prim;        // current answer, 0x7fffffff = none yet
    uint32_t slot;       // triangle record of the current answer
    uint32_t node;       // node to visit next, kNoNode = pop
    int sp;
};
constexpr uint32_t kNoNode = 0xffffffffu;
constexpr int32_t kNoPrim = 0x7fffffff;

RT_HD void point_init(PointTrav& t, float x, float y, float z, float max_d2) {
    t.x = x; t.y = y; t.z = z; t.best = max_d2; t.prim = kNoPrim; t.slot = 0u; t.node = 0u; t.sp = 0;
    // a non-finite point has no answer (x - x is NaN for NaN and +-inf)
    if (!(fsub(x, x) == 0.0f && fsub(y, y) == 0.0f && fsub(z, z) == 0.0f)) t.node = kNoNode;
}

// key of an inner slot for sorting: lower bound with its low 3 bits replaced by the slot's child offset.  Bounds are
// >= +0, so the bit pattern orders like the value, and clearing 3 bits only lowers it (still a lower bound).
RT_HD void cswap_lo(uint32_t& a, uint32_t& b) { const uint32_t lo = a < b ? a : b, hi = a < b ? b : a; a = lo; b = hi; }

// The space a walk runs in: how a node's slot bounds are formed and how a leaf record is tested.  MeshSpace is the
// single mesh (the point and the triangles in one space); the instanced scene (rt_scene.cuh) adds a world-space walk of
// one instance's tree and the top-level walk whose records are instances.  leaf() may lower t.best and sets the answer.
struct MeshSpace {
    RT_HD void bounds(const PointTrav& t, const U4& n0, const U4& n2, const U4& n3, const U4& n4, float lb[8]) const {
        slot_lower_bounds(t.x, t.y, t.z, n0, n2, n3, n4, lb);
    }
    RT_HD void leaf(PointTrav& t, uint32_t rec, const U4& a, const U4& b, const U4& c) const {
        const PointHit h = point_tri(t.x, t.y, t.z, as_float(a.x), as_float(a.y), as_float(a.z), as_float(b.x),
                                     as_float(b.y), as_float(b.z), as_float(c.x), as_float(c.y), as_float(c.z));
        const int32_t prim = (int32_t)a.w;
        if (h.d2 < t.best || (h.d2 == t.best && prim < t.prim)) { t.best = h.d2; t.prim = prim; t.slot = rec; }
    }
};

// One node visit or one pop; returns true when the point is finished.  Visitor: count_node(), count_tri().
template <class S, class StackT, class Space>
RT_HD bool point_step(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ tris, PointTrav& t, S& st,
                      StackT& stack, Space& space) {
    if (t.node != kNoNode) {
        const uint8_t* np = nodes + (size_t)t.node * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48), n4 = ldg128(np + 64);
        st.count_node();
        float lb[8];
        space.bounds(t, n0, n2, n3, n4, lb);
        const uint32_t imask = n0.w >> 24, tbase = n1.y, tmask = n1.z;
        // leaves first: their triangles can only lower `best`, which prunes the inner slots below
        for (int s = 0; s < 8; ++s) {
            const uint32_t un = (tmask >> (3 * s)) & 7u;
            if (un == 0u || !(lb[s] <= t.best)) continue;
            uint32_t rec = tbase + (uint32_t)popc32(tmask & ((1u << (3 * s)) - 1u));
            const uint32_t cnt = (uint32_t)popc32(un);
            for (uint32_t j = 0; j < cnt; ++j, ++rec) {
                const uint8_t* tp = tris + (size_t)rec * 48u;
                const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
                st.count_tri();
                space.leaf(t, rec, a, b, c);
            }
        }
        // inner children within reach, nearest first (sorting network on 8 keys; absent ones sort last as ~0)
        uint32_t k[8];
        uint32_t rel = 0u;
#pragma unroll
        for (int s = 0; s < 8; ++s) {
            const bool inner = (imask >> s) & 1u;
            k[s] = (inner && lb[s] <= t.best) ? ((as_uint(lb[s]) & ~7u) | rel) : 0xffffffffu;
            rel += inner ? 1u : 0u;
        }
        // Batcher's odd-even merge sort, 19 comparators
        cswap_lo(k[0], k[1]); cswap_lo(k[2], k[3]); cswap_lo(k[4], k[5]); cswap_lo(k[6], k[7]);
        cswap_lo(k[0], k[2]); cswap_lo(k[1], k[3]); cswap_lo(k[4], k[6]); cswap_lo(k[5], k[7]);
        cswap_lo(k[1], k[2]); cswap_lo(k[5], k[6]);
        cswap_lo(k[0], k[4]); cswap_lo(k[1], k[5]); cswap_lo(k[2], k[6]); cswap_lo(k[3], k[7]);
        cswap_lo(k[2], k[4]); cswap_lo(k[3], k[5]);
        cswap_lo(k[1], k[2]); cswap_lo(k[3], k[4]); cswap_lo(k[5], k[6]);
        if (k[0] == 0xffffffffu) {
            t.node = kNoNode;
        } else {
            const uint32_t base = n1.x;
            t.node = base + (k[0] & 7u);
            uint32_t list = 0u, n = 0u;
#pragma unroll
            for (int i = 7; i >= 1; --i) {
                if (k[i] != 0xffffffffu) { list = (list << 3) | (k[i] & 7u); ++n; }
            }
            if (n > 0u) {
                PointStackEntry e;
                e.base = base; e.list = list | (n << 29); e.bound = as_float(k[1] & ~7u);
                stack.push(t.sp, e);
                ++t.sp;
            }
        }
        return false;
    }
    while (t.sp > 0) {
        PointStackEntry e;
        stack.pop(t.sp - 1, e);
        if (!(e.bound <= t.best)) { --t.sp; continue; }   // the whole group is farther than the answer
        const uint32_t n = e.list >> 29;
        t.node = e.base + (e.list & 7u);
        if (n == 1u) {
            --t.sp;
        } else {
            e.list = (((e.list & 0x1fffffffu) >> 3)) | ((n - 1u) << 29);
            stack.push(t.sp - 1, e);
        }
        return false;
    }
    return true;
}

template <class S, class StackT>
RT_HD bool point_step(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ tris, PointTrav& t, S& st,
                      StackT& stack) {
    MeshSpace space;
    return point_step(nodes, tris, t, st, stack, space);
}

}  // namespace rt
