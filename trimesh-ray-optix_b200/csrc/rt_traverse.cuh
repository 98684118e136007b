// rt_traverse.cuh — stack-based traversal of the compressed BVH8 for one ray.
//
// Replaces the traversal hidden behind optixTrace (triro/backend/shaders.cu:86,112,163,191,238).
// One thread owns one ray.  The traversal state is the (node group, triangle group) pair of
// Ylitie et al. 2017: a node group is {child_base, hit bits 24..31 | imask}, so the stack
// holds at most one entry per tree level.
#pragma once
#include "rt_core.cuh"

namespace rt {

#if defined(__CUDA_ARCH__)
RT_HD int clz32(uint32_t x) { return __clz((int)x); }
RT_HD int popc32(uint32_t x) { return __popc(x); }
RT_HD int ffs32(uint32_t x) { return __ffs((int)x); }
RT_HD U4 ldg128(const void* p) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));   // ld.global.nc.v4.u32
    U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r;
}
#else
RT_HD int clz32(uint32_t x) { return x ? __builtin_clz(x) : 32; }
RT_HD int popc32(uint32_t x) { return __builtin_popcount(x); }
RT_HD int ffs32(uint32_t x) { return __builtin_ffs((int)x); }
RT_HD U4 ldg128(const void* p) { return *reinterpret_cast<const U4*>(p); }
#endif

// Per-ray traversal state: the current node group (gx = child_base, gy = inner hit bits 24..31 |
// imask) and the stack depth.  trav_step() advances one wide node: pick the nearest pending
// child, test its 8 slots, intersect the triangles of the hit leaf slots, pop when the group is
// exhausted.  Splitting traversal into steps lets the kernel re-fill finished lanes of a warp
// between steps (persistent threads with dynamic ray fetch, Aila & Laine 2009).
struct Trav {
    uint32_t gx, gy;
    int sp;
};
RT_HD void trav_init(Trav& t) { t.gx = 0u; t.gy = 0x80000000u; t.sp = 0; }   // root group: node 0, top priority

// Visitor concept:
//   float tmax            current far limit of the ray interval (closest-hit shrinks it)
//   bool hit(const Ray&, const TriHit&, int32_t prim, uint32_t tri_slot)  -> true = terminate ray
//   void count_node(), count_tri()   instrumentation hooks
// Returns true when the ray is finished.
template <class Visitor, class StackT>
RT_HD bool trav_step(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ tris, const Ray& r,
                     Visitor& vis, StackT& stack, Trav& t) {
    if (t.gy & 0xff000000u) {
        const uint32_t hits = t.gy;
        const int bit = 31 - clz32(hits);
        t.gy &= ~(1u << bit);
        if (t.gy & 0xff000000u) { stack.push(t.sp, t.gx, t.gy); ++t.sp; }
        const uint32_t slot = (uint32_t)(bit - 24) ^ r.octinv;
        const uint32_t rel = (uint32_t)popc32(hits & ~(0xffffffffu << slot));
        const uint8_t* np = nodes + (size_t)(t.gx + rel) * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48),
                 n4 = ldg128(np + 64);
        vis.count_node();
        const uint32_t hm = node_test(r, n0, n1, n2, n3, n4, 0.0f, vis.tmax);
        t.gx = n1.x;
        t.gy = (hm & 0xff000000u) | (n0.w >> 24);
        uint32_t ty = hm & 0x00ffffffu;
        const uint32_t tx = n1.y, tmask = n1.z;
        while (ty) {
            const int b = ffs32(ty) - 1;
            ty &= ty - 1u;
            const uint32_t slot_t = tx + (uint32_t)popc32(tmask & ~(0xffffffffu << b));
            const uint8_t* tp = tris + (size_t)slot_t * 48u;
            const U4 a = ldg128(tp), bb = ldg128(tp + 16), c = ldg128(tp + 32);
            vis.count_tri();
            TriHit h;
            if (tri_test(r, as_float(a.x), as_float(a.y), as_float(a.z), as_float(bb.x), as_float(bb.y),
                         as_float(bb.z), as_float(c.x), as_float(c.y), as_float(c.z), h)) {
                if (vis.hit(r, h, (int32_t)a.w, slot_t)) return true;
            }
        }
    }
    if (!(t.gy & 0xff000000u)) {
        if (t.sp == 0) return true;
        --t.sp;
        stack.pop(t.sp, t.gx, t.gy);
    }
    return false;
}

template <class Visitor, class StackT>
RT_HD void traverse(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ tris, const Ray& r,
                    Visitor& vis, StackT& stack) {
    Trav t;
    trav_init(t);
    while (!trav_step(nodes, tris, r, vis, stack, t)) {}
}

// ------------------------------------------------------------------ visitors
struct NoStats {
    RT_HD void count_node() {}
    RT_HD void count_tri() {}
    RT_HD uint32_t n_nodes() const { return 0; }
    RT_HD uint32_t n_tris() const { return 0; }
};
struct Stats {
    uint32_t nodes = 0, tris = 0;
    RT_HD void count_node() { ++nodes; }
    RT_HD void count_tri() { ++tris; }
    RT_HD uint32_t n_nodes() const { return nodes; }
    RT_HD uint32_t n_tris() const { return tris; }
};

// nearest hit in the open interval (0, tmax0); equal-t ties resolved towards the smaller
// primitive index so that the answer does not depend on BVH topology.
template <class S>
struct ClosestVisitor : S {
    float tmax;
    int32_t prim = -1;
    uint32_t slot = 0;
    RT_HD explicit ClosestVisitor(float tmax0) : tmax(tmax0) {}
    RT_HD bool hit(const Ray&, const TriHit& h, int32_t p, uint32_t s) {
        if (h.t > 0.0f && (h.t < tmax || (h.t == tmax && p < prim))) { tmax = h.t; prim = p; slot = s; }
        return false;
    }
};

template <class S>
struct AnyVisitor : S {
    float tmax;
    bool found = false;
    RT_HD explicit AnyVisitor(float tmax0) : tmax(tmax0) {}
    RT_HD bool hit(const Ray&, const TriHit& h, int32_t, uint32_t) {
        if (h.t > 0.0f && h.t < tmax) { found = true; return true; }
        return false;
    }
};

template <class S>
struct CountVisitor : S {
    float tmax;
    int32_t count = 0;
    RT_HD explicit CountVisitor(float tmax0) : tmax(tmax0) {}
    RT_HD bool hit(const Ray&, const TriHit& h, int32_t, uint32_t) {
        if (h.t > 0.0f && h.t < tmax) ++count;
        return false;
    }
};

}  // namespace rt
