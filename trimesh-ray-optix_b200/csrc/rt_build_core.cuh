// rt_build_core.cuh — per-element logic of the BVH builder (pure functions, host/device).
//
// Replaces what the reference obtains from optixAccelBuild/optixAccelCompact
// (triro/backend/ray.cpp:64-93): Morton codes, Karras' LBVH hierarchy, and the collapse of the
// binary hierarchy into 8-wide nodes with quantised child boxes.
#pragma once
#include "rt_core.cuh"

namespace rt {

struct alignas(16) BBox {
    float lx, ly, lz, pad0;
    float hx, hy, hz, pad1;
};

RT_HD float fmin_nan(float a, float b) { return fminf(a, b); }   // NaN-ignoring on both host and device
RT_HD float fmax_nan(float a, float b) { return fmaxf(a, b); }

RT_HD BBox bbox_union(const BBox& a, const BBox& b) {
    BBox r;
    r.lx = fminf(a.lx, b.lx); r.ly = fminf(a.ly, b.ly); r.lz = fminf(a.lz, b.lz);
    r.hx = fmaxf(a.hx, b.hx); r.hy = fmaxf(a.hy, b.hy); r.hz = fmaxf(a.hz, b.hz);
    r.pad0 = 0.f; r.pad1 = 0.f;
    return r;
}

// Written as explicit operations: the collapse compares these areas, and a sum of products left to the compiler is
// contracted into FMAs on the device but not on the host, which picks different children when two areas tie in exact
// arithmetic (congruent triangles of a symmetric mesh).  This is the sequence nvcc chose for the plain expression.
RT_HD float bbox_half_area(const BBox& b) {
    const float dx = b.hx - b.lx, dy = b.hy - b.ly, dz = b.hz - b.lz;
    return ffma(dz, dx, ffma(dx, dy, fmul(dy, dz)));
}

// Triangle box, widened by a few ulps so that the watertight triangle test (which may accept
// rays a rounding error outside the exact triangle) never reports a hit outside the box.
RT_HD BBox tri_bbox(float v0x, float v0y, float v0z, float v1x, float v1y, float v1z, float v2x, float v2y,
                    float v2z) {
    BBox b;
    b.lx = fminf(fminf(v0x, v1x), v2x); b.ly = fminf(fminf(v0y, v1y), v2y); b.lz = fminf(fminf(v0z, v1z), v2z);
    b.hx = fmaxf(fmaxf(v0x, v1x), v2x); b.hy = fmaxf(fmaxf(v0y, v1y), v2y); b.hz = fmaxf(fmaxf(v0z, v1z), v2z);
    const float k = 6.0e-7f, tiny = 1.0e-30f;   // |x| * k + tiny as one FMA, as nvcc contracts it, on the host as well
    b.lx -= ffma(fabsf(b.lx), k, tiny); b.ly -= ffma(fabsf(b.ly), k, tiny); b.lz -= ffma(fabsf(b.lz), k, tiny);
    b.hx += ffma(fabsf(b.hx), k, tiny); b.hy += ffma(fabsf(b.hy), k, tiny); b.hz += ffma(fabsf(b.hz), k, tiny);
    b.pad0 = 0.f; b.pad1 = 0.f;
    return b;
}

// Leaf box of the binary hierarchy: the triangle box united with the empty box, so that an axis on which all three
// vertices are NaN is empty (+inf, -inf) instead of NaN - the box refit_node computes for the same triangle, so that a
// refit to the build's own vertices reproduces the built nodes bit for bit.  (fminf ignores a NaN operand, so nothing
// changes on any other axis.)
RT_HD BBox leaf_bbox(const BBox& tb) {
    BBox e; e.lx = e.ly = e.lz = INFINITY; e.hx = e.hy = e.hz = -INFINITY; e.pad0 = e.pad1 = 0.f;
    return bbox_union(e, tb);
}

// ------------------------------------------------------------------ scene bounds
// The scene box is reduced in the ordered-uint encoding of binary32, a total order with -0 < +0 in which a NaN never
// wins: the result does not depend on the order of the reduction (fminf leaves min(-0, +0) open), and a mesh whose
// triangle boxes are all NaN keeps the initial values, an empty box (+inf, -inf) per axis.
#if defined(__CUDA_ARCH__)
RT_HD uint32_t float_bits(float f) { return __float_as_uint(f); }
#else
RT_HD uint32_t float_bits(float f) { union { float f; uint32_t u; } c; c.f = f; return c.u; }
#endif
RT_HD uint32_t f2ord(float f) {
    const uint32_t u = float_bits(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
RT_HD float ord2f(uint32_t u) { return as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }
constexpr uint32_t kOrdPosInf = 0xff800000u;   // f2ord(+inf): start of a min
constexpr uint32_t kOrdNegInf = 0x007fffffu;   // f2ord(-inf): start of a max
RT_HD uint32_t ord_lo(float f) { return f == f ? f2ord(f) : 0xffffffffu; }   // NaN: above every number, never a min
RT_HD uint32_t ord_hi(float f) { return f == f ? f2ord(f) : 0u; }            // NaN: below every number, never a max

// ------------------------------------------------------------------ blob layout behind the nodes
// The (parent << 3 | slot) array of the wide nodes sits right behind the nodes in use, so that the used prefix of the
// blob - what travels over NCCL or to disk - is complete; used_bytes ends 16-byte aligned behind it.
RT_HD uint64_t parents_offset_for(uint64_t nodes_offset, uint32_t n_nodes) {
    return (nodes_offset + (uint64_t)n_nodes * 80u + 255u) / 256u * 256u;
}
RT_HD uint64_t used_bytes_for(uint64_t parents_offset, uint32_t n_nodes) {
    return (parents_offset + (uint64_t)n_nodes * 4u + 15u) / 16u * 16u;
}

// ------------------------------------------------------------------ Morton codes (21 bits per axis)
RT_HD uint64_t expand21(uint64_t x) {
    x &= 0x1fffffull;
    x = (x | (x << 32)) & 0x001f00000000ffffull;
    x = (x | (x << 16)) & 0x001f0000ff0000ffull;
    x = (x | (x << 8)) & 0x100f00f00f00f00full;
    x = (x | (x << 4)) & 0x10c30c30c30c30c3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

// One uniform scale for all three axes (the largest scene extent maps to the full 21 bits): the
// Morton grid cells are cubes, so a flat scene (terrain) is not sliced along its thin axis before it
// has been subdivided along the long ones; bits that never vary simply create no hierarchy level.
RT_HD void morton_scale(const float lo[3], const float hi[3], float inv_ext[3]) {
    float m = 0.0f;
    for (int a = 0; a < 3; ++a) { const float e = hi[a] - lo[a]; if (e > m) m = e; }
    const float inv = m > 0.0f ? 1.0f / m : 0.0f;
    inv_ext[0] = inv_ext[1] = inv_ext[2] = inv;
}

RT_HD uint64_t morton63(float cx, float cy, float cz, const float lo[3], const float inv_ext[3]) {
    const float scale = 2097152.0f;   // 2^21
    float fx = (cx - lo[0]) * inv_ext[0] * scale;
    float fy = (cy - lo[1]) * inv_ext[1] * scale;
    float fz = (cz - lo[2]) * inv_ext[2] * scale;
    fx = fminf(fmaxf(fx, 0.0f), 2097151.0f);   // NaN -> 0
    fy = fminf(fmaxf(fy, 0.0f), 2097151.0f);
    fz = fminf(fmaxf(fz, 0.0f), 2097151.0f);
    if (!(fx == fx)) fx = 0.0f;
    if (!(fy == fy)) fy = 0.0f;
    if (!(fz == fz)) fz = 0.0f;
    return expand21((uint64_t)fx) | (expand21((uint64_t)fy) << 1) | (expand21((uint64_t)fz) << 2);
}

// Bits per axis that take part in the ordering.  The sort costs one pass per 8 key bits, and a Morton grid far finer
// than the triangle density orders nothing the index tie-break of the hierarchy would not order as well:
// RT_MORTON_BITS_MID bits per axis up to 2^24 triangles (13 -> 39 key bits -> 5 sort passes; 8192 cells per axis are
// still >= 2 per triangle edge of a 16.8 M-triangle surface), 10 bits (4 passes) for small meshes, 16 (6 passes) up to
// 2^25 triangles and the full 21 (8 passes) beyond.  The key is the top 3*B bits of the 63-bit code, right-aligned.
#ifndef RT_MORTON_BITS_MID
#define RT_MORTON_BITS_MID 13
#endif
RT_HD int morton_axis_bits(int64_t n) {
    return n > ((int64_t)1 << 25) ? 21 : (n > ((int64_t)1 << 24) ? 16 : (n > ((int64_t)1 << 14) ? RT_MORTON_BITS_MID : 10));
}
RT_HD int morton_sort_passes(int64_t n) { return (3 * morton_axis_bits(n) + 7) / 8; }

// ------------------------------------------------------------------ Karras 2012 hierarchy
#if defined(__CUDA_ARCH__)
RT_HD int clz64(uint64_t x) { return __clzll((long long)x); }
RT_HD int clz32u(uint32_t x) { return __clz((int)x); }
#else
RT_HD int clz64(uint64_t x) { return x ? __builtin_clzll(x) : 64; }
RT_HD int clz32u(uint32_t x) { return x ? __builtin_clz(x) : 32; }
#endif

// length of the common prefix of keys i and j (index as tie-break); -1 when j is out of range.
// Idx = int32_t for n <= 2^29 (every probe index i + 2*range stays below 2^31): the searches are index arithmetic,
// and 32-bit indices halve their instruction count on the GPU; int64_t beyond.
template <class Idx>
RT_HD int karras_delta(const uint64_t* __restrict__ keys, Idx n, Idx i, uint64_t key_i, Idx j) {
    if (j < 0 || j >= n) return -1;
    const uint64_t b = keys[j];
    if (key_i == b) return 64 + clz32u((uint32_t)i ^ (uint32_t)j);
    return clz64(key_i ^ b);
}

// Node references: internal node k -> k (0..n-2); leaf at sorted position k -> (n-1) + k.
struct KarrasNode { uint32_t left, right, first, last; };

template <class Idx>
RT_HD KarrasNode karras_node_t(const uint64_t* __restrict__ keys, Idx n, Idx i) {
    const uint64_t ki = keys[i];
    const int dl = karras_delta<Idx>(keys, n, i, ki, i - 1), dr = karras_delta<Idx>(keys, n, i, ki, i + 1);
    const Idx d = dr > dl ? 1 : -1;
    const int dmin = dr > dl ? dl : dr;
    Idx lmax = 2;
    while (karras_delta<Idx>(keys, n, i, ki, i + lmax * d) > dmin) lmax <<= 1;
    Idx l = 0;
    for (Idx t = lmax >> 1; t >= 1; t >>= 1)
        if (karras_delta<Idx>(keys, n, i, ki, i + (l + t) * d) > dmin) l += t;
    const Idx j = i + l * d;
    const int dnode = karras_delta<Idx>(keys, n, i, ki, j);
    Idx s = 0;
    for (Idx t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (karras_delta<Idx>(keys, n, i, ki, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const Idx gamma = i + s * d + (d < 0 ? -1 : 0);
    const Idx lo = i < j ? i : j, hi = i < j ? j : i;
    KarrasNode k;
    k.left = (uint32_t)(lo == gamma ? (n - 1) + gamma : gamma);
    k.right = (uint32_t)(hi == gamma + 1 ? (n - 1) + gamma + 1 : gamma + 1);
    k.first = (uint32_t)lo;
    k.last = (uint32_t)hi;
    return k;
}

RT_HD KarrasNode karras_node(const uint64_t* __restrict__ keys, int64_t n, int64_t i) {
    if (n <= ((int64_t)1 << 29)) return karras_node_t<int32_t>(keys, (int32_t)n, (int32_t)i);
    return karras_node_t<int64_t>(keys, n, i);
}

// ------------------------------------------------------------------ collapse to BVH8
struct BinaryTree {
    int64_t n;                    // triangles (= leaves)
    const uint32_t* left;         // [n-1]
    const uint32_t* right;        // [n-1]
    const uint32_t* first;        // [n-1] first sorted position covered
    const uint32_t* last;         // [n-1]
    const BBox* box;              // [2n-1] internal boxes then leaf boxes
    const uint32_t* sorted_prim;  // [n] triangle id at each sorted position
    int leaf_max;                 // subtrees of <= leaf_max triangles become one leaf slot (1..kLeafMaxTris)
    int flagged;                  // child references in the box pads carry "covers more than leaf_max triangles" in bit 31
                                  // (written by the GPU refit pass), so expanding a child needs no first/last loads
};
constexpr uint32_t kRefMask = 0x7fffffffu;

RT_HD uint32_t bt_count(const BinaryTree& t, uint32_t ref) {
    return ref >= (uint32_t)(t.n - 1) ? 1u : t.last[ref] - t.first[ref] + 1u;
}
RT_HD uint32_t bt_first(const BinaryTree& t, uint32_t ref) {
    return ref >= (uint32_t)(t.n - 1) ? ref - (uint32_t)(t.n - 1) : t.first[ref];
}

#if defined(__CUDA_ARCH__)
RT_HD uint32_t atomic_add_u32(uint32_t* p, uint32_t v) { return atomicAdd(p, v); }
#else
RT_HD uint32_t atomic_add_u32(uint32_t* p, uint32_t v) { const uint32_t o = *p; *p = o + v; return o; }
#endif

// L1-bypassing load for data produced earlier in the same (cooperative) kernel
#if defined(__CUDA_ARCH__)
RT_HD uint32_t load_cg_u32(const uint32_t* p) { return __ldcg(p); }
#else
RT_HD uint32_t load_cg_u32(const uint32_t* p) { return *p; }
#endif

#if defined(__CUDA_ARCH__)
RT_HD BBox load_box(const BBox* p) {
    const float4 a = __ldcg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldcg(reinterpret_cast<const float4*>(p) + 1);
    BBox r; r.lx = a.x; r.ly = a.y; r.lz = a.z; r.pad0 = 0.f; r.hx = b.x; r.hy = b.y; r.hz = b.z; r.pad1 = 0.f;
    return r;
}
#else
RT_HD BBox load_box(const BBox* p) { return *p; }
#endif

RT_HD float exp2_biased(uint32_t e) { return as_float(e << 23); }

// Smallest biased exponent e (1..254) with 255 * 2^(e-127) >= ext.
RT_HD uint32_t quant_exponent(float ext) {
    if (!(ext > 0.0f)) return 1u;
    int k;
    const float m = frexpf(ext / 255.0f, &k);   // ext/255 = m * 2^k, m in [0.5, 1)
    (void)m;
    int e = k + 127;                            // 2^k >= ext/255
    if (e < 1) e = 1;
    if (e > 254) e = 254;
    return (uint32_t)e;
}

struct CollapseOut {
    uint8_t* nodes;          // Node8 array (80 B each)
    uint8_t* tris;           // TriRecord array (48 B each)
    uint32_t* tri_pos;       // [n] sorted position of the triangle that record i will hold (filled by the collapse, consumed by
                             // fill_tri_record): a compact array, so a node writes its ~6 positions into one or two sectors
                             // instead of one 4-byte word into each 48-byte record (a partial-sector write per triangle)
    uint32_t* wide_src;      // binary reference expanded by each wide node
    uint32_t* parent;        // (parent node << 3) | slot of each wide node, 0xffffffff for the root (refit)
    uint32_t* node_count;    // atomic allocators
    uint32_t* tri_count;
    uint32_t node_cap;
};

// Allocates the node's inner children and triangle records from the two global bump counters.  On the device the
// threads of a warp that arrive together make ONE atomic per counter (the leader adds the group's total, every
// thread takes its exclusive prefix): with one atomic per node the two counters - single addresses hit by every
// thread of the grid - serialise in the L2 atomic unit (2.6 M nodes x 2 atomics was most of the collapse time at
// 16.8 M triangles).
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void alloc_children(const CollapseOut& o, uint32_t n_inner, uint32_t n_tris, uint32_t& child_base,
                                               uint32_t& tri_base) {
    const unsigned m = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs((int)m) - 1;
    // exclusive prefix and total over the lanes that arrived together (the group may have holes: walk its members);
    // both counts ride in one 64-bit value (no carry: a warp allocates far fewer than 2^32 of either)
    const unsigned long long mine = ((unsigned long long)n_tris << 32) | n_inner;
    unsigned long long total = 0, excl = 0;
    for (unsigned rest = m; rest != 0u; rest &= rest - 1u) {
        const int src = __ffs((int)rest) - 1;
        const unsigned long long v = __shfl_sync(m, mine, src);
        if (src < lane) excl += v;
        total += v;
    }
    unsigned long long base = 0;
    if (lane == leader) {
        const uint32_t nb = (uint32_t)total ? atomicAdd(o.node_count, (uint32_t)total) : 0u;
        const uint32_t tb = (uint32_t)(total >> 32) ? atomicAdd(o.tri_count, (uint32_t)(total >> 32)) : 0u;
        base = ((unsigned long long)tb << 32) | nb;
    }
    base = __shfl_sync(m, base, leader);
    child_base = n_inner ? (uint32_t)base + (uint32_t)excl : 0u;
    tri_base = n_tris ? (uint32_t)(base >> 32) + (uint32_t)(excl >> 32) : 0u;
}
#else
inline void alloc_children(const CollapseOut& o, uint32_t n_inner, uint32_t n_tris, uint32_t& child_base, uint32_t& tri_base) {
    child_base = n_inner ? atomic_add_u32(o.node_count, n_inner) : 0u;
    tri_base = n_tris ? atomic_add_u32(o.tri_count, n_tris) : 0u;
}
#endif

// Builds wide node `w` from the binary subtree `wide_src[w]`.  Greedy surface-area expansion:
// starting from the two children, repeatedly replace the child with the largest box that is
// still expandable (an inner node covering more than leaf_max triangles) by its own two
// children until there are 8 children.  Subtrees with <= leaf_max triangles become leaf
// slots (their triangles are contiguous in Morton order).
// Quantisation of the child boxes of one wide node: frame (p, 2^e) from the node box, 8-bit planes
// rounded outwards and verified in binary64 against the exact decode p + q * 2^e.  Shared by the
// builder (collapse) and the refit path.  Absent slots get an inverted box.
// slot s holds boxes[idx_of_slot[s]] (present bit s set) or nothing
RT_HD void quantise_slots(const BBox& nb, const BBox* boxes, const int idx_of_slot[8], uint32_t present, Node8& nd) {
    const float p[3] = {nb.lx, nb.ly, nb.lz};
    const float hi3[3] = {nb.hx, nb.hy, nb.hz};
    uint32_t e[3];
    for (int a = 0; a < 3; ++a) {
        e[a] = quant_exponent(hi3[a] - p[a]);
        // make sure every child's upper plane is representable (<= 255 steps)
        for (;;) {
            const double sc = (double)exp2_biased(e[a]);
            bool ok = true;
            for (int s = 0; s < 8; ++s) {
                if (!((present >> s) & 1u)) continue;
                const BBox& sb = boxes[idx_of_slot[s]];
                const float ch = a == 0 ? sb.hx : (a == 1 ? sb.hy : sb.hz);
                if ((double)p[a] + 255.0 * sc < (double)ch) { ok = false; break; }
            }
            if (ok || e[a] >= 254u) break;
            ++e[a];
        }
    }
    nd.px = p[0]; nd.py = p[1]; nd.pz = p[2];
    nd.ex = (uint8_t)e[0]; nd.ey = (uint8_t)e[1]; nd.ez = (uint8_t)e[2];
    for (int s = 0; s < 8; ++s) {
        if (!((present >> s) & 1u)) {
            nd.qlox[s] = nd.qloy[s] = nd.qloz[s] = 255;   // inverted box: never hit
            nd.qhix[s] = nd.qhiy[s] = nd.qhiz[s] = 0;
            continue;
        }
        uint8_t ql[3], qh[3];
        const BBox sb = boxes[idx_of_slot[s]];
        for (int a = 0; a < 3; ++a) {
            const float cl = a == 0 ? sb.lx : (a == 1 ? sb.ly : sb.lz);
            const float ch = a == 0 ? sb.hx : (a == 1 ? sb.hy : sb.hz);
            const double sc = (double)exp2_biased(e[a]);
            const double isc = (double)exp2_biased(254u - e[a]);   // exact 1/sc (power of two): no double division
            double fl = floor(((double)cl - (double)p[a]) * isc);
            if (!(fl >= 0.0)) fl = 0.0;
            if (fl > 255.0) fl = 255.0;
            while (fl > 0.0 && (double)p[a] + fl * sc > (double)cl) fl -= 1.0;
            double fh = ceil(((double)ch - (double)p[a]) * isc);
            if (!(fh >= 0.0)) fh = 0.0;
            if (fh > 255.0) fh = 255.0;
            while (fh < 255.0 && (double)p[a] + fh * sc < (double)ch) fh += 1.0;
            ql[a] = (uint8_t)fl; qh[a] = (uint8_t)fh;
        }
        nd.qlox[s] = ql[0]; nd.qloy[s] = ql[1]; nd.qloz[s] = ql[2];
        nd.qhix[s] = qh[0]; nd.qhiy[s] = qh[1]; nd.qhiz[s] = qh[2];
    }
}

RT_HD int32_t clamp_index(int32_t i, int64_t n) { return i < 0 ? 0 : (i >= n ? (int32_t)(n - 1) : i); }

// 48-byte triangle record `slot` <- vertices of face `prim`
RT_HD void write_tri_record(uint8_t* tris, uint32_t slot, uint32_t prim, const float* __restrict__ verts, int64_t n_verts,
                            const int32_t* __restrict__ faces) {
    const int32_t i0 = clamp_index(faces[3 * (size_t)prim], n_verts), i1 = clamp_index(faces[3 * (size_t)prim + 1], n_verts),
                  i2 = clamp_index(faces[3 * (size_t)prim + 2], n_verts);
    TriRecord tr;
    tr.v0x = verts[3 * (size_t)i0]; tr.v0y = verts[3 * (size_t)i0 + 1]; tr.v0z = verts[3 * (size_t)i0 + 2];
    tr.v1x = verts[3 * (size_t)i1]; tr.v1y = verts[3 * (size_t)i1 + 1]; tr.v1z = verts[3 * (size_t)i1 + 2];
    tr.v2x = verts[3 * (size_t)i2]; tr.v2y = verts[3 * (size_t)i2 + 1]; tr.v2z = verts[3 * (size_t)i2 + 2];
    tr.prim = (int32_t)prim; tr.pad1 = 0; tr.pad2 = 0;
    *reinterpret_cast<TriRecord*>(tris + (size_t)slot * 48u) = tr;
}

// second half of the collapse: tri_pos[slot] is the sorted position of record `slot`; resolve it to the face and write the record
RT_HD void fill_tri_record(uint8_t* tris, uint32_t slot, const uint32_t* __restrict__ tri_pos, const uint32_t* __restrict__ sorted_prim,
                           const float* __restrict__ verts, int64_t n_verts, const int32_t* __restrict__ faces) {
    write_tri_record(tris, slot, sorted_prim[tri_pos[slot]], verts, n_verts, faces);
}

// Bottom-up update of one wide node after its children are final (refit): recomputes the slot
// boxes (leaf slots from their triangle records, inner slots from child_box[]), re-quantises and
// returns the node's own box.  Topology fields are untouched.
RT_HD BBox refit_node(uint8_t* nodes, const uint8_t* tris, uint32_t w, const BBox* child_box_of_node) {
    Node8 nd = *reinterpret_cast<const Node8*>(nodes + (size_t)w * 80u);
    BBox slot_box[8];
    int idx_of_slot[8];
    BBox nb; nb.lx = nb.ly = nb.lz = INFINITY; nb.hx = nb.hy = nb.hz = -INFINITY; nb.pad0 = nb.pad1 = 0.f;
    uint32_t present = 0, rel = 0, toff = 0;
    for (int s = 0; s < 8; ++s) {
        idx_of_slot[s] = s;
        const bool inner = (nd.imask >> s) & 1u;
        const uint32_t un = (nd.trimask >> (3 * s)) & 7u;
        if (inner) {
            slot_box[s] = load_box(child_box_of_node + nd.child_base + rel);
            ++rel;
        } else if (un) {
            const uint32_t cnt = un == 1u ? 1u : (un == 3u ? 2u : 3u);
            BBox b; b.lx = b.ly = b.lz = INFINITY; b.hx = b.hy = b.hz = -INFINITY; b.pad0 = b.pad1 = 0.f;
            for (uint32_t j = 0; j < cnt; ++j) {
                const float* tp = reinterpret_cast<const float*>(tris + (size_t)(nd.tri_base + toff + j) * 48u);
                b = bbox_union(b, tri_bbox(tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10]));
            }
            toff += cnt;
            slot_box[s] = b;
        } else {
            continue;
        }
        present |= 1u << s;
        nb = bbox_union(nb, slot_box[s]);
    }
    if (present == 0u) { nb.lx = nb.ly = nb.lz = 0.f; nb.hx = nb.hy = nb.hz = 0.f; }
    quantise_slots(nb, slot_box, idx_of_slot, present, nd);
    *reinterpret_cast<Node8*>(nodes + (size_t)w * 80u) = nd;
    return nb;
}

RT_HD bool bt_expandable(const BinaryTree& t, uint32_t ref) {
    return ref < (uint32_t)(t.n - 1) && bt_count(t, ref) > (uint32_t)t.leaf_max;
}
RT_HD float box_area(const BBox& b) {
    const float a = bbox_half_area(b);
    return a >= 0.0f ? a : 0.0f;   // NaN / negative -> 0
}
// child references of an inner binary node, stored as bit patterns in the pad words of its box record
#if defined(__CUDA_ARCH__)
RT_HD uint32_t box_left(const BBox& b) { return __float_as_uint(b.pad0); }
RT_HD uint32_t box_right(const BBox& b) { return __float_as_uint(b.pad1); }
#else
RT_HD uint32_t box_left(const BBox& b) { union { float f; uint32_t u; } c; c.f = b.pad0; return c.u; }
RT_HD uint32_t box_right(const BBox& b) { union { float f; uint32_t u; } c; c.f = b.pad1; return c.u; }
#endif
RT_HD void collapse_node(const BinaryTree& t, const CollapseOut& o, uint32_t w, const float* __restrict__ verts,
                         int64_t n_verts, const int32_t* __restrict__ faces) {
    uint32_t ref[8];
    float area[8];
    bool inner[8];
    BBox cb[8];        // (tried: in shared memory, one column per thread, to shrink the 700-byte stack frame - the kernel
                       //  moves 4 GB of DRAM at 16.8 M triangles - but 80 registers / 32 KB cost more occupancy than it saved)
    int k = 0;
    const uint32_t src = load_cg_u32(&o.wide_src[w]);
    const BBox nb = t.box[src];
    if (t.n <= (int64_t)t.leaf_max) {
        // whole mesh fits one leaf slot: root with a single leaf child
        ref[0] = src; area[0] = 0.0f; inner[0] = false; cb[0] = nb; k = 1;
    } else {
        // the box record of an inner binary node carries its two child references in the pad words
        // (written by the refit pass), so expanding a child costs no extra dependent load
        const uint32_t raw0 = box_left(nb), raw1 = box_right(nb);
        ref[0] = raw0 & kRefMask; ref[1] = raw1 & kRefMask; k = 2;
        inner[0] = t.flagged ? (raw0 >> 31) != 0u : bt_expandable(t, ref[0]);
        inner[1] = t.flagged ? (raw1 >> 31) != 0u : bt_expandable(t, ref[1]);
        for (int i = 0; i < 2; ++i) { cb[i] = t.box[ref[i]]; area[i] = box_area(cb[i]); }
        while (k < 8) {
            int best = -1; float ba = -1.0f;
            for (int i = 0; i < k; ++i)
                if (inner[i] && area[i] > ba) { best = i; ba = area[i]; }
            if (best < 0) break;
            const uint32_t lraw = box_left(cb[best]), rraw = box_right(cb[best]);
            const uint32_t l = lraw & kRefMask, r = rraw & kRefMask;
            ref[best] = l; cb[best] = t.box[l]; inner[best] = t.flagged ? (lraw >> 31) != 0u : bt_expandable(t, l); area[best] = box_area(cb[best]);
            ref[k] = r; cb[k] = t.box[r]; inner[k] = t.flagged ? (rraw >> 31) != 0u : bt_expandable(t, r); area[k] = box_area(cb[k]);
            ++k;
        }
        // free slots left: split multi-triangle leaves (largest box first) so that each triangle
        // gets a tighter slot box — the node test costs the same for 2 or 8 occupied slots
        while (k < 8) {
            int best = -1; float ba = -1.0f;
            for (int i = 0; i < k; ++i)
                if (!inner[i] && ref[i] < (uint32_t)(t.n - 1) && area[i] > ba) { best = i; ba = area[i]; }
            if (best < 0) break;
            const uint32_t l = box_left(cb[best]) & kRefMask, r = box_right(cb[best]) & kRefMask;
            ref[best] = l; cb[best] = t.box[l]; inner[best] = false; area[best] = box_area(cb[best]);
            ref[k] = r; cb[k] = t.box[r]; inner[k] = false; area[k] = box_area(cb[k]);
            ++k;
        }
    }
    // triangle count and first sorted position of every leaf child.  A leaf child is a single triangle or a binary
    // node over <= leaf_max of them; when both children of that node are leaves (always, at the default leaf_max of 2)
    // its range is read off the child references already loaded with its box - no first[] / last[] sector loads
    uint32_t n_inner = 0, n_tris = 0;
    uint32_t lcount[8], lfirst[8];
    const uint32_t leaf0 = (uint32_t)(t.n - 1);
    for (int i = 0; i < k; ++i) {
        if (inner[i]) { ++n_inner; lcount[i] = 0; lfirst[i] = 0; continue; }
        if (ref[i] >= leaf0) { lcount[i] = 1; lfirst[i] = ref[i] - leaf0; }
        else {
            const uint32_t cl = box_left(cb[i]) & kRefMask, cr = box_right(cb[i]) & kRefMask;
            if (cl >= leaf0 && cr >= leaf0) { lcount[i] = 2; lfirst[i] = cl - leaf0; }
            else { lcount[i] = bt_count(t, ref[i]); lfirst[i] = bt_first(t, ref[i]); }
        }
        n_tris += lcount[i];
    }
    // greedy slot assignment: child i goes to the free slot whose octant direction agrees
    // best with (child centre - node centre); traversal visits slots in ray-octant order.
    const float ncx = 0.5f * (nb.lx + nb.hx), ncy = 0.5f * (nb.ly + nb.hy), ncz = 0.5f * (nb.lz + nb.hz);
    int child_in_slot[8];
    for (int s = 0; s < 8; ++s) child_in_slot[s] = -1;
    for (int i = 0; i < k; ++i) {
        const float vx = 0.5f * (cb[i].lx + cb[i].hx) - ncx, vy = 0.5f * (cb[i].ly + cb[i].hy) - ncy,
                    vz = 0.5f * (cb[i].lz + cb[i].hz) - ncz;
        int bs = -1; float bsc = 0.0f;
        for (int s = 0; s < 8; ++s) {
            if (child_in_slot[s] >= 0) continue;
            const float sc = ((s & 1) ? vx : -vx) + ((s & 2) ? vy : -vy) + ((s & 4) ? vz : -vz);
            if (bs < 0 || sc > bsc) { bs = s; bsc = sc; }
        }
        child_in_slot[bs] = i;
    }
    uint32_t child_base, tri_base;
    alloc_children(o, n_inner, n_tris, child_base, tri_base);

    uint32_t present = 0;
    for (int s = 0; s < 8; ++s)
        if (child_in_slot[s] >= 0) present |= 1u << s;
    Node8 nd;
    quantise_slots(nb, cb, child_in_slot, present, nd);
    nd.child_base = child_base;
    nd.tri_base = tri_base;
    uint32_t imask = 0, trimask = 0, rel = 0, toff = 0;
    for (int s = 0; s < 8; ++s) {
        const int i = child_in_slot[s];
        if (i < 0) continue;
        if (inner[i]) {
            imask |= 1u << s;
            if (child_base + rel < o.node_cap) {
                o.wide_src[child_base + rel] = ref[i];
                o.parent[child_base + rel] = (w << 3) | (uint32_t)s;
            }
            ++rel;
        } else {
            const uint32_t cnt = lcount[i];
            const uint32_t unary = cnt == 1 ? 1u : (cnt == 2 ? 3u : 7u);
            trimask |= unary << (3 * s);
            const uint32_t f0 = lfirst[i];
            // only the SORTED POSITION of each triangle is recorded here (in tri_pos); the dependent gathers
            // position -> face -> vertices run afterwards in a fully parallel pass (fill_tri_record), not serially
            // inside this node's thread
            for (uint32_t j = 0; j < cnt; ++j) o.tri_pos[tri_base + toff + j] = f0 + j;
            toff += cnt;
        }
    }
    nd.imask = (uint8_t)imask;
    nd.trimask = trimask;
    nd.reserved = 0;
    if (w < o.node_cap) *reinterpret_cast<Node8*>(o.nodes + (size_t)w * 80u) = nd;
    if (w == 0) o.parent[0] = 0xffffffffu;
}

}  // namespace rt
