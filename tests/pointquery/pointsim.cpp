// pointsim.cpp — TEST INFRASTRUCTURE ONLY.  Steps the closest-point traversal of rt_point.cuh (RT_HD, the code
// k_closest_point runs) on the CPU over a blob built by tests/hostsim, and checks its lower bounds exhaustively.
// Never linked into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC pointsim.cpp -o libpointsim.so
#include <cstring>
#include <vector>
#include "../../include/raymesh_b200.h"
#include "../../trimesh-ray-optix_b200/csrc/rt_point.cuh"

using namespace rt;

namespace {
struct HostPointStack {
    PointStackEntry e[kMaxDepth];
    int max_sp = 0;
    void push(int sp, const PointStackEntry& v) { e[sp] = v; if (sp + 1 > max_sp) max_sp = sp + 1; }
    void pop(int sp, PointStackEntry& v) { v = e[sp]; }
};
}  // namespace

// Same outputs as rt_closest_point for a dense [n,3] batch; stats = {nodes, triangles, points, found}, max_stack = deepest
// group stack seen.
extern "C" int hs_closest_point(const uint8_t* blob, int64_t n, const float* pts, float max_distance, float* closest,
                                float* distance, int32_t* tri, float* uv, uint64_t* stats, int32_t* max_stack) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* tris = blob + h->tris_offset;
    const uint8_t* nodes = blob + h->nodes_offset;
    uint64_t sn = 0, stt = 0, sf = 0;
    int ms = 0;
    for (int64_t i = 0; i < n; ++i) {
        PointTrav t;
        point_init(t, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], fmul(max_distance, max_distance));
        HostPointStack stack;
        Stats st;
        while (!point_step(nodes, tris, t, st, stack)) {}
        sn += st.nodes; stt += st.tris;
        if (stack.max_sp > ms) ms = stack.max_sp;
        if (t.prim != kNoPrim) {
            ++sf;
            const float* tp = reinterpret_cast<const float*>(tris + (size_t)t.slot * 48u);
            const PointHit ph = point_tri(t.x, t.y, t.z, tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10]);
            closest[3 * i] = ph.cx; closest[3 * i + 1] = ph.cy; closest[3 * i + 2] = ph.cz;
            distance[i] = fsqrt(t.best); tri[i] = t.prim; uv[2 * i] = ph.w0; uv[2 * i + 1] = ph.w1;
        } else {
            closest[3 * i] = closest[3 * i + 1] = closest[3 * i + 2] = 0.0f;
            distance[i] = INFINITY; tri[i] = -1; uv[2 * i] = uv[2 * i + 1] = 0.0f;
        }
    }
    if (stats) { stats[0] = sn; stats[1] = stt; stats[2] = (uint64_t)n; stats[3] = sf; }
    if (max_stack) *max_stack = ms;
    return 0;
}

// Exhaustive check of slot_lower_bounds: for every point, node and non-empty slot, the bound must not exceed the d2
// point_tri computes for any triangle below the slot (NaN d2 excluded: such triangles are never selected).
// out[0] = violations, out[1] = slot/subtree pairs checked; worst[0] = largest bound / min d2 over pairs with d2 > 0.
namespace {
struct BoundChecker {
    const uint8_t* nodes; const uint8_t* tris; float x, y, z;
    uint64_t violations = 0, checked = 0; double worst = 0.0;
    // smallest non-NaN d2 of the subtree of node `idx` (+inf when none)
    float walk(uint32_t idx) {
        const uint8_t* np = nodes + (size_t)idx * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48), n4 = ldg128(np + 64);
        float lb[8];
        slot_lower_bounds(x, y, z, n0, n2, n3, n4, lb);
        const uint32_t imask = n0.w >> 24, tmask = n1.z;
        float node_min = INFINITY;
        uint32_t rel = 0;
        for (int s = 0; s < 8; ++s) {
            const bool inner = (imask >> s) & 1u;
            const uint32_t un = (tmask >> (3 * s)) & 7u;
            if (!inner && un == 0u) continue;
            float m = INFINITY;
            if (inner) {
                m = walk(n1.x + rel);
                ++rel;
            } else {
                uint32_t rec = n1.y + (uint32_t)popc32(tmask & ((1u << (3 * s)) - 1u));
                for (int j = 0; j < popc32(un); ++j, ++rec) {
                    const float* tp = reinterpret_cast<const float*>(tris + (size_t)rec * 48u);
                    const PointHit ph = point_tri(x, y, z, tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10]);
                    if (ph.d2 < m) m = ph.d2;
                }
            }
            if (m < INFINITY) {
                ++checked;
                if (!(lb[s] <= m)) ++violations;
                if (m > 0.0f && (double)lb[s] / (double)m > worst) worst = (double)lb[s] / (double)m;
            }
            if (m < node_min) node_min = m;
        }
        return node_min;
    }
};
}  // namespace

extern "C" int hs_slot_bounds_check(const uint8_t* blob, int64_t n, const float* pts, uint64_t* out, double* worst) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    out[0] = out[1] = 0;
    *worst = 0.0;
    for (int64_t i = 0; i < n; ++i) {
        BoundChecker c;
        c.nodes = blob + h->nodes_offset; c.tris = blob + h->tris_offset;
        c.x = pts[3 * i]; c.y = pts[3 * i + 1]; c.z = pts[3 * i + 2];
        c.walk(0);
        out[0] += c.violations; out[1] += c.checked;
        if (c.worst > *worst) *worst = c.worst;
    }
    return 0;
}

// point_tri for one (point, triangle) pair: out = {cx, cy, cz, d2, w0, w1}
extern "C" void hs_point_tri(const float* p, const float* v, float* out) {
    const PointHit h = point_tri(p[0], p[1], p[2], v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
    out[0] = h.cx; out[1] = h.cy; out[2] = h.cz; out[3] = h.d2; out[4] = h.w0; out[5] = h.w1;
}
