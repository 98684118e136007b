// scenepointsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the point queries of rt_scene.cuh (RT_HD, the code
// rt_scene_point.cu runs) on the CPU over a scene table prepared by scenesim.cpp (ss_prepare) on host blobs: the side
// array, closest point and signed distance with the top-level tree, with every instance in order and by brute force
// over every triangle of every instance, and the exhaustive check of the instance walk's world bound.  Never linked
// into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC scenepointsim.cpp -o libscenepointsim.so
#include "../../trimesh-ray-optix_b200/csrc/rt_scene.cuh"

using namespace rt;

// rt_scene_point_prepare: side = n_inst x 16 bytes
extern "C" void ss_point_prepare(const uint8_t* table, ScenePointSide* side) {
    const SceneView sv = scene_view(table);
    const int64_t n_inst = (int64_t)reinterpret_cast<const SceneHeader*>(table)->n_inst;
    for (int64_t i = 0; i < n_inst; ++i)
        side[i] = prepare_point_side(reinterpret_cast<const uint8_t*>(sv.blobs[sv.inst[i].mesh]), sv.inst[i]);
}

// Closest point (normals NULL) or signed distance (normals = host addresses of each mesh's pseudo-normal rows; sd
// written, distance not) over n dense points.  mode 0: the top-level tree (k_scene_point); 1: no top-level tree, every
// instance in order through the same leaf visit (box bound, instance walk); 2: brute force, every triangle of every
// instance through point_tri with no bound at all.
extern "C" int ss_point_query(const uint8_t* table, const uint8_t* tlas, const ScenePointSide* side, int mode, int64_t n,
                              const float* pts, float max_distance, const uint64_t* normals, float* closest, float* distance,
                              int32_t* inst_idx, int32_t* tri_idx, float* uv, float* sd) {
    const SceneView sv = scene_view(table);
    const int32_t n_inst = (int32_t)reinterpret_cast<const SceneHeader*>(table)->n_inst;
    const float max_d2 = normals ? INFINITY : fmul(max_distance, max_distance);
    for (int64_t r = 0; r < n; ++r) {
        ArrayStack<PointStackEntry> top, below;
        SceneTopSpace<ArrayStack<PointStackEntry>> sp{sv, side, &below};
        PointTrav t;
        point_init(t, pts[3 * r], pts[3 * r + 1], pts[3 * r + 2], max_d2);
        NoStats st;
        if (mode == 0) {
            const rt_blob_header* th = reinterpret_cast<const rt_blob_header*>(tlas);
            while (!point_step(tlas + th->nodes_offset, tlas + th->tris_offset, t, st, top, sp)) {}
        } else if (t.node != kNoNode && mode == 1) {
            for (int32_t i = 0; i < n_inst; ++i) {
                const SceneInst& s = sv.inst[i];
                if (box_point_lower(t.x, t.y, t.z, s.lo, s.hi) <= t.best) sp.visit(t, i);
            }
        } else if (t.node != kNoNode) {
            for (int32_t i = 0; i < n_inst; ++i) {
                const SceneInst& s = sv.inst[i];
                if (s.flags & kInstEmpty) continue;
                const uint8_t* blob = reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]);
                const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
                const uint8_t* tris = blob + h->tris_offset;
                for (uint32_t rec = 0; rec < h->n_tris; ++rec) {
                    const uint8_t* tp = tris + (size_t)rec * 48u;
                    const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
                    float w[9];
                    world_tri(s.fwd, a, b, c, w);
                    const PointHit ph = point_tri(t.x, t.y, t.z, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w[8]);
                    const int32_t prim = (int32_t)a.w;
                    if (ph.d2 < t.best || (ph.d2 == t.best && (sp.inst < 0 || i < sp.inst || (i == sp.inst && prim < sp.prim)))) {
                        t.best = ph.d2; sp.inst = i; sp.prim = prim; sp.slot = rec;
                    }
                }
            }
        }
        if (sp.inst >= 0) {
            float v[9];
            const PointHit h = scene_point_attr(sv, sp.inst, sp.slot, t.x, t.y, t.z, v);
            const float d = fsqrt(t.best);
            if (normals) {
                const SceneInst& s = sv.inst[sp.inst];
                sd[r] = scene_pseudonormal_sign(s, reinterpret_cast<const uint8_t*>(normals[s.mesh]), sp.slot, h, t.x, t.y,
                                                t.z, v, d);
            } else {
                distance[r] = d;
            }
            closest[3 * r] = h.cx; closest[3 * r + 1] = h.cy; closest[3 * r + 2] = h.cz;
            inst_idx[r] = sp.inst; tri_idx[r] = sp.prim; uv[2 * r] = h.w0; uv[2 * r + 1] = h.w1;
        } else {
            if (normals) sd[r] = -INFINITY;
            else distance[r] = INFINITY;
            closest[3 * r] = closest[3 * r + 1] = closest[3 * r + 2] = 0.0f;
            inst_idx[r] = tri_idx[r] = -1; uv[2 * r] = uv[2 * r + 1] = 0.0f;
        }
    }
    return 0;
}

// Exhaustive check of the instance walk's world bound: for every point, instance, node and non-empty slot, the bound
// InstanceSpace::bounds gives must not exceed the d2 point_tri computes for any world triangle below the slot (NaN d2
// excluded).  Also checks the top-level leaf bound against every world triangle of the instance.  out[0] = violations,
// out[1] = pairs checked; worst = largest bound / min d2 over pairs with d2 > 0.
namespace {
struct WorldBoundChecker {
    const uint8_t* nodes; const uint8_t* tris; InstanceSpace sp; PointTrav t;
    uint64_t violations = 0, checked = 0; double worst = 0.0;
    void count(float lb, float m) {
        if (!(m < INFINITY)) return;
        ++checked;
        if (!(lb <= m)) ++violations;
        if (m > 0.0f && (double)lb / (double)m > worst) worst = (double)lb / (double)m;
    }
    float walk(uint32_t idx) {
        const uint8_t* np = nodes + (size_t)idx * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48), n4 = ldg128(np + 64);
        float lb[8];
        sp.bounds(t, n0, n2, n3, n4, lb);
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
                    const uint8_t* tp = tris + (size_t)rec * 48u;
                    float w[9];
                    world_tri(sp.fwd, ldg128(tp), ldg128(tp + 16), ldg128(tp + 32), w);
                    const PointHit ph = point_tri(t.x, t.y, t.z, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], w[8]);
                    if (ph.d2 < m) m = ph.d2;
                }
            }
            count(lb[s], m);
            if (m < node_min) node_min = m;
        }
        return node_min;
    }
};
}  // namespace

extern "C" int ss_bound_check(const uint8_t* table, const ScenePointSide* side, int64_t n, const float* pts, uint64_t* out,
                              double* worst) {
    const SceneView sv = scene_view(table);
    const int32_t n_inst = (int32_t)reinterpret_cast<const SceneHeader*>(table)->n_inst;
    out[0] = out[1] = 0;
    *worst = 0.0;
    for (int64_t r = 0; r < n; ++r) {
        for (int32_t i = 0; i < n_inst; ++i) {
            const SceneInst& s = sv.inst[i];
            if (s.flags & kInstEmpty) continue;
            const uint8_t* blob = reinterpret_cast<const uint8_t*>(sv.blobs[s.mesh]);
            const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
            WorldBoundChecker c;
            c.nodes = blob + h->nodes_offset; c.tris = blob + h->tris_offset;
            point_init(c.t, pts[3 * r], pts[3 * r + 1], pts[3 * r + 2], INFINITY);
            // the same InstanceSpace scene_point_instance builds
            for (int k = 0; k < 12; ++k) c.sp.fwd[k] = s.fwd[k];
            c.sp.ox = affine_row(s.inv[0], s.inv[1], s.inv[2], s.inv[3], c.t.x, c.t.y, c.t.z);
            c.sp.oy = affine_row(s.inv[4], s.inv[5], s.inv[6], s.inv[7], c.t.x, c.t.y, c.t.z);
            c.sp.oz = affine_row(s.inv[8], s.inv[9], s.inv[10], s.inv[11], c.t.x, c.t.y, c.t.z);
            const float pmax = fmaxf(fmaxf(fabsf(c.t.x), fabsf(c.t.y)), fabsf(c.t.z));
            c.sp.sigma = side[i].sigma;
            c.sp.mu = fadd(side[i].alpha, fmul(side[i].beta, pmax));
            const float m = c.walk(0);
            c.count(box_point_lower(c.t.x, c.t.y, c.t.z, s.lo, s.hi), m);
            out[0] += c.violations; out[1] += c.checked;
            if (c.worst > *worst) *worst = c.worst;
        }
    }
    return 0;
}
