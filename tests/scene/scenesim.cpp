// scenesim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the instance preparation and the two-level walk of rt_scene.cuh (RT_HD,
// the code rt_scene.cu runs) on the CPU, over blobs from tests/hostsim or GPU blobs copied to the host, plus a
// brute-force mode that skips the top-level tree and walks every instance.  Never linked into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC scenesim.cpp -o libscenesim.so
#include <cstring>
#include "../../trimesh-ray-optix_b200/csrc/rt_scene.cuh"

using namespace rt;

namespace {
struct HostStack {
    uint32_t x[kMaxDepth], y[kMaxDepth];
    void push(int sp, uint32_t a, uint32_t b) { x[sp] = a; y[sp] = b; }
    void pop(int sp, uint32_t& a, uint32_t& b) { a = x[sp]; b = y[sp]; }
};
size_t align256(size_t x) { return (x + 255) / 256 * 256; }
size_t inst_offset() { return 256; }
size_t blobs_offset(int64_t n_inst) { return align256(256 + (size_t)n_inst * sizeof(SceneInst)); }
}  // namespace

// rt_scene_prepare_sizes
extern "C" size_t ss_table_bytes(int64_t n_meshes, int64_t n_inst) { return align256(blobs_offset(n_inst) + (size_t)n_meshes * 8u); }

// rt_scene_prepare with host blobs: the same checks (-1 = a bad mesh index or transform, nothing written), then
// prepare_instance for every instance.  blob_addrs: host addresses of the M blobs.
extern "C" int ss_prepare(int64_t n_meshes, const uint64_t* blob_addrs, int64_t n_inst, const int32_t* inst_mesh,
                          const float* transforms, uint8_t* table, float* tlas_v, int32_t* tlas_f) {
    for (int64_t i = 0; i < n_inst; ++i) {
        SceneInst s;
        for (int k = 0; k < 12; ++k) s.fwd[k] = transforms[12 * i + k];
        double det, kappa;
        if (inst_mesh[i] < 0 || inst_mesh[i] >= n_meshes || !invert_transform(s.fwd, s.inv, &det, &kappa)) return -1;
    }
    SceneHeader h = {};
    h.n_meshes = (uint64_t)n_meshes; h.n_inst = (uint64_t)n_inst; h.inst_offset = inst_offset(); h.blobs_offset = blobs_offset(n_inst);
    memcpy(table, &h, sizeof(h));
    memcpy(table + h.blobs_offset, blob_addrs, (size_t)n_meshes * 8u);
    SceneInst* inst = reinterpret_cast<SceneInst*>(table + h.inst_offset);
    for (int64_t i = 0; i < n_inst; ++i) {
        SceneInst s;
        memset(&s, 0, sizeof(s));
        s.mesh = inst_mesh[i];
        for (int k = 0; k < 12; ++k) s.fwd[k] = transforms[12 * i + k];
        prepare_instance(reinterpret_cast<const uint8_t*>(blob_addrs[s.mesh]), s, (uint32_t)i, tlas_v + 6 * i, tlas_f + 3 * i);
        inst[i] = s;
    }
    return 0;
}

// mode 0 closest, 1 any, 2 count over n dense rays.  tlas = the top-level blob, or NULL for the brute-force loop over
// every instance (each walked on its own from tmax, the answers combined by the same key / OR / sum).
extern "C" int ss_trace(const uint8_t* table, const uint8_t* tlas, int mode, int64_t n, const float* o, const float* d,
                        float tmax, uint8_t* hit, uint8_t* front, int32_t* inst_idx, int32_t* tri_idx, float* loc, float* uv,
                        int32_t* count) {
    const SceneView sv = scene_view(table);
    const int64_t n_inst = (int64_t)reinterpret_cast<const SceneHeader*>(table)->n_inst;
    for (int64_t r = 0; r < n; ++r) {
        const float w[6] = {o[3 * r], o[3 * r + 1], o[3 * r + 2], d[3 * r], d[3 * r + 1], d[3 * r + 2]};
        HostStack top, below;
        SceneClosest<HostStack> vc{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, tmax};
        SceneAny<HostStack> va{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, tmax};
        SceneCount<HostStack> vn{sv, {w[0], w[1], w[2], w[3], w[4], w[5]}, tmax};
        vc.stack = va.stack = vn.stack = &below;
        if (tlas) {
            const rt_blob_header* th = reinterpret_cast<const rt_blob_header*>(tlas);
            Ray wr;
            ray_setup(wr, w[0], w[1], w[2], w[3], w[4], w[5]);
            Trav t;
            trav_init(t);
            if (mode == 0) while (!scene_step(tlas + th->nodes_offset, tlas + th->tris_offset, wr, vc, top, t)) {}
            else if (mode == 1) while (!scene_step(tlas + th->nodes_offset, tlas + th->tris_offset, wr, va, top, t)) {}
            else while (!scene_step(tlas + th->nodes_offset, tlas + th->tris_offset, wr, vn, top, t)) {}
        } else {
            for (int32_t i = 0; i < (int32_t)n_inst; ++i) {
                Ray ir;
                const uint8_t *nodes, *tris;
                if (!instance_ray(sv, i, w, ir, nodes, tris)) continue;
                if (mode == 0) {
                    ClosestVisitor<NoStats> vis(tmax);
                    traverse(nodes, tris, ir, vis, below);
                    if (vis.prim >= 0 && (vc.inst < 0 || vis.tmax < vc.tmax ||
                                          (vis.tmax == vc.tmax && (i < vc.inst || (i == vc.inst && vis.prim < vc.prim))))) {
                        vc.tmax = vis.tmax; vc.inst = i; vc.prim = vis.prim; vc.slot = vis.slot;
                    }
                } else if (mode == 1) {
                    AnyVisitor<NoStats> vis(tmax);
                    traverse(nodes, tris, ir, vis, below);
                    va.found = va.found || vis.found;
                } else {
                    CountVisitor<NoStats> vis(tmax);
                    traverse(nodes, tris, ir, vis, below);
                    vn.count += vis.count;
                }
            }
        }
        if (mode == 0) {
            if (vc.inst >= 0) {
                const SceneHitOut a = scene_hit_attr(sv, vc.inst, vc.slot, w);
                hit[r] = 1; front[r] = a.front ? 1 : 0; inst_idx[r] = vc.inst; tri_idx[r] = vc.prim;
                for (int k = 0; k < 3; ++k) loc[3 * r + k] = a.loc[k];
                uv[2 * r] = a.uv[0]; uv[2 * r + 1] = a.uv[1];
            } else {
                hit[r] = 0; front[r] = 0; inst_idx[r] = -1; tri_idx[r] = -1;
                for (int k = 0; k < 3; ++k) loc[3 * r + k] = 0.0f;
                uv[2 * r] = uv[2 * r + 1] = 0.0f;
            }
        } else if (mode == 1) {
            hit[r] = va.found ? 1 : 0;
        } else {
            count[r] = vn.count;
        }
    }
    return 0;
}

// affine_row over n triples (the binary32 transform sequence, for the identity and sign-of-zero tests)
extern "C" void ss_affine_row(int64_t n, const float* m, const float* xyz, float* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = affine_row(m[0], m[1], m[2], m[3], xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
}
