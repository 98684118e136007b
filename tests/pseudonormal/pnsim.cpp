// pnsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the pseudo-normal precompute of rt_pseudonormal.cu and the signed
// distance of rt_closest.cu on the CPU with their own RT_HD functions (rt_pseudonormal.cuh, rt_point.cuh), over a blob
// from tests/hostsim or a GPU blob copied to the host.  The onesweep sorts are replaced by std::stable_sort on the same
// keys: a stable sort of the same keys yields the same permutation.  Never linked into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC pnsim.cpp -o libpnsim.so
#include <algorithm>
#include <numeric>
#include <vector>
#include "../../include/raymesh_b200.h"
#include "../../trimesh-ray-optix_b200/csrc/rt_pseudonormal.cuh"

using namespace rt;

namespace {
std::vector<uint32_t> stable_order(const std::vector<uint64_t>& keys, std::vector<uint32_t> order) {
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    return order;
}
}  // namespace

// normals: n_tris x 96 bytes; counts = {boundary, non-manifold, inconsistent}
extern "C" int pn_normals(const uint8_t* blob, uint8_t* normals, uint64_t* counts) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* tris = blob + h->tris_offset;
    const uint32_t m = 3u * h->n_tris;
    counts[0] = counts[1] = counts[2] = 0;
    std::vector<uint64_t> kz(m, kPnNoKey), kxy(m, kPnNoKey);
    for (uint32_t c = 0; c < m; ++c) {
        float v[9];
        load_tri(tris, c / 3u, v);
        if (tri_finite(v)) { kz[c] = corner_key_z(v, c % 3u); kxy[c] = corner_key_xy(v, c % 3u); }
    }
    std::vector<uint32_t> order(m);
    std::iota(order.begin(), order.end(), 0u);
    const std::vector<uint32_t> sorted = stable_order(kxy, stable_order(kz, order));
    std::vector<uint32_t> vid(m);
    for (uint32_t j = 0; j < m; ++j) weld_run(tris, sorted.data(), m, j, vid.data(), normals);
    std::vector<uint64_t> ek(m);
    for (uint32_t e = 0; e < m; ++e) ek[e] = half_edge_key(vid.data(), e);
    const std::vector<uint32_t> es = stable_order(ek, order);
    std::vector<uint64_t> keys(m);
    for (uint32_t j = 0; j < m; ++j) keys[j] = ek[es[j]];
    for (uint32_t j = 0; j < m; ++j) {
        if (keys[j] == kPnNoKey) {
            store_row_slot(normals, es[j] / 3u, half_edge_slot(es[j] % 3u), 0.0f, 0.0f, 0.0f);
            continue;
        }
        if (!edge_head(keys.data(), j)) continue;
        const uint32_t cls = edge_class(edge_run(tris, es.data(), keys.data(), m, j, vid.data(), normals));
        if (cls < 3u) ++counts[cls];
    }
    return 0;
}

// signed distances of a dense [n,3] batch with the given normals; stats = {nodes, triangles, points, found}
extern "C" int pn_signed_distance(const uint8_t* blob, const uint8_t* normals, int64_t n, const float* pts, float* sd,
                                  uint64_t* stats) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* tris = blob + h->tris_offset;
    const uint8_t* nodes = blob + h->nodes_offset;
    uint64_t sn = 0, stt = 0, sf = 0;
    for (int64_t i = 0; i < n; ++i) {
        PointTrav t;
        point_init(t, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], INFINITY);
        ArrayStack<PointStackEntry> stack;
        Stats st;
        while (!point_step(nodes, tris, t, st, stack)) {}
        sn += st.nodes; stt += st.tris;
        if (t.prim != kNoPrim) {
            ++sf;
            float v[9];
            load_tri(tris, t.slot, v);
            const PointHit ph = point_tri(t.x, t.y, t.z, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
            sd[i] = pseudonormal_sign(normals, t.slot, ph, t.x, t.y, t.z, v, fsqrt(t.best));
        } else {
            sd[i] = -INFINITY;
        }
    }
    if (stats) { stats[0] = sn; stats[1] = stt; stats[2] = (uint64_t)n; stats[3] = sf; }
    return 0;
}

// point_tri's region code for one (point, triangle) pair
extern "C" uint32_t pn_region(const float* p, const float* v) {
    return point_tri(p[0], p[1], p[2], v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]).region;
}
