// hostsim.cpp — TEST INFRASTRUCTURE ONLY.  Host-side single-threaded stepping of the product's
// per-element device functions (rt_core.cuh / rt_traverse.cuh / rt_build_core.cuh, which are
// __host__ __device__) so that the builder and traversal LOGIC can be checked against the oracle
// in the CPU-only test tier, and so that a blob produced on the GPU can be validated structurally
// (hs_check_blob).  It is compiled into tests/hostsim/libhostsim.so by tests; it is never linked
// into libtriro_b200.so and nothing under trimesh-ray-optix_b200/ refers to it: the product has
// no CPU path.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC hostsim.cpp -o libhostsim.so
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>
#include "../../include/raymesh_b200.h"
#include "../../trimesh-ray-optix_b200/csrc/rt_build_core.cuh"
#include "../../trimesh-ray-optix_b200/csrc/rt_traverse.cuh"

using namespace rt;

namespace {
size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
// same rule as rt_api.h: kLeafTrisDefault, or TRIRO_LEAF_TRIS=1..3 (read at every call here, so tests can switch it)
int leaf_setting() {
    const char* e = getenv("TRIRO_LEAF_TRIS");
    const int x = e ? atoi(e) : kLeafTrisDefault;
    return x < 1 ? 1 : (x > kLeafMaxTris ? kLeafMaxTris : x);
}
// rt_api.h blob_layout: the allocation holds node_cap nodes and parent links; the links of the nodes in use are placed
// right behind those nodes (parents_offset_for)
struct Layout { size_t tris_offset, nodes_offset, total; uint32_t node_cap; };
Layout layout(int64_t n) {
    Layout l;
    l.tris_offset = RT_BLOB_HEADER_BYTES;
    l.nodes_offset = align_up(l.tris_offset + (size_t)n * 48u, 256);
    l.node_cap = wide_node_cap(n, leaf_setting());
    l.total = align_up(l.nodes_offset + (size_t)l.node_cap * 80u, 256) + align_up((size_t)l.node_cap * 4u, 256);
    return l;
}
struct VecStack {
    uint32_t x[kMaxDepth], y[kMaxDepth];
    int max_sp = 0;
    void push(int sp, uint32_t a, uint32_t b) { x[sp] = a; y[sp] = b; if (sp + 1 > max_sp) max_sp = sp + 1; }
    void pop(int sp, uint32_t& a, uint32_t& b) { a = x[sp]; b = y[sp]; }
};
void tri_verts(const float* verts, int64_t nv, const int32_t* faces, int64_t prim, float v[9]) {
    for (int c = 0; c < 3; ++c) {
        const int32_t i = clamp_index(faces[3 * prim + c], nv);
        v[3 * c] = verts[3 * (size_t)i]; v[3 * c + 1] = verts[3 * (size_t)i + 1]; v[3 * c + 2] = verts[3 * (size_t)i + 2];
    }
}
}  // namespace

extern "C" size_t hs_blob_bytes(int64_t n_faces) { return layout(n_faces).total; }

// Same pipeline as rt_bvh_build, one element at a time, and the same blob: k_scene_bounds (ordered-uint bounds and the
// bad-index count), k_morton (keys cut to morton_axis_bits(n) bits per axis), the stable sort, k_karras, k_refit (child
// references with the bit-31 "covers more than leaf_max triangles" flag in the box pads), k_collapse run with
// flagged = 1, k_fill_tris, k_place_parents (parent links right behind the nodes in use) and k_finalize (header, zeroed
// gaps).  Only the numbering of nodes and records may differ from a GPU build (hs_canonical removes that difference).
extern "C" int hs_build(const float* verts, int64_t nv, const int32_t* faces, int64_t n, uint8_t* blob, size_t blob_bytes) {
    const Layout lay = layout(n);
    if (blob_bytes < lay.total) return -3;
    memset(blob, 0, lay.total);
    rt_blob_header h;
    memset(&h, 0, sizeof(h));
    h.magic = RT_BLOB_MAGIC; h.abi_version = RT_ABI_VERSION; h.n_tris = (uint32_t)n; h.n_nodes_cap = lay.node_cap;
    h.tris_offset = lay.tris_offset; h.nodes_offset = lay.nodes_offset;
    if (n == 0) {
        Node8 nd; memset(&nd, 0, sizeof(nd)); nd.ex = nd.ey = nd.ez = 1;
        memcpy(blob + lay.nodes_offset, &nd, 80);
        h.n_nodes = 1; h.depth = 1;
        h.parents_offset = parents_offset_for(lay.nodes_offset, 1);
        h.used_bytes = used_bytes_for(h.parents_offset, 1);
        const uint32_t root = 0xffffffffu;
        memcpy(blob + h.parents_offset, &root, 4);
        memcpy(blob, &h, sizeof(h));
        return 0;
    }
    // scene bounds (ordered-uint encoding, like k_scene_bounds) + Morton codes
    uint32_t olo[3] = {kOrdPosInf, kOrdPosInf, kOrdPosInf}, ohi[3] = {kOrdNegInf, kOrdNegInf, kOrdNegInf};
    uint32_t bad = 0;
    std::vector<BBox> tb((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        float v[9]; tri_verts(verts, nv, faces, i, v);
        bool ok = true;
        for (int c = 0; c < 3; ++c) ok = ok && faces[3 * i + c] >= 0 && faces[3 * i + c] < nv;
        bad += ok ? 0u : 1u;
        tb[i] = tri_bbox(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
        olo[0] = std::min(olo[0], ord_lo(tb[i].lx)); olo[1] = std::min(olo[1], ord_lo(tb[i].ly)); olo[2] = std::min(olo[2], ord_lo(tb[i].lz));
        ohi[0] = std::max(ohi[0], ord_hi(tb[i].hx)); ohi[1] = std::max(ohi[1], ord_hi(tb[i].hy)); ohi[2] = std::max(ohi[2], ord_hi(tb[i].hz));
    }
    float lo[3], hi[3], inv[3];
    for (int a = 0; a < 3; ++a) { lo[a] = ord2f(olo[a]); hi[a] = ord2f(ohi[a]); }
    morton_scale(lo, hi, inv);
    const int drop = 3 * (21 - morton_axis_bits(n));
    std::vector<uint64_t> keys((size_t)n);
    std::vector<uint32_t> vals((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        keys[i] = morton63(0.5f * (tb[i].lx + tb[i].hx), 0.5f * (tb[i].ly + tb[i].hy), 0.5f * (tb[i].lz + tb[i].hz), lo, inv) >> drop;
        vals[i] = (uint32_t)i;
    }
    std::stable_sort(vals.begin(), vals.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    std::vector<uint64_t> skeys((size_t)n);
    for (int64_t i = 0; i < n; ++i) skeys[i] = keys[vals[i]];
    // hierarchy
    const size_t ni = (size_t)(n - 1);
    std::vector<uint32_t> left(ni), right(ni), first(ni), last(ni), parent((size_t)2 * n, 0xffffffffu), flags(ni, 0);
    for (int64_t i = 0; i < n - 1; ++i) {
        const KarrasNode k = karras_node(skeys.data(), n, i);
        left[i] = k.left; right[i] = k.right; first[i] = k.first; last[i] = k.last;
        parent[k.left] = (uint32_t)i; parent[k.right] = (uint32_t)i;
    }
    // refit: child references ride in the pads, bit 31 set when the child covers more than leaf_max triangles
    const uint32_t leaf_max = (uint32_t)leaf_setting();
    auto count = [&](uint32_t ref) { return ref >= (uint32_t)(n - 1) ? 1u : last[ref] - first[ref] + 1u; };
    std::vector<BBox> box((size_t)2 * n);
    for (int64_t k = 0; k < n; ++k) {
        box[(n - 1) + k] = leaf_bbox(tb[vals[k]]);
        if (n == 1) continue;
        uint32_t cur = parent[(n - 1) + k];
        for (;;) {
            if (flags[cur]++ == 0) break;
            box[cur] = bbox_union(box[left[cur]], box[right[cur]]);
            const uint32_t l = left[cur] | (count(left[cur]) > leaf_max ? 0x80000000u : 0u);
            const uint32_t r = right[cur] | (count(right[cur]) > leaf_max ? 0x80000000u : 0u);
            memcpy(&box[cur].pad0, &l, 4); memcpy(&box[cur].pad1, &r, 4);
            if (cur == 0) break;
            cur = parent[cur];
        }
    }
    // collapse, level by level
    std::vector<uint32_t> wide_src(lay.node_cap, 0), wide_parent(lay.node_cap, 0);
    uint32_t node_count = 1, tri_count = 0;
    BinaryTree t; t.n = n; t.left = left.data(); t.right = right.data(); t.first = first.data(); t.last = last.data();
    t.box = box.data(); t.sorted_prim = vals.data(); t.leaf_max = (int)leaf_max; t.flagged = 1;
    std::vector<uint32_t> tri_pos((size_t)n, 0);
    CollapseOut o; o.nodes = blob + lay.nodes_offset; o.tris = blob + lay.tris_offset; o.wide_src = wide_src.data(); o.tri_pos = tri_pos.data();
    o.node_count = &node_count; o.tri_count = &tri_count; o.node_cap = lay.node_cap; o.parent = wide_parent.data();
    uint32_t begin = 0, end = 1, depth = 0;
    while (begin < end) {
        for (uint32_t w = begin; w < end; ++w) collapse_node(t, o, w, verts, nv, faces);
        ++depth;
        begin = end;
        end = node_count < lay.node_cap ? node_count : lay.node_cap;
    }
    for (int64_t i = 0; i < n; ++i) fill_tri_record(blob + lay.tris_offset, (uint32_t)i, tri_pos.data(), vals.data(), verts, nv, faces);
    h.n_nodes = node_count < lay.node_cap ? node_count : lay.node_cap; h.depth = depth;
    h.parents_offset = parents_offset_for(lay.nodes_offset, h.n_nodes);
    h.used_bytes = used_bytes_for(h.parents_offset, h.n_nodes);
    memcpy(blob + h.parents_offset, wide_parent.data(), (size_t)h.n_nodes * 4u);
    for (int a = 0; a < 3; ++a) { h.aabb_lo[a] = lo[a]; h.aabb_hi[a] = hi[a]; }
    h.bad_index_faces = bad;
    h.node_overflow = node_count > lay.node_cap ? 1u : 0u;
    memcpy(blob, &h, sizeof(h));
    return 0;
}

// EXPERIMENT HOOK: same as hs_build, but the binary topology comes from a top-down binned-SAH
// builder (16 bins, centroid bounds) instead of Morton order + Karras.  Used to measure how much
// of the traversal cost is tree quality (tools/sah_probe.py); the product builds LBVH only.
namespace {
struct SahBuilder {
    const std::vector<BBox>& tb; std::vector<uint32_t>& order;
    std::vector<uint32_t>&left, &right, &first, &last; uint32_t next = 0; int64_t n;
    // returns ref of the subtree over order[lo..hi] (inclusive)
    uint32_t build(uint32_t lo, uint32_t hi, uint32_t self) {
        if (lo == hi) return (uint32_t)(n - 1) + lo;
        float cl[3] = {INFINITY, INFINITY, INFINITY}, ch[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (uint32_t i = lo; i <= hi; ++i) {
            const BBox& b = tb[order[i]];
            const float c[3] = {0.5f * (b.lx + b.hx), 0.5f * (b.ly + b.hy), 0.5f * (b.lz + b.hz)};
            for (int a = 0; a < 3; ++a) { cl[a] = fminf(cl[a], c[a]); ch[a] = fmaxf(ch[a], c[a]); }
        }
        constexpr int NB = 16;
        float best = INFINITY; int best_axis = -1, best_split = 0;
        for (int a = 0; a < 3; ++a) {
            const float ext = ch[a] - cl[a];
            if (!(ext > 0.0f)) continue;
            BBox bb[NB]; uint32_t cnt[NB] = {0};
            for (auto& b : bb) { b.lx = b.ly = b.lz = INFINITY; b.hx = b.hy = b.hz = -INFINITY; b.pad0 = b.pad1 = 0; }
            for (uint32_t i = lo; i <= hi; ++i) {
                const BBox& b = tb[order[i]];
                const float c = a == 0 ? 0.5f * (b.lx + b.hx) : a == 1 ? 0.5f * (b.ly + b.hy) : 0.5f * (b.lz + b.hz);
                int k = (int)((c - cl[a]) / ext * NB); if (k >= NB) k = NB - 1; if (k < 0) k = 0;
                bb[k] = bbox_union(bb[k], b); ++cnt[k];
            }
            float la[NB], ra[NB]; uint32_t lc[NB], rc[NB];
            BBox acc = bb[0]; uint32_t c = 0;
            for (int k = 0; k < NB; ++k) { if (k == 0) acc = bb[0]; else acc = bbox_union(acc, bb[k]); c += cnt[k]; la[k] = c ? bbox_half_area(acc) : 0.f; lc[k] = c; }
            c = 0;
            for (int k = NB - 1; k >= 0; --k) { if (k == NB - 1) acc = bb[k]; else acc = bbox_union(acc, bb[k]); c += cnt[k]; ra[k] = c ? bbox_half_area(acc) : 0.f; rc[k] = c; }
            for (int k = 0; k + 1 < NB; ++k) {
                if (lc[k] == 0 || rc[k + 1] == 0) continue;
                const float cost = la[k] * lc[k] + ra[k + 1] * rc[k + 1];
                if (cost < best) { best = cost; best_axis = a; best_split = k; }
            }
        }
        uint32_t mid;
        if (best_axis < 0) mid = lo + (hi - lo) / 2;      // all centroids equal: split in the middle
        else {
            const int a = best_axis; const float ext = ch[a] - cl[a];
            auto it = std::stable_partition(order.begin() + lo, order.begin() + hi + 1, [&](uint32_t id) {
                const BBox& b = tb[id];
                const float c = a == 0 ? 0.5f * (b.lx + b.hx) : a == 1 ? 0.5f * (b.ly + b.hy) : 0.5f * (b.lz + b.hz);
                int k = (int)((c - cl[a]) / ext * 16); if (k >= 16) k = 15; if (k < 0) k = 0;
                return k <= best_split; });
            mid = (uint32_t)(it - order.begin()) - 1;
            if (mid < lo || mid >= hi) mid = lo + (hi - lo) / 2;
        }
        first[self] = lo; last[self] = hi;
        const uint32_t ls = (mid > lo) ? ++next : 0, rs = (hi > mid + 1) ? ++next : 0;
        left[self] = build(lo, mid, ls);
        right[self] = build(mid + 1, hi, rs);
        return self;
    }
};
}  // namespace

extern "C" int hs_build_sah(const float* verts, int64_t nv, const int32_t* faces, int64_t n, uint8_t* blob, size_t blob_bytes) {
    const Layout lay = layout(n);
    if (blob_bytes < lay.total || n < 2) return -3;
    memset(blob, 0, lay.total);
    rt_blob_header h;
    memset(&h, 0, sizeof(h));
    h.magic = RT_BLOB_MAGIC; h.abi_version = RT_ABI_VERSION; h.n_tris = (uint32_t)n; h.n_nodes_cap = lay.node_cap;
    h.tris_offset = lay.tris_offset; h.nodes_offset = lay.nodes_offset;
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    std::vector<BBox> tb((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        float v[9]; tri_verts(verts, nv, faces, i, v);
        tb[i] = tri_bbox(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]);
        lo[0] = fminf(lo[0], tb[i].lx); lo[1] = fminf(lo[1], tb[i].ly); lo[2] = fminf(lo[2], tb[i].lz);
        hi[0] = fmaxf(hi[0], tb[i].hx); hi[1] = fmaxf(hi[1], tb[i].hy); hi[2] = fmaxf(hi[2], tb[i].hz);
    }
    std::vector<uint32_t> vals((size_t)n);
    std::iota(vals.begin(), vals.end(), 0u);
    const size_t ni = (size_t)(n - 1);
    std::vector<uint32_t> left(ni), right(ni), first(ni), last(ni);
    SahBuilder sb{tb, vals, left, right, first, last, 0, n};
    sb.build(0, (uint32_t)(n - 1), 0);
    // boxes bottom-up (post-order via explicit recursion on the finished topology)
    std::vector<BBox> box((size_t)2 * n);
    for (int64_t k = 0; k < n; ++k) box[(n - 1) + k] = tb[vals[k]];
    std::vector<uint32_t> stack{0}; std::vector<uint32_t> post;
    while (!stack.empty()) { const uint32_t c = stack.back(); stack.pop_back(); post.push_back(c);
        if (left[c] < ni) stack.push_back(left[c]); if (right[c] < ni) stack.push_back(right[c]); }
    for (auto it = post.rbegin(); it != post.rend(); ++it) {
        const uint32_t c = *it;
        box[c] = bbox_union(box[left[c]], box[right[c]]);
        memcpy(&box[c].pad0, &left[c], 4); memcpy(&box[c].pad1, &right[c], 4);
    }
    std::vector<uint32_t> wide_src(lay.node_cap, 0), wide_parent(lay.node_cap, 0);
    uint32_t node_count = 1, tri_count = 0;
    BinaryTree t; t.n = n; t.left = left.data(); t.right = right.data(); t.first = first.data(); t.last = last.data();
    t.box = box.data(); t.sorted_prim = vals.data(); t.leaf_max = leaf_setting(); t.flagged = 0;
    std::vector<uint32_t> tri_pos((size_t)n, 0);
    CollapseOut o; o.nodes = blob + lay.nodes_offset; o.tris = blob + lay.tris_offset; o.wide_src = wide_src.data(); o.tri_pos = tri_pos.data();
    o.node_count = &node_count; o.tri_count = &tri_count; o.node_cap = lay.node_cap;
    o.parent = wide_parent.data();
    uint32_t begin = 0, end = 1, depth = 0;
    while (begin < end) {
        for (uint32_t w = begin; w < end; ++w) collapse_node(t, o, w, verts, nv, faces);
        ++depth;
        begin = end;
        end = node_count < lay.node_cap ? node_count : lay.node_cap;
    }
    for (int64_t i = 0; i < n; ++i) fill_tri_record(blob + lay.tris_offset, (uint32_t)i, tri_pos.data(), vals.data(), verts, nv, faces);
    h.n_nodes = node_count < lay.node_cap ? node_count : lay.node_cap; h.depth = depth;
    h.parents_offset = parents_offset_for(lay.nodes_offset, h.n_nodes);     // the product's layout, like hs_build
    h.used_bytes = used_bytes_for(h.parents_offset, h.n_nodes);
    memcpy(blob + h.parents_offset, wide_parent.data(), (size_t)h.n_nodes * 4u);
    for (int a = 0; a < 3; ++a) { h.aabb_lo[a] = lo[a]; h.aabb_hi[a] = hi[a]; }
    h.node_overflow = node_count > lay.node_cap ? 1u : 0u;
    memcpy(blob, &h, sizeof(h));
    return 0;
}

// mode: 0 closest (writes hit/front/tri/loc/uv), 1 any (hit), 2 count (count).  stats[0..3] as rt_trace_stats.
extern "C" int hs_trace(const uint8_t* blob, int mode, int64_t nray, const float* o, const float* d, uint8_t* hit,
                        uint8_t* front, int32_t* tri, float* loc, float* uv, int32_t* count, uint64_t* stats,
                        int32_t* max_stack) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* tris = blob + h->tris_offset;
    const uint8_t* nodes = blob + h->nodes_offset;
    uint64_t sn = 0, st = 0, sh = 0;
    int ms = 0;
    for (int64_t r = 0; r < nray; ++r) {
        Ray ray;
        ray_setup(ray, o[3 * r], o[3 * r + 1], o[3 * r + 2], d[3 * r], d[3 * r + 1], d[3 * r + 2]);
        VecStack stack;
        if (mode == 0) {
            ClosestVisitor<Stats> vis(RT_TMAX_DEFAULT);
            traverse(nodes, tris, ray, vis, stack);
            sn += vis.nodes; st += vis.tris; sh += vis.prim >= 0;
            if (vis.prim >= 0) {
                const float* tp = reinterpret_cast<const float*>(tris + (size_t)vis.slot * 48u);
                TriHit th;
                tri_test(ray, tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10], th);
                const HitAttr at = tri_attr(th, tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10]);
                hit[r] = 1; front[r] = tri_front(ray, th) ? 1 : 0; tri[r] = vis.prim;
                loc[3 * r] = at.lx; loc[3 * r + 1] = at.ly; loc[3 * r + 2] = at.lz; uv[2 * r] = at.uv0; uv[2 * r + 1] = at.uv1;
            } else {
                hit[r] = 0; front[r] = 0; tri[r] = -1;
                loc[3 * r] = loc[3 * r + 1] = loc[3 * r + 2] = 0.f; uv[2 * r] = uv[2 * r + 1] = 0.f;
            }
        } else if (mode == 1) {
            AnyVisitor<Stats> vis(RT_TMAX_DEFAULT);
            traverse(nodes, tris, ray, vis, stack);
            sn += vis.nodes; st += vis.tris; sh += vis.found;
            hit[r] = vis.found ? 1 : 0;
        } else {
            CountVisitor<Stats> vis(RT_TMAX_DEFAULT);
            traverse(nodes, tris, ray, vis, stack);
            sn += vis.nodes; st += vis.tris; sh += vis.count > 0;
            count[r] = vis.count;
        }
        if (stack.max_sp > ms) ms = stack.max_sp;
    }
    if (stats) { stats[0] = sn; stats[1] = st; stats[2] = (uint64_t)nray; stats[3] = sh; }
    if (max_stack) *max_stack = ms;
    return 0;
}

// Validation of a blob (built here, copied back from the GPU, re-fitted or adopted).  Each check has its own code:
//   100 shorter than a header, 101 magic / ABI version, 102 a section ends beyond the blob, 103 node pool overflow (or,
//   without faces to compare with, a non-zero bad_index_faces);
//   30 n_nodes_cap is not wide_node_cap(n_tris), 31 an offset differs from the product's layout (tris behind the
//   header, nodes 256-aligned behind them, parent links parents_offset_for), 32 used_bytes is not used_bytes_for;
//   1 node index out of range, 2 node reached twice, 3 deeper than 200 levels, 5 slot both inner and leaf, 7 bad unary
//   leaf count, 8 record index out of range, 9 record referenced twice, 10 a dequantised slot box does not contain the
//   exact boxes of the triangles below it, 11 node never reached, 12 record never referenced, 13 header depth;
//   20 a parent link is not (parent << 3 | slot) of the slot that references the node, or the root's is not 0xffffffff;
//   25 a node's reserved word, a record's pad words or an alignment gap inside the used prefix is not zero;
//   33 the header box is not the ordered union of the records' triangle boxes (tri_bbox; the zero box when empty).
// With vertices and faces:
//   24 n_tris differs from the number of faces, 22 the records' prim ids are not a permutation of the faces,
//   21 a record's vertices are not bit-equal to vertices[clamp_index(faces[prim])], 34 bad_index_faces is not the
//   number of faces with an index outside [0, n_verts).
// Returns 0 when valid; info[0]=nodes, info[1]=tris, info[2]=max depth, info[3]=sum of children over nodes.
namespace {
struct Checker {
    const uint8_t* nodes; const uint8_t* tris; uint32_t n_nodes, n_tris;
    std::vector<uint8_t> node_seen, tri_seen;
    uint64_t children = 0; int max_depth = 0; int error = 0;
    std::vector<uint32_t> expect_parent;   // (parent << 3 | slot) of every node reached, 0xffffffff for the root
    // returns exact box of subtree
    BBox walk(uint32_t idx, int depth) {
        BBox acc; acc.lx = acc.ly = acc.lz = INFINITY; acc.hx = acc.hy = acc.hz = -INFINITY; acc.pad0 = acc.pad1 = 0;
        if (idx >= n_nodes) { error = 1; return acc; }
        if (node_seen[idx]) { error = 2; return acc; }
        node_seen[idx] = 1;
        if (depth + 1 > max_depth) max_depth = depth + 1;
        if (depth > 200) { error = 3; return acc; }
        Node8 nd; memcpy(&nd, nodes + (size_t)idx * 80u, 80);
        const float sx = exp2_biased(nd.ex), sy = exp2_biased(nd.ey), sz = exp2_biased(nd.ez);
        uint32_t rel = 0;
        for (int s = 0; s < 8; ++s) {
            const bool inner = (nd.imask >> s) & 1u;
            const uint32_t un = (nd.trimask >> (3 * s)) & 7u;
            if (!inner && un == 0) continue;
            ++children;
            BBox cb;
            if (inner) {
                if (un != 0) error = 5;
                if (nd.child_base + rel < n_nodes) expect_parent[nd.child_base + rel] = (idx << 3) | (uint32_t)s;
                cb = walk(nd.child_base + rel, depth + 1);
                ++rel;
            } else {
                const uint32_t cnt = un == 1 ? 1 : (un == 3 ? 2 : (un == 7 ? 3 : 0));
                if (cnt == 0) { error = 7; continue; }
                const uint32_t off = (uint32_t)__builtin_popcount(nd.trimask & ((1u << (3 * s)) - 1u));
                cb.lx = cb.ly = cb.lz = INFINITY; cb.hx = cb.hy = cb.hz = -INFINITY; cb.pad0 = cb.pad1 = 0;
                for (uint32_t j = 0; j < cnt; ++j) {
                    const uint32_t ti = nd.tri_base + off + j;
                    if (ti >= n_tris) { error = 8; continue; }
                    if (tri_seen[ti]) error = 9;
                    tri_seen[ti] = 1;
                    const float* tp = reinterpret_cast<const float*>(tris + (size_t)ti * 48u);
                    BBox b; // exact (not inflated) triangle box
                    b.lx = fminf(fminf(tp[0], tp[4]), tp[8]); b.ly = fminf(fminf(tp[1], tp[5]), tp[9]); b.lz = fminf(fminf(tp[2], tp[6]), tp[10]);
                    b.hx = fmaxf(fmaxf(tp[0], tp[4]), tp[8]); b.hy = fmaxf(fmaxf(tp[1], tp[5]), tp[9]); b.hz = fmaxf(fmaxf(tp[2], tp[6]), tp[10]);
                    b.pad0 = b.pad1 = 0;
                    cb = bbox_union(cb, b);
                }
            }
            if (error) return acc;
            // dequantised slot box (real arithmetic in double)
            const double qlx = (double)nd.px + nd.qlox[s] * (double)sx, qhx = (double)nd.px + nd.qhix[s] * (double)sx;
            const double qly = (double)nd.py + nd.qloy[s] * (double)sy, qhy = (double)nd.py + nd.qhiy[s] * (double)sy;
            const double qlz = (double)nd.pz + nd.qloz[s] * (double)sz, qhz = (double)nd.pz + nd.qhiz[s] * (double)sz;
            if (cb.lx <= cb.hx) {   // skip NaN / empty subtrees
                if (qlx > cb.lx || qly > cb.ly || qlz > cb.lz || qhx < cb.hx || qhy < cb.hy || qhz < cb.hz) { error = 10; return acc; }
            }
            acc = bbox_union(acc, cb);
        }
        return acc;
    }
};
}  // namespace

// The root-frame test of the pooled kernels' fill (rt_core.cuh frame_missed) against the full root node test, ray by ray:
// out[0] = rays the frame rejects, out[1] = of those, rays for which node_test still reports a hit slot (must be 0),
// out[2] = rays the root node test rejects (>= out[0]).  Same code as the device runs (RT_HD).
extern "C" int hs_frame_check(const uint8_t* blob, int64_t nray, const float* o, const float* d, uint64_t* out) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* np = blob + h->nodes_offset;
    const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48), n4 = ldg128(np + 64);
    const RootFrame f = root_frame(n0, n2, n3, n4);
    out[0] = out[1] = out[2] = 0;
    for (int64_t r = 0; r < nray; ++r) {
        Ray ray;
        ray_setup(ray, o[3 * r], o[3 * r + 1], o[3 * r + 2], d[3 * r], d[3 * r + 1], d[3 * r + 2]);
        float idx, idy, idz;
        ray_inverse(d[3 * r], d[3 * r + 1], d[3 * r + 2], idx, idy, idz);
        if (idx != ray.idx || idy != ray.idy || idz != ray.idz) return -5;      // the fill and the set-up must agree bit for bit
        const bool rejected = frame_missed(ray.ox, ray.oy, ray.oz, idx, idy, idz, f, RT_TMAX_DEFAULT);
        const uint32_t hm = node_test(ray, n0, n1, n2, n3, n4, 0.0f, RT_TMAX_DEFAULT);
        out[0] += rejected; out[1] += rejected && hm != 0u; out[2] += hm == 0u;
    }
    return 0;
}

extern "C" void hs_tile_map(uint32_t n, uint32_t tiles_per_row, uint32_t width, uint32_t w_log2, uint32_t* out) {
    for (uint32_t t = 0; t < n; ++t) out[t] = tile_map(t, tiles_per_row, width, w_log2);
}

namespace {
bool all_zero(const uint8_t* p, size_t n) {
    for (size_t i = 0; i < n; ++i) if (p[i]) return false;
    return true;
}
}  // namespace

extern "C" int hs_check_blob(const uint8_t* blob, size_t blob_bytes, const float* verts, int64_t nv, const int32_t* faces,
                             int64_t nf, uint64_t* info) {
    if (blob_bytes < RT_BLOB_HEADER_BYTES) return 100;
    rt_blob_header h; memcpy(&h, blob, sizeof(h));
    if (h.magic != RT_BLOB_MAGIC || h.abi_version != RT_ABI_VERSION) return 101;
    if (h.used_bytes > blob_bytes || h.nodes_offset + (uint64_t)h.n_nodes * 80u > blob_bytes ||
        h.tris_offset + (uint64_t)h.n_tris * 48u > blob_bytes || h.parents_offset + (uint64_t)h.n_nodes * 4u > blob_bytes)
        return 102;
    if (h.node_overflow != 0 || (faces == nullptr && h.bad_index_faces != 0)) return 103;
    if (h.n_nodes_cap != wide_node_cap(h.n_tris, leaf_setting())) return 30;
    if (h.tris_offset != RT_BLOB_HEADER_BYTES || h.nodes_offset != align_up(h.tris_offset + (size_t)h.n_tris * 48u, 256) ||
        h.parents_offset != parents_offset_for(h.nodes_offset, h.n_nodes))
        return 31;
    if (h.used_bytes != used_bytes_for(h.parents_offset, h.n_nodes)) return 32;
    Checker c; c.nodes = blob + h.nodes_offset; c.tris = blob + h.tris_offset; c.n_nodes = h.n_nodes; c.n_tris = h.n_tris;
    c.node_seen.assign(h.n_nodes, 0); c.tri_seen.assign(h.n_tris, 0); c.expect_parent.assign(h.n_nodes, 0xffffffffu);
    c.walk(0, 0);
    if (c.error) return c.error;
    for (uint32_t i = 0; i < h.n_nodes; ++i) if (!c.node_seen[i]) return 11;
    for (uint32_t i = 0; i < h.n_tris; ++i) if (!c.tri_seen[i]) return 12;
    if ((uint32_t)c.max_depth != h.depth) return 13;
    const uint32_t* parent = reinterpret_cast<const uint32_t*>(blob + h.parents_offset);
    for (uint32_t i = 0; i < h.n_nodes; ++i) {
        uint32_t p; memcpy(&p, &parent[i], 4);
        if (p != c.expect_parent[i]) return 20;
    }
    for (uint32_t i = 0; i < h.n_nodes; ++i) {
        Node8 nd; memcpy(&nd, c.nodes + (size_t)i * 80u, 80);
        if (nd.reserved != 0) return 25;
    }
    for (uint32_t i = 0; i < h.n_tris; ++i) {
        TriRecord tr; memcpy(&tr, c.tris + (size_t)i * 48u, 48);
        if (tr.pad1 != 0 || tr.pad2 != 0) return 25;
    }
    const uint64_t tris_end = h.tris_offset + (uint64_t)h.n_tris * 48u, nodes_end = h.nodes_offset + (uint64_t)h.n_nodes * 80u,
                   parents_end = h.parents_offset + (uint64_t)h.n_nodes * 4u;
    if (!all_zero(blob + sizeof(rt_blob_header), RT_BLOB_HEADER_BYTES - sizeof(rt_blob_header)) ||
        !all_zero(blob + tris_end, h.nodes_offset - tris_end) || !all_zero(blob + nodes_end, h.parents_offset - nodes_end) ||
        !all_zero(blob + parents_end, h.used_bytes - parents_end))
        return 25;
    {   // header box: ordered union of the records' triangle boxes, as k_scene_bounds reduces it
        uint32_t lo[3] = {kOrdPosInf, kOrdPosInf, kOrdPosInf}, hi[3] = {kOrdNegInf, kOrdNegInf, kOrdNegInf};
        for (uint32_t i = 0; i < h.n_tris; ++i) {
            const float* tp = reinterpret_cast<const float*>(c.tris + (size_t)i * 48u);
            const BBox b = tri_bbox(tp[0], tp[1], tp[2], tp[4], tp[5], tp[6], tp[8], tp[9], tp[10]);
            lo[0] = std::min(lo[0], ord_lo(b.lx)); lo[1] = std::min(lo[1], ord_lo(b.ly)); lo[2] = std::min(lo[2], ord_lo(b.lz));
            hi[0] = std::max(hi[0], ord_hi(b.hx)); hi[1] = std::max(hi[1], ord_hi(b.hy)); hi[2] = std::max(hi[2], ord_hi(b.hz));
        }
        for (int a = 0; a < 3; ++a) {
            const float el = h.n_tris ? ord2f(lo[a]) : 0.0f, eh = h.n_tris ? ord2f(hi[a]) : 0.0f;
            if (memcmp(&el, &h.aabb_lo[a], 4) != 0 || memcmp(&eh, &h.aabb_hi[a], 4) != 0) return 33;
        }
    }
    if (faces != nullptr) {
        if (nf != (int64_t)h.n_tris) return 24;
        std::vector<uint8_t> prim_seen((size_t)nf, 0);
        for (uint32_t i = 0; i < h.n_tris; ++i) {
            int32_t prim; memcpy(&prim, c.tris + (size_t)i * 48u + 12, 4);
            if (prim < 0 || prim >= nf || prim_seen[prim]) return 22;
            prim_seen[prim] = 1;
        }
        for (uint32_t i = 0; i < h.n_tris; ++i) {
            const float* tp = reinterpret_cast<const float*>(c.tris + (size_t)i * 48u);
            int32_t prim; memcpy(&prim, tp + 3, 4);
            float v[9]; tri_verts(verts, nv, faces, prim, v);
            if (memcmp(tp, v, 12) != 0 || memcmp(tp + 4, v + 3, 12) != 0 || memcmp(tp + 8, v + 6, 12) != 0) return 21;
        }
        uint32_t bad = 0;
        for (int64_t i = 0; i < nf; ++i) {
            bool ok = true;
            for (int k = 0; k < 3; ++k) ok = ok && faces[3 * i + k] >= 0 && faces[3 * i + k] < nv;
            bad += ok ? 0u : 1u;
        }
        if (bad != h.bad_index_faces) return 34;
    }
    if (info) { info[0] = h.n_nodes; info[1] = h.n_tris; info[2] = (uint64_t)c.max_depth; info[3] = c.children; }
    return 0;
}

// Canonical numbering of a valid blob into `out` (same size): nodes breadth-first from the root, the inner children of
// each node contiguous in slot order; triangle records in the order the nodes (in that order) reference them.
// child_base / tri_base (0 for a node without inner children / triangles, as alloc_children leaves them), the records'
// positions and the parent links - renumbered, not recomputed - are rewritten; every other byte is copied.  Two correct
// builds of one mesh differ only in the numbering k_collapse's bump allocators hand out, so their canonical forms are
// equal byte for byte.  Returns 0, or -1 when the tree does not reach every node and record exactly once.
extern "C" int hs_canonical(const uint8_t* blob, size_t blob_bytes, uint8_t* out) {
    rt_blob_header h; memcpy(&h, blob, sizeof(h));
    if (blob_bytes < RT_BLOB_HEADER_BYTES || h.magic != RT_BLOB_MAGIC || h.parents_offset + (uint64_t)h.n_nodes * 4u > blob_bytes ||
        h.nodes_offset + (uint64_t)h.n_nodes * 80u > blob_bytes || h.tris_offset + (uint64_t)h.n_tris * 48u > blob_bytes)
        return -1;
    memcpy(out, blob, blob_bytes);
    const uint8_t* nodes = blob + h.nodes_offset;
    const uint8_t* tris = blob + h.tris_offset;
    std::vector<uint32_t> order;                                  // old index of new node i
    std::vector<uint32_t> new_of(h.n_nodes, 0xffffffffu);
    order.reserve(h.n_nodes);
    order.push_back(0); new_of[0] = 0;
    uint32_t next_tri = 0;
    for (size_t q = 0; q < order.size(); ++q) {
        const uint32_t w = order[q];
        Node8 nd; memcpy(&nd, nodes + (size_t)w * 80u, 80);
        const uint32_t n_inner = (uint32_t)__builtin_popcount(nd.imask), n_rec = (uint32_t)__builtin_popcount(nd.trimask);
        const uint32_t base = (uint32_t)order.size();
        for (uint32_t r = 0; r < n_inner; ++r) {
            const uint32_t ch = nd.child_base + r;
            if (ch >= h.n_nodes || new_of[ch] != 0xffffffffu) return -1;
            new_of[ch] = (uint32_t)order.size();
            order.push_back(ch);
        }
        if (n_rec && (nd.tri_base + (uint64_t)n_rec > h.n_tris || next_tri + (uint64_t)n_rec > h.n_tris)) return -1;
        memcpy(out + h.tris_offset + (size_t)next_tri * 48u, tris + (size_t)nd.tri_base * 48u, (size_t)n_rec * 48u);
        nd.child_base = n_inner ? base : 0u;
        nd.tri_base = n_rec ? next_tri : 0u;
        next_tri += n_rec;
        memcpy(out + h.nodes_offset + q * 80u, &nd, 80);
    }
    if (order.size() != h.n_nodes || next_tri != h.n_tris) return -1;
    const uint32_t* par = reinterpret_cast<const uint32_t*>(blob + h.parents_offset);
    uint32_t* opar = reinterpret_cast<uint32_t*>(out + h.parents_offset);
    for (uint32_t i = 0; i < h.n_nodes; ++i) {
        const uint32_t p = par[order[i]];
        opar[i] = (p == 0xffffffffu || (p >> 3) >= h.n_nodes) ? p : ((new_of[p >> 3] << 3) | (p & 7u));
    }
    return 0;
}

// prim ids stored in the triangle records (to check the permutation)
extern "C" int hs_blob_prims(const uint8_t* blob, int32_t* prims_out) {
    rt_blob_header h; memcpy(&h, blob, sizeof(h));
    for (uint32_t i = 0; i < h.n_tris; ++i) memcpy(&prims_out[i], blob + h.tris_offset + (size_t)i * 48u + 12, 4);
    return 0;
}

// Refit with new vertex positions (same faces): sequential version of k_refit_tris / k_refit_nodes.
extern "C" int hs_refit(const float* verts, int64_t nv, const int32_t* faces, int64_t n, uint8_t* blob, size_t blob_bytes) {
    rt_blob_header h; memcpy(&h, blob, sizeof(h));
    if (h.magic != RT_BLOB_MAGIC || h.n_tris != (uint32_t)n) return -4;
    if (h.parents_offset + (uint64_t)h.n_nodes * 4u > blob_bytes) return -3;
    if (n == 0) return 0;
    uint8_t* tris = blob + h.tris_offset;
    uint8_t* nodes = blob + h.nodes_offset;
    const uint32_t* parent = reinterpret_cast<const uint32_t*>(blob + h.parents_offset);
    for (int64_t i = 0; i < n; ++i) {
        int32_t prim; memcpy(&prim, tris + (size_t)i * 48u + 12, 4);
        write_tri_record(tris, (uint32_t)i, (uint32_t)prim, verts, nv, faces);
    }
    std::vector<BBox> node_box(h.n_nodes);
    std::vector<uint32_t> counters(h.n_nodes, 0);
    for (uint32_t w0 = 0; w0 < h.n_nodes; ++w0) {
        if (nodes[(size_t)w0 * 80u + 15] != 0) continue;
        uint32_t w = w0;
        for (;;) {
            node_box[w] = refit_node(nodes, tris, w, node_box.data());
            if (w == 0) {
                h.aabb_lo[0] = node_box[0].lx; h.aabb_lo[1] = node_box[0].ly; h.aabb_lo[2] = node_box[0].lz;
                h.aabb_hi[0] = node_box[0].hx; h.aabb_hi[1] = node_box[0].hy; h.aabb_hi[2] = node_box[0].hz;
                break;
            }
            const uint32_t pw = parent[w] >> 3;
            const uint32_t need = (uint32_t)__builtin_popcount((uint32_t)nodes[(size_t)pw * 80u + 15]);
            if (++counters[pw] != need) break;
            w = pw;
        }
    }
    memcpy(blob, &h, sizeof(h));
    return 0;
}
