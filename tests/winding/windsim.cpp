// windsim.cpp — TEST INFRASTRUCTURE ONLY.  Runs the moment pass and the traversal of rt_winding.cuh (RT_HD, the code
// rt_winding.cu runs) on the CPU over a blob from tests/hostsim or a GPU blob copied to the host, and checks every
// moment record (radius bound, centroid, N, M) exhaustively in binary64 against the node's own triangles.  Never linked
// into libtriro_b200.so.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -mfma -shared -fPIC windsim.cpp -o libwindsim.so
#include <cmath>
#include <cstring>
#include <vector>
#include "../../include/raymesh_b200.h"
#include "../../trimesh-ray-optix_b200/csrc/rt_winding.cuh"

using namespace rt;

namespace {
struct HostWindStack {
    WindStackEntry e[kMaxDepth];
    int max_sp = 0;
    void push(int sp, const WindStackEntry& v) { e[sp] = v; if (sp + 1 > max_sp) max_sp = sp + 1; }
    void pop(int sp, WindStackEntry& v) { v = e[sp]; }
};

// children before parents, each node once (post-order from the root)
void moments_rec(const uint8_t* nodes, const uint8_t* tris, uint32_t w, uint8_t* moments, float* weights) {
    const Node8* nd = reinterpret_cast<const Node8*>(nodes + (size_t)w * 80u);
    const int nin = popc32(nd->imask);
    for (int c = 0; c < nin; ++c) moments_rec(nodes, tris, nd->child_base + (uint32_t)c, moments, weights);
    const WindNodeOut o = node_moment(nodes, tris, w, moments, weights);
    store_moment(moments, w, o.mo, weights, o.weight);
}
}  // namespace

// moments: n_nodes x 64 bytes, weights: n_nodes floats (the subtree areas the moment pass keeps in its workspace)
extern "C" int ws_moments(const uint8_t* blob, uint8_t* moments, float* weights) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    moments_rec(blob + h->nodes_offset, blob + h->tris_offset, 0u, moments, weights);
    return 0;
}

extern "C" uint32_t ws_n_nodes(const uint8_t* blob) { return reinterpret_cast<const rt_blob_header*>(blob)->n_nodes; }

// winding numbers of a dense [n,3] batch with the given moments; stats = {nodes, triangles, points, far terms},
// max_stack = deepest group stack seen
extern "C" int ws_winding(const uint8_t* blob, const uint8_t* moments, int64_t n, const float* pts, float beta, float* w,
                          uint64_t* stats, int32_t* max_stack) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    const uint8_t* tris = blob + h->tris_offset;
    const uint8_t* nodes = blob + h->nodes_offset;
    uint64_t sn = 0, stt = 0, sf = 0;
    int ms = 0;
    for (int64_t i = 0; i < n; ++i) {
        WindTrav t;
        wind_init(t, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]);
        HostWindStack stack;
        WindStats st;
        while (!wind_step(nodes, tris, moments, beta, t, st, stack)) {}
        w[i] = wind_result(t);
        sn += st.nodes; stt += st.tris; sf += st.fars;
        if (stack.max_sp > ms) ms = stack.max_sp;
    }
    if (stats) { stats[0] = sn; stats[1] = stt; stats[2] = (uint64_t)n; stats[3] = sf; }
    if (max_stack) *max_stack = ms;
    return 0;
}

// Exhaustive check of every moment record in binary64, from the node's subtree alone (no stored child record is used):
//   rho: every finite vertex of every triangle record below the node lies within rho of the stored p~;
//   p~:  the area-weighted centroid sum_t |A_t| c_t / sum_t |A_t| over the finite triangles (when the area is > 0);
//   N:   sum_t A_t;  M: sum_t (c_t - p~)_i A_t,j about the STORED p~ (the far field uses that centre).
// out[0] = rho violations, out[1] = (node, vertex) pairs checked, out[2] = nodes checked;
// worst[0] = largest |v - p~| / rho, worst[1] = largest |p~ - centroid| / rho, worst[2] = largest |N - N64| / sum_t |A_t|,
// worst[3] = largest |M_ij - M64_ij| / sum_t |A_t| |c_t - p~|, each scale with the rounding floors below.
namespace {
struct Tri64 { double c[3], a[3], area, ee; };   // ee = |v1 - v0| |v2 - v0|
struct MomentChecker {
    const uint8_t* nodes; const uint8_t* tris; const WindMoment* mo;
    uint64_t violations = 0, checked = 0, nodes_checked = 0; double worst[4] = {0, 0, 0, 0};
    // appends the finite vertices and the finite triangles of the subtree of `w`, then checks w's record against them
    void walk(uint32_t w, std::vector<double>& verts, std::vector<Tri64>& ts) {
        const size_t v0 = verts.size(), t0 = ts.size();
        const Node8* nd = reinterpret_cast<const Node8*>(nodes + (size_t)w * 80u);
        const int ntri = popc32(nd->trimask), nin = popc32(nd->imask);
        for (int j = 0; j < ntri; ++j) {
            const float* tp = reinterpret_cast<const float*>(tris + (size_t)(nd->tri_base + (uint32_t)j) * 48u);
            bool fin = true;
            for (int k = 0; k < 3; ++k) {
                const float* v = tp + 4 * k;
                if (std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]))
                    for (int a = 0; a < 3; ++a) verts.push_back(v[a]);
                else
                    fin = false;
            }
            if (!fin) continue;
            Tri64 t;
            double e1[3], e2[3];
            for (int a = 0; a < 3; ++a) {
                t.c[a] = ((double)tp[a] + (double)tp[4 + a] + (double)tp[8 + a]) / 3.0;
                e1[a] = (double)tp[4 + a] - tp[a];
                e2[a] = (double)tp[8 + a] - tp[a];
            }
            t.a[0] = 0.5 * (e1[1] * e2[2] - e1[2] * e2[1]);
            t.a[1] = 0.5 * (e1[2] * e2[0] - e1[0] * e2[2]);
            t.a[2] = 0.5 * (e1[0] * e2[1] - e1[1] * e2[0]);
            t.area = std::sqrt(t.a[0] * t.a[0] + t.a[1] * t.a[1] + t.a[2] * t.a[2]);
            t.ee = std::sqrt((e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]) * (e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2]));
            ts.push_back(t);
        }
        for (int c = 0; c < nin; ++c) walk(nd->child_base + (uint32_t)c, verts, ts);
        const WindMoment& m = mo[w];
        const double p[3] = {m.px, m.py, m.pz};
        for (size_t i = v0; i < verts.size(); i += 3) {
            const double dx = verts[i] - p[0], dy = verts[i + 1] - p[1], dz = verts[i + 2] - p[2];
            const double d = std::sqrt(dx * dx + dy * dy + dz * dz);
            ++checked;
            if (!(d <= (double)m.rho)) ++violations;
            if (m.rho > 0.0f && d / m.rho > worst[0]) worst[0] = d / m.rho;
        }
        // Scales: a binary32 area vector is exact to a few u of |e1||e2| (so a sliver's is rounding noise), a centroid
        // difference to a few u of |p~| + rho.  Both floors enter the scales at 2^-20; the centroid is compared only
        // where the areas dominate their floors (elsewhere any point of the subtree is a valid centre).
        const double pa = std::fabs(p[0]) + std::fabs(p[1]) + std::fabs(p[2]) + m.rho;
        double W = 0, s[3] = {0, 0, 0}, n[3] = {0, 0, 0}, M[9] = {0}, sn = 0, sm = 0, ee = 0;
        for (size_t i = t0; i < ts.size(); ++i) {
            const Tri64& t = ts[i];
            W += t.area;
            ee += t.ee;
            double d[3];
            for (int a = 0; a < 3; ++a) { s[a] += t.area * t.c[a]; n[a] += t.a[a]; d[a] = t.c[a] - p[a]; }
            for (int a = 0; a < 3; ++a)
                for (int b = 0; b < 3; ++b) M[3 * a + b] += d[a] * t.a[b];
            const double af = t.area + std::ldexp(t.ee, -20);
            sn += af;
            sm += af * (std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]) + std::ldexp(pa, -20));
        }
        ++nodes_checked;
        if (W > std::ldexp(ee, -10)) {
            const double scale = (double)m.rho + std::ldexp(pa, -20);
            for (int a = 0; a < 3; ++a) worst[1] = std::fmax(worst[1], std::fabs(p[a] - s[a] / W) / scale);
        }
        const double sn_ = sn > 0 ? sn : 1.0, sm_ = sm > 0 ? sm : 1.0;
        const float mn[3] = {m.nx, m.ny, m.nz};
        for (int a = 0; a < 3; ++a) worst[2] = std::fmax(worst[2], std::fabs((double)mn[a] - n[a]) / sn_);
        for (int k = 0; k < 9; ++k) worst[3] = std::fmax(worst[3], std::fabs((double)m.m[k] - M[k]) / sm_);
    }
};
}  // namespace

extern "C" int ws_moment_check(const uint8_t* blob, const uint8_t* moments, uint64_t* out, double* worst) {
    const rt_blob_header* h = reinterpret_cast<const rt_blob_header*>(blob);
    if (h->magic != RT_BLOB_MAGIC) return -4;
    MomentChecker c;
    c.nodes = blob + h->nodes_offset; c.tris = blob + h->tris_offset; c.mo = reinterpret_cast<const WindMoment*>(moments);
    std::vector<double> verts;
    std::vector<Tri64> ts;
    c.walk(0u, verts, ts);
    out[0] = c.violations; out[1] = c.checked; out[2] = c.nodes_checked;
    for (int k = 0; k < 4; ++k) worst[k] = c.worst[k];
    return 0;
}

// far_field() of one moment record rec[16] seen from each of n points, with r and |r| formed as wind_step forms them:
// 4 pi times the node's approximate winding number
extern "C" void ws_far_field(const float* rec, int64_t n, const float* q, float* out) {
    WindMoment m;
    std::memcpy(&m, rec, sizeof(m));
    for (int64_t i = 0; i < n; ++i) {
        const float rx = fsub(m.px, q[3 * i]), ry = fsub(m.py, q[3 * i + 1]), rz = fsub(m.pz, q[3 * i + 2]);
        out[i] = far_field(m, rx, ry, rz, fsqrt(dot3f(rx, ry, rz, rx, ry, rz)));
    }
}

extern "C" void ws_atan2(int64_t n, const float* y, const float* x, float* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = atan2_rn(y[i], x[i]);
}

// solid angle (binary32, the kernel's) of triangle tri[9] seen from each of n points
extern "C" void ws_solid_angle(int64_t n, const float* q, const float* tri, float* out) {
    for (int64_t i = 0; i < n; ++i)
        out[i] = solid_angle(q[3 * i], q[3 * i + 1], q[3 * i + 2], tri[0], tri[1], tri[2], tri[3], tri[4], tri[5], tri[6],
                             tri[7], tri[8]);
}
