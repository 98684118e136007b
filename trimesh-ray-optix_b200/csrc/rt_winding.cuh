// rt_winding.cuh — generalized winding numbers on the BVH8 (Jacobson, Kavan, Sorkine-Hornung 2013) with the far-field
// expansion of Barill et al. 2018 ("Fast Winding Numbers for Soups and Clouds"): the solid angle of one triangle, an
// own atan2, the per-node moments and one traversal step.  Everything here is RT_HD, like rt_point.cuh, so that
// tests/winding/ runs exactly the code of rt_winding.cu on the CPU.
//
// Contract (DESIGN.md §4.7): w(q) = sum_t Omega_t(q) / 4pi.  Triangles in leaf slots are always summed exactly; an
// inner child whose moment ball is far (|r| > beta * rho) contributes its two-term expansion instead of being visited.
// Only the correctly rounded wrappers of rt_core.cuh / rt_point.cuh are used and every point visits its nodes in a
// fixed order, so the result is a function of (blob, moments, point, beta) alone: kernel and host simulator agree bit
// for bit.
#pragma once
#include "rt_point.cuh"

namespace rt {

// ------------------------------------------------------------------ moment record
// One 64-byte record per node (four 16-byte loads), a side array indexed like the nodes:
//   p[3], rho          area-weighted centroid p~ of the node's triangles and a radius bound: every finite vertex below
//                      the node lies within rho of p~ (in real arithmetic, for the rounded p~ that is stored)
//   n[3]               N = sum_t A_t, A_t = (v1 - v0) x (v2 - v0) / 2
//   m[9]               M_ij = sum_t (c_t - p~)_i A_t,j, row-major, c_t = centroid of t
// A triangle with a non-finite vertex contributes to none of these; its finite vertices still count for rho.
struct alignas(16) WindMoment {
    float px, py, pz, rho;
    float nx, ny, nz;
    float m[9];
};
static_assert(sizeof(WindMoment) == 64, "WindMoment must be 64 bytes");

constexpr float kInv4Pi = 0.0795774715459476679f;   // 1 / (4 pi), rounded to binary32

#if defined(__CUDA_ARCH__)
// moments written by other threads of the moment pass: read from L2, never from a stale L1 line
RT_HD U4 ldcg128(const void* p) {
    const uint4 v = __ldcg(reinterpret_cast<const uint4*>(p));
    U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r;
}
RT_HD float ldcgf(const float* p) { return __ldcg(p); }
#else
RT_HD U4 ldcg128(const void* p) { return *reinterpret_cast<const U4*>(p); }
RT_HD float ldcgf(const float* p) { return *p; }
#endif

RT_HD bool finite3(float x, float y, float z) {
    return fsub(x, x) == 0.0f && fsub(y, y) == 0.0f && fsub(z, z) == 0.0f;   // x - x is NaN for NaN and +-inf
}

// ------------------------------------------------------------------ atan2
// atan2(y, x) over the full plane as a fixed sequence of correctly rounded binary32 operations.  The ratio
// t = min(|x|,|y|) / max(|x|,|y|) in [0, 1] is reduced to |s| <= tan(pi/8) (s = (t - 1) / (t + 1) + pi/4 above it),
// where the degree-9 odd minimax polynomial of Cephes' atanf is used; then the octant is unfolded (pi/2 - a, pi - a,
// -a); the sign is that of y including a signed zero (atan2(-0, x < 0) = -pi).  atan2(0, 0) = 0 whatever the signs of
// the zeros.  Error against binary64 atan2 of the same binary32 inputs,
// measured over all four quadrants with ratios from 2^-40 to 2^40 (tests/test_winding_logic.py checks it):
// |error| <= 3e-7 (about 1.3 ulp of pi) and |error| <= 2.5e-7 |atan2(y, x)|.
RT_HD float atan2_rn(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    if (!(mx > 0.0f)) return 0.0f;
    const float t = fdiv(mn, mx);
    const bool big = t > 0.414213562373f;
    const float s = big ? fdiv(fsub(t, 1.0f), fadd(t, 1.0f)) : t;
    const float z = fmul(s, s);
    float p = ffma(8.05374449538e-2f, z, -1.38776856032e-1f);
    p = ffma(p, z, 1.99777106478e-1f);
    p = ffma(p, z, -3.33329491539e-1f);
    float a = ffma(fmul(p, z), s, s);
    if (big) a = fadd(a, 0.785398163397f);                   // pi/4
    if (ay > ax) a = fsub(1.57079632679f, a);                // pi/2
    if (x < 0.0f) a = fsub(3.14159265359f, a);               // pi
    return signbit(y) ? -a : a;
}

// ------------------------------------------------------------------ solid angle of one triangle
// van Oosterom & Strackee 1983 on unit vectors: with a = v0 - q, b = v1 - q, c = v2 - q and a^ = a / |a| etc.,
//   Omega = 2 atan2(det[a^ b^ c^], 1 + a^.b^ + b^.c^ + c^.a^),
// the textbook form divided by |a||b||c| > 0.  det[a b c] = a . n with n = (v1 - v0) x (v2 - v0), so
//   det[a^ b^ c^] = ((a^ . n) / |b|) / |c|,
// which is exactly 0 whenever the computed n is (a repeated vertex, exactly collinear vertices) and whenever a^ is
// orthogonal to n in every product (q in the plane of an axis-aligned triangle).  Every intermediate stays near L^k,
// k <= 2, at length scale L, so no product of three lengths can leave the binary32 range.  Returns 0 for a triangle
// with a non-finite vertex, for q at a vertex (|a|, |b| or |c| = 0, also when the square underflows) and whenever the
// computed det is exactly 0.
RT_HD float unit3(float& x, float& y, float& z) {
    const float l = fsqrt(dot3f(x, y, z, x, y, z));
    if (l > 0.0f) {
        const float il = fdiv(1.0f, l);
        x = fmul(x, il); y = fmul(y, il); z = fmul(z, il);
    }
    return l;
}

RT_HD float solid_angle(float qx, float qy, float qz, float v0x, float v0y, float v0z, float v1x, float v1y, float v1z,
                        float v2x, float v2y, float v2z) {
    if (!(finite3(v0x, v0y, v0z) && finite3(v1x, v1y, v1z) && finite3(v2x, v2y, v2z))) return 0.0f;
    const float e1x = fsub(v1x, v0x), e1y = fsub(v1y, v0y), e1z = fsub(v1z, v0z);
    const float e2x = fsub(v2x, v0x), e2y = fsub(v2y, v0y), e2z = fsub(v2z, v0z);
    const float nx = fsub(fmul(e1y, e2z), fmul(e1z, e2y));
    const float ny = fsub(fmul(e1z, e2x), fmul(e1x, e2z));
    const float nz = fsub(fmul(e1x, e2y), fmul(e1y, e2x));
    float ax = fsub(v0x, qx), ay = fsub(v0y, qy), az = fsub(v0z, qz);
    float bx = fsub(v1x, qx), by = fsub(v1y, qy), bz = fsub(v1z, qz);
    float cx = fsub(v2x, qx), cy = fsub(v2y, qy), cz = fsub(v2z, qz);
    const float la = unit3(ax, ay, az), lb = unit3(bx, by, bz), lc = unit3(cx, cy, cz);
    if (!(la > 0.0f && lb > 0.0f && lc > 0.0f)) return 0.0f;
    const float det = fdiv(fdiv(dot3f(ax, ay, az, nx, ny, nz), lb), lc);
    if (det == 0.0f) return 0.0f;
    const float den = fadd(fadd(fadd(1.0f, dot3f(ax, ay, az, bx, by, bz)), dot3f(bx, by, bz, cx, cy, cz)),
                           dot3f(cx, cy, cz, ax, ay, az));
    return fmul(2.0f, atan2_rn(det, den));
}

// ------------------------------------------------------------------ far field
// 4 pi w of a node seen from q, its first two expansion terms, with r = p~ - q, l = |r|, u = r / l:
//   (N.r)/l^3 + tr(M)/l^3 - 3 (r^T M r)/l^5  =  ((N.u) / l) / l + (((tr M - 3 u^T M u) / l) / l) / l,
// each factor divided out in turn so that no power of l is formed: N ~ L^2 and M ~ L^3 at length scale L, and every
// intermediate stays near L^k for k <= 3 (the raw |r|^5 leaves the binary32 range at L ~ 5e7 or L ~ 1e-8).
RT_HD float far_field(const WindMoment& mo, float rx, float ry, float rz, float l) {
    const float il = fdiv(1.0f, l);
    const float ux = fmul(rx, il), uy = fmul(ry, il), uz = fmul(rz, il);
    const float nu = dot3f(mo.nx, mo.ny, mo.nz, ux, uy, uz);
    const float mux = dot3f(mo.m[0], mo.m[1], mo.m[2], ux, uy, uz);
    const float muy = dot3f(mo.m[3], mo.m[4], mo.m[5], ux, uy, uz);
    const float muz = dot3f(mo.m[6], mo.m[7], mo.m[8], ux, uy, uz);
    const float umu = dot3f(ux, uy, uz, mux, muy, muz);
    const float tr = fadd(fadd(mo.m[0], mo.m[4]), mo.m[8]);
    const float t1 = fmul(fmul(nu, il), il);
    const float t2 = fmul(fmul(fmul(fsub(tr, fmul(3.0f, umu)), il), il), il);
    return fadd(t1, t2);
}

// ------------------------------------------------------------------ moment of one node
// From the node's own triangle records (record order) and its inner children's records (slot order), so the result
// is the same whichever thread of the moment pass computes it.  `weight` is the side value the parent needs besides
// the record: the total area sum_t |A_t| of the subtree (the centroid's denominator).
//
// p~ = o + (sum_t |A_t| (c_t - o) + sum_c W_c (p~_c - o)) / W with o the node's quantisation origin (finite vertices
// near o keep the differences exact or nearly so at any offset; o = 0 if it is not finite).  W = 0 (no triangle of
// non-zero computed area): p~ = o, the documented fallback; N and M are then sums of zero vectors.
// rho: the largest of |v - p~| over the node's own finite vertices and |p~_c - p~| + rho_c over children that have any
// (rho_c > 0), then times (1 + 2^-20) plus 2^-64.  Per vertex the computed |v - p~| (three roundings in the
// differences, three in the squares and sums, one in the sqrt) is at least (1 - 4u) times the exact one, u = 2^-24,
// while the squares stay normal; a square below 2^-126 costs at most 2^-74 absolute after the sqrt, which the 2^-64
// covers; the fadd of a child's two terms is off by at most u.  The factor 1 + 16u rounded down once more still
// exceeds 1 + 5u, so rho bounds every finite vertex of the subtree in real arithmetic.  rho = 0: no finite vertex.
struct WindNodeOut { WindMoment mo; float weight; };

RT_HD void tri_area_vec(const float* v, float& x, float& y, float& z) {
    const float e1x = fsub(v[3], v[0]), e1y = fsub(v[4], v[1]), e1z = fsub(v[5], v[2]);
    const float e2x = fsub(v[6], v[0]), e2y = fsub(v[7], v[1]), e2z = fsub(v[8], v[2]);
    x = fmul(0.5f, fsub(fmul(e1y, e2z), fmul(e1z, e2y)));
    y = fmul(0.5f, fsub(fmul(e1z, e2x), fmul(e1x, e2z)));
    z = fmul(0.5f, fsub(fmul(e1x, e2y), fmul(e1y, e2x)));
}

// (v0 - p) + (v1 - p) + (v2 - p), divided by 3: the centroid relative to p
RT_HD float rel_centroid(float a, float b, float c, float p) {
    return fdiv(fadd(fadd(fsub(a, p), fsub(b, p)), fsub(c, p)), 3.0f);
}

RT_HD float dist3(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = fsub(ax, bx), dy = fsub(ay, by), dz = fsub(az, bz);
    return fsqrt(dot3f(dx, dy, dz, dx, dy, dz));
}

RT_HD void load_tri(const uint8_t* tris, uint32_t rec, float v[9]) {
    const uint8_t* tp = tris + (size_t)rec * 48u;
    const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
    v[0] = as_float(a.x); v[1] = as_float(a.y); v[2] = as_float(a.z);
    v[3] = as_float(b.x); v[4] = as_float(b.y); v[5] = as_float(b.z);
    v[6] = as_float(c.x); v[7] = as_float(c.y); v[8] = as_float(c.z);
}

// COHERENT: the moment pass, whose records other threads have just written, reads them from L2 (ld.global.cg); the
// traversal reads records that are constant for the launch and shares the top levels across all points, so it takes
// the read-only path through L1 (ld.global.nc, like the nodes).
template <bool COHERENT>
RT_HD WindMoment load_moment(const uint8_t* moments, uint32_t node) {
    const uint8_t* p = moments + (size_t)node * 64u;
    const U4 a = COHERENT ? ldcg128(p) : ldg128(p), b = COHERENT ? ldcg128(p + 16) : ldg128(p + 16),
             c = COHERENT ? ldcg128(p + 32) : ldg128(p + 32), d = COHERENT ? ldcg128(p + 48) : ldg128(p + 48);
    WindMoment m;
    m.px = as_float(a.x); m.py = as_float(a.y); m.pz = as_float(a.z); m.rho = as_float(a.w);
    m.nx = as_float(b.x); m.ny = as_float(b.y); m.nz = as_float(b.z); m.m[0] = as_float(b.w);
    m.m[1] = as_float(c.x); m.m[2] = as_float(c.y); m.m[3] = as_float(c.z); m.m[4] = as_float(c.w);
    m.m[5] = as_float(d.x); m.m[6] = as_float(d.y); m.m[7] = as_float(d.z); m.m[8] = as_float(d.w);
    return m;
}

RT_HD WindNodeOut node_moment(const uint8_t* nodes, const uint8_t* tris, uint32_t w, const uint8_t* moments,
                              const float* weights) {
    const uint8_t* np = nodes + (size_t)w * 80u;
    const U4 n0 = ldg128(np), n1 = ldg128(np + 16);
    const uint32_t nin = (uint32_t)popc32(n0.w >> 24), base = n1.x, tbase = n1.y, ntri = (uint32_t)popc32(n1.z);
    float ox = as_float(n0.x), oy = as_float(n0.y), oz = as_float(n0.z);
    if (!finite3(ox, oy, oz)) ox = oy = oz = 0.0f;
    // pass 1: total area and the area-weighted centroid
    float W = 0.0f, sx = 0.0f, sy = 0.0f, sz = 0.0f;
    for (uint32_t j = 0; j < ntri; ++j) {
        float v[9];
        load_tri(tris, tbase + j, v);
        if (!(finite3(v[0], v[1], v[2]) && finite3(v[3], v[4], v[5]) && finite3(v[6], v[7], v[8]))) continue;
        float ax, ay, az;
        tri_area_vec(v, ax, ay, az);
        const float wt = fsqrt(dot3f(ax, ay, az, ax, ay, az));
        sx = fadd(sx, fmul(wt, rel_centroid(v[0], v[3], v[6], ox)));
        sy = fadd(sy, fmul(wt, rel_centroid(v[1], v[4], v[7], oy)));
        sz = fadd(sz, fmul(wt, rel_centroid(v[2], v[5], v[8], oz)));
        W = fadd(W, wt);
    }
    for (uint32_t c = 0; c < nin; ++c) {
        const float wc = ldcgf(weights + base + c);
        if (!(wc > 0.0f)) continue;
        const U4 pc = ldcg128(moments + (size_t)(base + c) * 64u);
        sx = fadd(sx, fmul(wc, fsub(as_float(pc.x), ox)));
        sy = fadd(sy, fmul(wc, fsub(as_float(pc.y), oy)));
        sz = fadd(sz, fmul(wc, fsub(as_float(pc.z), oz)));
        W = fadd(W, wc);
    }
    WindNodeOut out;
    WindMoment& mo = out.mo;
    if (W > 0.0f) {
        mo.px = fadd(ox, fdiv(sx, W)); mo.py = fadd(oy, fdiv(sy, W)); mo.pz = fadd(oz, fdiv(sz, W));
    } else {
        mo.px = ox; mo.py = oy; mo.pz = oz;
    }
    out.weight = W;
    // pass 2: N, M and the radius about p~
    mo.nx = mo.ny = mo.nz = 0.0f;
    for (int k = 0; k < 9; ++k) mo.m[k] = 0.0f;
    float r = 0.0f;
    bool any = false;
    for (uint32_t j = 0; j < ntri; ++j) {
        float v[9];
        load_tri(tris, tbase + j, v);
        bool fin = true;
        for (int k = 0; k < 3; ++k) {
            if (finite3(v[3 * k], v[3 * k + 1], v[3 * k + 2])) {
                r = fmaxf(r, dist3(v[3 * k], v[3 * k + 1], v[3 * k + 2], mo.px, mo.py, mo.pz));
                any = true;
            } else {
                fin = false;
            }
        }
        if (!fin) continue;
        float ax, ay, az;
        tri_area_vec(v, ax, ay, az);
        const float d[3] = {rel_centroid(v[0], v[3], v[6], mo.px), rel_centroid(v[1], v[4], v[7], mo.py),
                            rel_centroid(v[2], v[5], v[8], mo.pz)};
        mo.nx = fadd(mo.nx, ax); mo.ny = fadd(mo.ny, ay); mo.nz = fadd(mo.nz, az);
        for (int i = 0; i < 3; ++i) {
            mo.m[3 * i] = fadd(mo.m[3 * i], fmul(d[i], ax));
            mo.m[3 * i + 1] = fadd(mo.m[3 * i + 1], fmul(d[i], ay));
            mo.m[3 * i + 2] = fadd(mo.m[3 * i + 2], fmul(d[i], az));
        }
    }
    for (uint32_t c = 0; c < nin; ++c) {
        const WindMoment cm = load_moment<true>(moments, base + c);
        const float d[3] = {fsub(cm.px, mo.px), fsub(cm.py, mo.py), fsub(cm.pz, mo.pz)};
        mo.nx = fadd(mo.nx, cm.nx); mo.ny = fadd(mo.ny, cm.ny); mo.nz = fadd(mo.nz, cm.nz);
        const float cn[3] = {cm.nx, cm.ny, cm.nz};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) mo.m[3 * i + j] = fadd(mo.m[3 * i + j], fadd(cm.m[3 * i + j], fmul(d[i], cn[j])));
        if (cm.rho > 0.0f) {
            r = fmaxf(r, fadd(dist3(cm.px, cm.py, cm.pz, mo.px, mo.py, mo.pz), cm.rho));
            any = true;
        }
    }
    mo.rho = any ? fadd(fmul(r, 1.00000095367431640625f), 5.42101086242752217e-20f) : 0.0f;   // 1 + 2^-20, 2^-64
    return out;
}

RT_HD void store_moment(uint8_t* moments, uint32_t node, const WindMoment& m, float* weights, float weight) {
#if defined(__CUDA_ARCH__)
    float4* p = reinterpret_cast<float4*>(moments + (size_t)node * 64u);
    __stcg(p, make_float4(m.px, m.py, m.pz, m.rho));
    __stcg(p + 1, make_float4(m.nx, m.ny, m.nz, m.m[0]));
    __stcg(p + 2, make_float4(m.m[1], m.m[2], m.m[3], m.m[4]));
    __stcg(p + 3, make_float4(m.m[5], m.m[6], m.m[7], m.m[8]));
    __stcg(weights + node, weight);
#else
    *reinterpret_cast<WindMoment*>(moments + (size_t)node * 64u) = m;
    weights[node] = weight;
#endif
}

// ------------------------------------------------------------------ traversal
// Group stack: one entry per tree level, (child_base, mask of the near inner children of that node still to visit,
// by child offset).  Children are visited in offset (= slot) order, so the order of the additions is fixed.
struct WindStackEntry { uint32_t base, mask; };

struct WindTrav {
    float x, y, z;
    float sum;           // 4 pi w accumulated so far
    uint32_t node;       // node to visit next, kNoNode = pop
    int sp;
};

RT_HD void wind_init(WindTrav& t, float x, float y, float z) {
    t.x = x; t.y = y; t.z = z; t.sum = 0.0f; t.node = 0u; t.sp = 0;
    if (!finite3(x, y, z)) t.node = kNoNode;     // the caller writes NaN for it
}

struct WindNoStats : NoStats {
    RT_HD void count_far() {}
    RT_HD uint32_t n_fars() const { return 0; }
};
struct WindStats : Stats {
    uint32_t fars = 0;
    RT_HD void count_far() { ++fars; }
    RT_HD uint32_t n_fars() const { return fars; }
};

// One node visit or one pop; returns true when the point is finished.  beta = +inf never approximates (inf * rho is
// +inf or, for rho = 0, NaN: both fail the `>`).
template <class S, class StackT>
RT_HD bool wind_step(const uint8_t* __restrict__ nodes, const uint8_t* __restrict__ tris, const uint8_t* __restrict__ moments,
                     float beta, WindTrav& t, S& st, StackT& stack) {
    if (t.node != kNoNode) {
        const uint8_t* np = nodes + (size_t)t.node * 80u;
        const U4 n0 = ldg128(np), n1 = ldg128(np + 16);
        st.count_node();
        const uint32_t nin = (uint32_t)popc32(n0.w >> 24), base = n1.x, tbase = n1.y, ntri = (uint32_t)popc32(n1.z);
        for (uint32_t j = 0; j < ntri; ++j) {
            float v[9];
            load_tri(tris, tbase + j, v);
            st.count_tri();
            t.sum = fadd(t.sum, solid_angle(t.x, t.y, t.z, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]));
        }
        uint32_t near = 0u;
        for (uint32_t c = 0; c < nin; ++c) {
            const WindMoment mo = load_moment<false>(moments, base + c);
            const float rx = fsub(mo.px, t.x), ry = fsub(mo.py, t.y), rz = fsub(mo.pz, t.z);
            const float l = fsqrt(dot3f(rx, ry, rz, rx, ry, rz));
            if (l > fmul(beta, mo.rho)) {
                st.count_far();
                t.sum = fadd(t.sum, far_field(mo, rx, ry, rz, l));
            } else {
                near |= 1u << c;
            }
        }
        if (near == 0u) {
            t.node = kNoNode;
        } else {
            t.node = base + (uint32_t)(ffs32(near) - 1);
            near &= near - 1u;
            if (near != 0u) {
                WindStackEntry e; e.base = base; e.mask = near;
                stack.push(t.sp, e);
                ++t.sp;
            }
        }
        return false;
    }
    if (t.sp > 0) {
        WindStackEntry e;
        stack.pop(t.sp - 1, e);
        t.node = e.base + (uint32_t)(ffs32(e.mask) - 1);
        e.mask &= e.mask - 1u;
        if (e.mask != 0u) stack.push(t.sp - 1, e); else --t.sp;
        return false;
    }
    return true;
}

RT_HD float wind_result(const WindTrav& t) {
    return finite3(t.x, t.y, t.z) ? fmul(t.sum, kInv4Pi) : as_float(0x7fc00000u);
}

}  // namespace rt
