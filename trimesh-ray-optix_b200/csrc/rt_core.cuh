// rt_core.cuh — data layout and per-ray arithmetic of the B200 ray/mesh intersector.
//
// Everything in this header is a pure function of its arguments (RT_HD = __host__ __device__)
// so that the same source can be stepped through by the host-side simulator under
// tests/hostsim/ (a debugging harness, never linked into libtriro_b200.so).
//
// What this replaces in the reference: the arithmetic that lives inside the closed OptiX
// runtime behind optixTrace (triro/backend/shaders.cu:86,112,163,191,238) — BVH traversal and
// the watertight ray/triangle test — plus the closest-hit attribute code of
// shaders.cu:137-153.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define RT_HD __host__ __device__ __forceinline__
#else
#define RT_HD inline
#endif

namespace rt {

// ------------------------------------------------------------------ exact float ops
// The triangle test must be evaluated with a fixed sequence of IEEE-754 binary32
// operations: (1) the edge functions of two triangles sharing an edge must be exact
// negations of each other (watertightness, Woop/Benthin/Wald 2013) which an FMA contraction
// chosen by the compiler would break; (2) the float32 mirror in oracle/ reproduces the
// sequence bit for bit.
#if defined(__CUDA_ARCH__)
RT_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
RT_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
RT_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
RT_HD float ffma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
RT_HD float fdiv(float a, float b) { return __fdiv_rn(a, b); }
RT_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
RT_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
#else
// host build is compiled with -ffp-contract=off
RT_HD float fmul(float a, float b) { return a * b; }
RT_HD float fadd(float a, float b) { return a + b; }
RT_HD float fsub(float a, float b) { return a - b; }
RT_HD float ffma(float a, float b, float c) { return fmaf(a, b, c); }
RT_HD float fdiv(float a, float b) { return a / b; }
RT_HD double dmul(double a, double b) { return a * b; }
RT_HD double dsub(double a, double b) { return a - b; }
#endif

RT_HD float sel3(int k, float x, float y, float z) { return k == 0 ? x : (k == 1 ? y : z); }
// (x,y,z) -> components (kx,ky,kz) with kx = kz+1, ky = kz+2 (mod 3); written as selects on two
// predicates so that the compiler emits SEL, not branches
RT_HD void permute3(int kz, float x, float y, float z, float& vkx, float& vky, float& vkz) {
    const bool k0 = kz == 0, k1 = kz == 1;
    vkz = k0 ? x : (k1 ? y : z);
    vkx = k0 ? y : (k1 ? z : x);
    vky = k0 ? z : (k1 ? x : y);
}

#if defined(__CUDA_ARCH__)
RT_HD float as_float(uint32_t u) { return __uint_as_float(u); }
#else
RT_HD float as_float(uint32_t u) { union { uint32_t u; float f; } c; c.u = u; return c.f; }
#endif

// Element offset of row r of a [*b, 3] batch flattened to shape[0..2] with element strides stride[0..2]; packed: the
// batch is row-major contiguous (batch_packed, rt_api.h).
RT_HD int64_t batch_offset(const int64_t shape[4], const int64_t stride[4], bool packed, int64_t r) {
    if (packed) return 3 * r;
    const int64_t i2 = r % shape[2];
    const int64_t q = r / shape[2];
    const int64_t i1 = q % shape[1];
    const int64_t i0 = q / shape[1];
    return i0 * stride[0] + i1 * stride[1] + i2 * stride[2];
}

// ------------------------------------------------------------------ layout in HBM
// Blob = [header 256 B][triangle records 48 B each][BVH8 nodes 80 B each].
// All sections are 16-byte aligned so every fetch is a 128-bit ld.global.nc.

constexpr int kLeafMaxTris = 3;    // most triangles a leaf slot can hold (unary-coded in 3 bits)
constexpr int kLeafTrisDefault = 2; // what the builder puts into one leaf slot (TRIRO_LEAF_TRIS=1..3 overrides, for experiments)
constexpr int kNodeMaxTris = 24;   // 8 slots x 3
// Upper bound of the number of wide nodes for n triangles.  A bottom node holds more than leaf_max triangles
// (else it would have been a leaf slot of its parent), upper levels add at most 1/7 on top.
RT_HD uint32_t wide_node_cap(int64_t n, int leaf_max) {
    const int64_t m = n > 0 ? n : 0;
    return (uint32_t)(leaf_max >= 3 ? m / 3 + 2 : (leaf_max == 2 ? (2 * m) / 5 + 2 : (5 * m) / 8 + 2));
}
constexpr int kMaxDepth = 60;      // wide-tree levels the traversal stack can hold

struct alignas(16) TriRecord {     // 48 B: three 128-bit loads
    float v0x, v0y, v0z;
    int32_t prim;                  // row of `faces` (reference: optixGetPrimitiveIndex)
    float v1x, v1y, v1z;
    uint32_t pad1;
    float v2x, v2y, v2z;
    uint32_t pad2;
};
static_assert(sizeof(TriRecord) == 48, "TriRecord must be 48 bytes");

// Compressed 8-wide node after Ylitie, Karras, Laine 2017 (80 B: five 128-bit loads).
// Child boxes are quantised to 8 bits per plane relative to (p, 2^e):
//   plane = p + q * 2^(e-127)    (lo planes rounded down, hi planes rounded up)
// Slot s (0..7) holds either an inner child (bit s of imask), a leaf of 1..3 triangles
// (unary count 001/011/111 in bits [3s, 3s+3) of trimask) or nothing.  Inner children are
// contiguous from child_base in slot order, triangles contiguous from tri_base in bit order:
//   child index    = child_base + popc(imask   & ((1 << s) - 1))
//   triangle index = tri_base   + popc(trimask & ((1 << b) - 1))
struct alignas(16) Node8 {
    float px, py, pz;
    uint8_t ex, ey, ez, imask;
    uint32_t child_base;           // index of the first inner child
    uint32_t tri_base;             // index of this node's first triangle record
    uint32_t trimask;              // 24 bits, 3 per slot
    uint32_t reserved;
    uint8_t qlox[8], qloy[8], qloz[8];
    uint8_t qhix[8], qhiy[8], qhiz[8];
};
static_assert(sizeof(Node8) == 80, "Node8 must be 80 bytes");

struct U4 { uint32_t x, y, z, w; };

// ------------------------------------------------------------------ ray set-up
struct Ray {
    float ox, oy, oz;
    // watertight test set-up: kzf = kz | 4 * (d[kz] > 0); the direction itself is not kept (registers)
    int kzf;
    float Sx, Sy, Sz;
    float okx, oky, okz;           // origin permuted to (kx, ky, kz)
    // slab test set-up
    float idx, idy, idz;           // 1/d with zero components replaced by +-tiny
    uint32_t octinv;               // 7 - octant, octant bit a = (d_a < 0)
    // kByteMagic (0x47000000 = 32768.0f), passed in at run time on the device: it must live in
    // a register so that node_test's PRMT can take the byte selector as its one immediate
    uint32_t magic;
};
constexpr uint32_t kByteMagic = 0x47000000u;

// 1/d with zero components replaced by +-tiny; returns octinv = 7 - octant (octant bit a = (d_a < 0)).
RT_HD uint32_t ray_inverse(float dx, float dy, float dz, float& idx, float& idy, float& idz) {
    const float tiny = 1e-20f;
    const float sx = fabsf(dx) < tiny ? (signbit(dx) ? -tiny : tiny) : dx;
    const float sy = fabsf(dy) < tiny ? (signbit(dy) ? -tiny : tiny) : dy;
    const float sz = fabsf(dz) < tiny ? (signbit(dz) ? -tiny : tiny) : dz;
    idx = 1.0f / sx; idy = 1.0f / sy; idz = 1.0f / sz;
    const uint32_t oct = (sx < 0.0f ? 1u : 0u) | (sy < 0.0f ? 2u : 0u) | (sz < 0.0f ? 4u : 0u);
    return 7u - oct;
}

RT_HD void ray_setup(Ray& r, float ox, float oy, float oz, float dx, float dy, float dz) {
    r.ox = ox; r.oy = oy; r.oz = oz;
    // kz = dimension where |d| is maximal (first maximum in x,y,z order)
    int kz = 0;
    float m = fabsf(dx);
    if (fabsf(dy) > m) { kz = 1; m = fabsf(dy); }
    if (fabsf(dz) > m) { kz = 2; }
    const int kx = kz == 2 ? 0 : kz + 1;
    const int ky = kx == 2 ? 0 : kx + 1;
    const float dkx = sel3(kx, dx, dy, dz), dky = sel3(ky, dx, dy, dz), dkz = sel3(kz, dx, dy, dz);
    // (the Woop kx/ky swap for d[kz] < 0 only flips the sign of U,V,W; it is folded into
    //  the front-face decision instead, see tri_front())
    r.Sx = fdiv(dkx, dkz);
    r.Sy = fdiv(dky, dkz);
    r.Sz = fdiv(1.0f, dkz);
    r.okx = sel3(kx, ox, oy, oz);
    r.oky = sel3(ky, ox, oy, oz);
    r.okz = sel3(kz, ox, oy, oz);
    r.octinv = ray_inverse(dx, dy, dz, r.idx, r.idy, r.idz);
    r.magic = kByteMagic;
    r.kzf = kz | (dkz > 0.0f ? 4 : 0);
}

// ------------------------------------------------------------------ watertight triangle test
// Woop, Benthin, Wald, "Watertight Ray/Triangle Intersection", JCGT 2013, in binary32 with a
// binary64 fallback when an edge function is exactly zero.  Reports a hit iff the sheared
// origin lies inside or on the boundary of the triangle and det != 0; returns
//   t = T/det, and the unnormalised barycentrics U (weight of v0), V (v1), W (v2), det = U+V+W.
// The caller applies the open interval 0 < t < tmax (reference: tmin 0, tmax 1e7).
struct TriHit { float t, U, V, W, det; };

RT_HD bool tri_test(const Ray& r, float v0x, float v0y, float v0z, float v1x, float v1y, float v1z,
                    float v2x, float v2y, float v2z, TriHit& h) {
    float Akx, Aky, Akz, Bkx, Bky, Bkz, Ckx, Cky, Ckz;
    permute3(r.kzf & 3, v0x, v0y, v0z, Akx, Aky, Akz);
    permute3(r.kzf & 3, v1x, v1y, v1z, Bkx, Bky, Bkz);
    permute3(r.kzf & 3, v2x, v2y, v2z, Ckx, Cky, Ckz);
    Akx = fsub(Akx, r.okx); Aky = fsub(Aky, r.oky); Akz = fsub(Akz, r.okz);
    Bkx = fsub(Bkx, r.okx); Bky = fsub(Bky, r.oky); Bkz = fsub(Bkz, r.okz);
    Ckx = fsub(Ckx, r.okx); Cky = fsub(Cky, r.oky); Ckz = fsub(Ckz, r.okz);
    const float Ax = ffma(-r.Sx, Akz, Akx), Ay = ffma(-r.Sy, Akz, Aky);
    const float Bx = ffma(-r.Sx, Bkz, Bkx), By = ffma(-r.Sy, Bkz, Bky);
    const float Cx = ffma(-r.Sx, Ckz, Ckx), Cy = ffma(-r.Sy, Ckz, Cky);
    float U = fsub(fmul(Cx, By), fmul(Cy, Bx));
    float V = fsub(fmul(Ax, Cy), fmul(Ay, Cx));
    float W = fsub(fmul(Bx, Ay), fmul(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        const double Ud = dsub(dmul((double)Cx, (double)By), dmul((double)Cy, (double)Bx));
        const double Vd = dsub(dmul((double)Ax, (double)Cy), dmul((double)Ay, (double)Cx));
        const double Wd = dsub(dmul((double)Bx, (double)Ay), dmul((double)By, (double)Ax));
        if ((Ud < 0.0 || Vd < 0.0 || Wd < 0.0) && (Ud > 0.0 || Vd > 0.0 || Wd > 0.0)) return false;
        U = (float)Ud; V = (float)Vd; W = (float)Wd;
    } else {
        if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    }
    const float det = fadd(fadd(U, V), W);
    if (!(det != 0.0f)) return false;   // det == 0: degenerate / edge-on.  A NaN det passes here (NaN != 0) and leaves t = NaN,
                                        // which every visitor drops with its `t > 0` test
    const float Az = fmul(r.Sz, Akz), Bz = fmul(r.Sz, Bkz), Cz = fmul(r.Sz, Ckz);
    const float T = ffma(U, Az, ffma(V, Bz, fmul(W, Cz)));
    h.t = fdiv(T, det);
    h.U = U; h.V = V; h.W = W; h.det = det;
    return true;
}

// front face = triangle seen counter-clockwise from the ray origin, i.e.
// dot(d, (v1-v0) x (v2-v0)) < 0 (reference: optixIsFrontFaceHit, shaders.cu:151).
// With the fixed cyclic (kx,ky,kz) the sheared edge functions carry the sign of
// -dot(d, n) * sign(d[kz]) ... so: front <=> (det > 0) == (d[kz] > 0).
RT_HD bool tri_front(const Ray& r, const TriHit& h) {
    return (h.det > 0.0f) == ((r.kzf & 4) != 0);
}

// Closest-hit attributes exactly as the reference computes them (shaders.cu:137-153):
//   (u,v) = OptiX barycentrics = weights of v1, v2;  loc = u*v1 + v*v2 + (1-u-v)*v0;
//   returned uv = (1-u-v, u) = (weight of v0, weight of v1).
struct HitAttr { float lx, ly, lz, uv0, uv1; };
RT_HD HitAttr tri_attr(const TriHit& h, float v0x, float v0y, float v0z, float v1x, float v1y, float v1z,
                       float v2x, float v2y, float v2z) {
    const float bu = fdiv(h.V, h.det);
    const float bv = fdiv(h.W, h.det);
    const float w0 = fsub(fsub(1.0f, bu), bv);
    HitAttr a;
    a.lx = ffma(bu, v1x, ffma(bv, v2x, fmul(w0, v0x)));
    a.ly = ffma(bu, v1y, ffma(bv, v2y, fmul(w0, v0y)));
    a.lz = ffma(bu, v1z, ffma(bv, v2z, fmul(w0, v0z)));
    a.uv0 = w0;
    a.uv1 = bu;
    return a;
}

// ------------------------------------------------------------------ BVH8 node test
// Returns the 32-bit hit mask of Ylitie et al.: bits 24..31 = hit inner children ordered by
// traversal priority (bit 24 + (slot ^ octinv)), bits 0..23 = triangles of hit leaf slots
// (bit positions of trimask).
//
// Slab test, conservative and branch-free.  With a = 2^e * idir, b = (p - o) * idir a plane
// sits at t = q*a + b.  The byte q is turned into a float without an I2F: PRMT drops it into
// bits 8..15 of 0x47000000, which reads 32768 + q, and the 32768*a is pre-subtracted from b:
//   t = fma(32768 + q, a, b - 32768*a)
// Rounding: |error| <= ~6u(256|a| + |b|) + |a|/512, u = 2^-24; that margin is subtracted from
// the near and added to the far planes.  NaNs drop out of fminf/fmaxf, which only widens.
#if defined(__CUDA_ARCH__)
// byte I of w -> bits 8..15 of `magic` (= 0x47000000 held in a register so that the selector
// can be the PRMT immediate)
template <int I>
RT_HD float byte_plus_32768(uint32_t w, uint32_t magic) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(magic), "n"(0x7604 | (I << 4)));
    return __uint_as_float(d);
}
#else
template <int I>
RT_HD float byte_plus_32768(uint32_t w, uint32_t magic) {
    return as_float(magic | (((w >> (8u * I)) & 0xffu) << 8));
}
#endif

// (acc << 1) | signbit(x)
#if defined(__CUDA_ARCH__)
RT_HD uint32_t shift_in_sign(float x, uint32_t acc) { return __funnelshift_l(__float_as_uint(x), acc, 1); }
#else
RT_HD uint32_t shift_in_sign(float x, uint32_t acc) {
    union { float f; uint32_t u; } c; c.f = x;
    return (acc << 1) | (c.u >> 31);
}
#endif

RT_HD uint32_t spread3(uint32_t x) {   // bit i (0..7) -> bit 3i
    x = (x | (x << 8)) & 0x0000f00fu;
    x = (x | (x << 4)) & 0x000c30c3u;
    x = (x | (x << 2)) & 0x00249249u;
    return x;
}

// hm8 (slot hit mask) -> Ylitie hit mask: inner hits moved to priority position (slot ^ octinv) in
// bits 24..31, triangle bits (3 per slot) masked by trimask in bits 0..23.
RT_HD uint32_t permute_by_octant(uint32_t in8, uint32_t octinv) {   // three conditional delta swaps
    const uint32_t m1 = (octinv & 1u) ? 0x55u : 0u, m2 = (octinv & 2u) ? 0x33u : 0u, m4 = (octinv & 4u) ? 0x0fu : 0u;
    uint32_t t;
    t = ((in8 >> 1) ^ in8) & m1; in8 ^= t | (t << 1);
    t = ((in8 >> 2) ^ in8) & m2; in8 ^= t | (t << 2);
    t = ((in8 >> 4) ^ in8) & m4; in8 ^= t | (t << 4);
    return in8;
}
#if defined(__CUDACC__) && defined(RT_MASK_LUT)
// Shared-memory lookup tables for the two bit permutations: ~30 ALU-pipe instructions per node
// become two LDS (the ALU pipe is the traversal kernel's bottleneck, the LSU pipe is idle).
__shared__ uint32_t g_lut_spread7[256];     // spread3(x) * 7
__shared__ uint8_t g_lut_perm[8][256];      // permute_by_octant(x, o)
__device__ __forceinline__ void init_mask_luts() {
    for (uint32_t i = threadIdx.x; i < 256u; i += blockDim.x) g_lut_spread7[i] = spread3(i) * 7u;
    for (uint32_t i = threadIdx.x; i < 2048u; i += blockDim.x) g_lut_perm[i >> 8][i & 255u] = (uint8_t)permute_by_octant(i & 255u, i >> 8);
    __syncthreads();
}
#endif
RT_HD uint32_t finish_masks(uint32_t hm8, uint32_t imask, uint32_t trimask, uint32_t octinv) {
#if defined(__CUDA_ARCH__) && defined(RT_MASK_LUT)
    const uint32_t in8 = g_lut_perm[octinv][hm8 & imask];
    return (in8 << 24) | (g_lut_spread7[hm8] & trimask);
#else
    return (permute_by_octant(hm8 & imask, octinv) << 24) | ((spread3(hm8) * 7u) & trimask);
#endif
}

// The ray interval is (0, tmax): `tmin` is kept in the signature for the call sites' readability and must be 0.
RT_HD uint32_t node_test(const Ray& r, const U4& n0, const U4& n1, const U4& n2, const U4& n3, const U4& n4,
                         float tmin, float tmax) {
    (void)tmin;
    const float px = as_float(n0.x), py = as_float(n0.y), pz = as_float(n0.z);
    const float sx = as_float((n0.w & 0xffu) << 23);
    const float sy = as_float(((n0.w >> 8) & 0xffu) << 23);
    const float sz = as_float(((n0.w >> 16) & 0xffu) << 23);
    const float ax = sx * r.idx, ay = sy * r.idy, az = sz * r.idz;
    const float bx = (px - r.ox) * r.idx, by = (py - r.oy) * r.idy, bz = (pz - r.oz) * r.idz;
    const float ku = 3.6e-7f;            // 6 * 2^-24
    const float kq = 256.0f * ku + 0.00390625f;   // + 1/256 for the pre-subtraction
    const float ex = fmaf(kq, fabsf(ax), ku * fabsf(bx));
    const float ey = fmaf(kq, fabsf(ay), ku * fabsf(by));
    const float ez = fmaf(kq, fabsf(az), ku * fabsf(bz));
    const float cnx = fmaf(-32768.0f, ax, bx - ex), cfx = fmaf(-32768.0f, ax, bx + ex);
    const float cny = fmaf(-32768.0f, ay, by - ey), cfy = fmaf(-32768.0f, ay, by + ey);
    const float cnz = fmaf(-32768.0f, az, bz - ez), cfz = fmaf(-32768.0f, az, bz + ez);
    // near/far plane bytes by ray octant: d >= 0 -> near = lo, far = hi
    const bool negx = r.idx < 0.0f, negy = r.idy < 0.0f, negz = r.idz < 0.0f;
    // words: n2 = (qlox[0..3], qlox[4..7], qloy[0..3], qloy[4..7])
    //        n3 = (qloz[0..3], qloz[4..7], qhix[0..3], qhix[4..7])
    //        n4 = (qhiy[0..3], qhiy[4..7], qhiz[0..3], qhiz[4..7])
    // miss bits are collected from the sign of (tf - tn) with a funnel shift: FADD runs on the FMA
    // pipe, leaving one ALU-pipe instruction per child (the ALU pipe is the kernel's bottleneck)
    uint32_t miss = 0;
    const uint32_t magic = r.magic;
#pragma unroll
    for (int half = 1; half >= 0; --half) {
        const uint32_t lox = half ? n2.y : n2.x, loy = half ? n2.w : n2.z, loz = half ? n3.y : n3.x;
        const uint32_t hix = half ? n3.w : n3.z, hiy = half ? n4.y : n4.x, hiz = half ? n4.w : n4.z;
        const uint32_t nx = negx ? hix : lox, fx = negx ? lox : hix;
        const uint32_t ny = negy ? hiy : loy, fy = negy ? loy : hiy;
        const uint32_t nz = negz ? hiz : loz, fz = negz ? loz : hiz;
        // A slot is missed iff min(tf, tmax) < max(tn, 0): clamp, subtract, collect the sign with a funnel shift.  (Sign-bit
        // tests without the clamps and packed FFMA2 plane arithmetic were measured slower, DESIGN.md 4.1.)
#define RT_SLAB(I)                                                                                              \
        {                                                                                                       \
            const float tnx = fmaf(byte_plus_32768<I>(nx, magic), ax, cnx), tfx = fmaf(byte_plus_32768<I>(fx, magic), ax, cfx); \
            const float tny = fmaf(byte_plus_32768<I>(ny, magic), ay, cny), tfy = fmaf(byte_plus_32768<I>(fy, magic), ay, cfy); \
            const float tnz = fmaf(byte_plus_32768<I>(nz, magic), az, cnz), tfz = fmaf(byte_plus_32768<I>(fz, magic), az, cfz); \
            const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));                                          \
            const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmax));                                          \
            miss = shift_in_sign(tf - tn, miss);                                                                \
        }
        RT_SLAB(3) RT_SLAB(2) RT_SLAB(1) RT_SLAB(0)
#undef RT_SLAB
    }
    const uint32_t hm8 = ~miss & 0xffu;
    return finish_masks(hm8, n0.w >> 24, n1.z, r.octinv);
}

// Work index -> pixel index of an image of width `width` (a multiple of the tile width) traced in tiles of
// 2^w_log2 x (32 >> w_log2) pixels: 32 consecutive work items are one tile, tiles run row-major.  A bijection on
// [0, H * width) when H is a multiple of the tile height (tests/test_hostsim_logic.py).
RT_HD uint32_t tile_map(uint32_t t, uint32_t tiles_per_row, uint32_t width, uint32_t w_log2) {
    const uint32_t tile_w = 1u << w_log2, tile_h = 32u >> w_log2;
    const uint32_t tile = t >> 5, j = t & 31u;
    const uint32_t trow = tile / tiles_per_row, tcol = tile - trow * tiles_per_row;
    return (trow * tile_h + (j >> w_log2)) * width + tcol * tile_w + (j & (tile_w - 1u));
}

// The box that bounds every child slot of a node, in the node's quantised frame: smallest lower and largest upper
// plane byte per axis (empty slots are stored inverted, 255 / 0, and drop out), as the floats 32768 + q node_test feeds
// into its FMAs.
struct RootFrame { float px, py, pz, sx, sy, sz, lox, loy, loz, hix, hiy, hiz; };
RT_HD uint32_t bytes_min(uint32_t a, uint32_t b) {
    uint32_t m = 255u;
    for (int i = 0; i < 4; ++i) { const uint32_t x = (a >> (8 * i)) & 0xffu, y = (b >> (8 * i)) & 0xffu; m = x < m ? x : m; m = y < m ? y : m; }
    return m;
}
RT_HD uint32_t bytes_max(uint32_t a, uint32_t b) {
    uint32_t m = 0u;
    for (int i = 0; i < 4; ++i) { const uint32_t x = (a >> (8 * i)) & 0xffu, y = (b >> (8 * i)) & 0xffu; m = x > m ? x : m; m = y > m ? y : m; }
    return m;
}
RT_HD RootFrame root_frame(const U4& n0, const U4& n2, const U4& n3, const U4& n4) {
    RootFrame f;
    f.px = as_float(n0.x); f.py = as_float(n0.y); f.pz = as_float(n0.z);
    f.sx = as_float((n0.w & 0xffu) << 23); f.sy = as_float(((n0.w >> 8) & 0xffu) << 23); f.sz = as_float(((n0.w >> 16) & 0xffu) << 23);
    f.lox = 32768.0f + (float)bytes_min(n2.x, n2.y); f.loy = 32768.0f + (float)bytes_min(n2.z, n2.w); f.loz = 32768.0f + (float)bytes_min(n3.x, n3.y);
    f.hix = 32768.0f + (float)bytes_max(n3.z, n3.w); f.hiy = 32768.0f + (float)bytes_max(n4.x, n4.y); f.hiz = 32768.0f + (float)bytes_max(n4.z, n4.w);
    return f;
}

// true: the ray misses that box under node_test's own arithmetic (same a, b, margins, plane FMAs and clamp).  fmaf
// is monotone in the plane byte, so each slot's near plane is >= and its far plane <= the frame's: a ray rejected here is
// rejected by every slot of the node.
RT_HD bool frame_missed(float ox, float oy, float oz, float idx, float idy, float idz, const RootFrame& f, float tmax) {
    const float ax = f.sx * idx, ay = f.sy * idy, az = f.sz * idz;
    const float bx = (f.px - ox) * idx, by = (f.py - oy) * idy, bz = (f.pz - oz) * idz;
    const float ku = 3.6e-7f;
    const float kq = 256.0f * ku + 0.00390625f;
    const float ex = fmaf(kq, fabsf(ax), ku * fabsf(bx));
    const float ey = fmaf(kq, fabsf(ay), ku * fabsf(by));
    const float ez = fmaf(kq, fabsf(az), ku * fabsf(bz));
    const float cnx = fmaf(-32768.0f, ax, bx - ex), cfx = fmaf(-32768.0f, ax, bx + ex);
    const float cny = fmaf(-32768.0f, ay, by - ey), cfy = fmaf(-32768.0f, ay, by + ey);
    const float cnz = fmaf(-32768.0f, az, bz - ez), cfz = fmaf(-32768.0f, az, bz + ez);
    const bool negx = idx < 0.0f, negy = idy < 0.0f, negz = idz < 0.0f;
    const float tnx = fmaf(negx ? f.hix : f.lox, ax, cnx), tfx = fmaf(negx ? f.lox : f.hix, ax, cfx);
    const float tny = fmaf(negy ? f.hiy : f.loy, ay, cny), tfy = fmaf(negy ? f.loy : f.hiy, ay, cfy);
    const float tnz = fmaf(negz ? f.hiz : f.loz, az, cnz), tfz = fmaf(negz ? f.loz : f.hiz, az, cfz);
    const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));
    const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmax));
    return shift_in_sign(tf - tn, 0u) != 0u;
}

}  // namespace rt
