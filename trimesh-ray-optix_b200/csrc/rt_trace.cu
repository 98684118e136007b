// rt_trace.cu — persistent traversal kernels (sm_100a) and the rt_trace_* / rt_allhits_trace /
// rt_contains_parity / rt_trace_stats entry points.
//
// Replaces the five OptiX pipelines of the reference (sbtdef.h:37-42): the launchers
// intersectsAny/First/Closest/Count/Location (triro/backend/ray.cpp:161-378) and their device
// programs (triro/backend/shaders.cu:67-246), including the strided ray fetch getRay
// (shaders.cu:27-63).
//
// Execution model: persistent CTAs (grid = SMs x resident CTAs), one ray per lane.  A warp
// advances all its rays one wide node at a time and, whenever too few lanes are still busy,
// retires the finished rays and re-fills those lanes from a global ray counter with one
// warp-aggregated atomic (Aila & Laine 2009).  Two schedule families give bit-identical results
// (rt_trace_opts::schedule, DESIGN.md 4.1):
//   this file           k_trace<MODE, STATS>: every lane tests its own triangles inside the node step (direct;
//                       the reference path the host simulation reproduces)
//   rt_trace_coop.cuh   k_trace_coop: (triangle, lane) pairs in a warp-shared list, tested by all 32 lanes -
//                       the default for every query (coherent and incoherent variants)
// launch() below resolves rt_trace_opts (tmax, ray window, schedule, knobs) - there is no state
// behind a call: no environment variable, no thread-local setting, one kernel launch.
#include <stdlib.h>
#include <type_traits>
#define RT_MASK_LUT 1
#include "rt_api.h"
#include "rt_traverse.cuh"

namespace rt {

enum TraceMode { kClosest = 0, kFirst = 1, kAny = 2, kCount = 3, kAllHits = 4, kContains = 5 };

constexpr int kTraceThreads = 128;

struct TraceParams {
    const uint8_t* blob;
    rt_ray_desc rays;
    int64_t ray_first;           // window [ray_first, ray_first + nray) of the descriptor's index space; outputs are
    int64_t nray;                // indexed by (ray - ray_first)
    int o_mode, d_mode;          // kGeneral / kPacked (offset 3*r) / kConstant (offset 0) / kGeneral32
    int refill_threshold, tri_threshold;
    float tmax;
    uint32_t byte_magic;         // rt::kByteMagic, kept opaque to ptxas (see rt_core.cuh)
    unsigned long long* ray_counter;
    // outputs (per mode)
    uint8_t* hit;
    uint8_t* front;
    int32_t* tri;
    float* loc;
    float* uv;
    int32_t* count;
    // all hits
    int max_hits;
    uint4* staging;
    // contains
    float dir[3], aabb_lo[3], aabb_hi[3];
    const uint8_t* active;       // optional per-point mask (may alias `broken`)
    int stop_on_broken;          // RT_OPT_STOP_WHEN_BROKEN
    int share_lanes;             // !RT_OPT_NO_LANE_SHARING
    // coherent image batches [.., H, W, 3]: work index -> ray index by 8x4-pixel tiles (0 = identity), see tile_order();
    // tile_hw is unused and only holds the offsets of the fields after it
    uint32_t tile_per_row, tile_w, tile_hw;
    uint8_t* contain;
    uint8_t* broken;
    int32_t* flags;
    // instrumentation
    unsigned long long* counters;
    // fused pinhole ray generation (o_mode == kPinhole): r -> pixel (x = r % w, y = r / w)
    long long cam_w;
    float cam_half_w, cam_half_h, cam_f;
    float cam_mat[9], cam_origin[3];
};

// Every launch leaves its scratch zeroed: the last CTA to finish resets the ray counter and the CTA count, so the
// next call on the same stream can skip its memset (RT_OPT_SCRATCH_ZEROED) and a launch is a single kernel.
__device__ __forceinline__ void release_scratch(const TraceParams& p);

// Work order of coherent image batches.  Lanes draw consecutive WORK indices; with the identity a warp holds 32
// consecutive pixels of one row.  For a batch shaped [.., H, W, 3] with H % 4 == 0 and W % 8 == 0 the work index is
// mapped to the ray index so that 32 consecutive work items are an 8x4-pixel tile: the rays of a warp then visit
// fewer distinct leaf-level nodes per step (fewer L1 lines per request), and a warp on the silhouette of an object
// mixes grazing rays with short ones (idle lanes for lane sharing).  Results are indexed by ray, so nothing else changes.
#ifndef RT_TILE_W_LOG2
#define RT_TILE_W_LOG2 3
#endif
constexpr uint32_t kTileWLog2 = RT_TILE_W_LOG2, kTileW = 1u << kTileWLog2, kTileH = 32u >> kTileWLog2;   // 8 x 4 pixels per warp
__device__ __forceinline__ int64_t tile_order(const TraceParams& p, int64_t w) {
    if (p.tile_per_row == 0u) return w;
    const uint32_t t = (uint32_t)w;                         // one image (launch() enables tiles for those only)
    return (int64_t)tile_map(t, p.tile_per_row, p.tile_w, kTileWLog2);
}

enum FetchMode { kGeneral = 0, kPacked = 1, kConstant = 2, kGeneral32 = 3, kPinhole = 4 };

__device__ __forceinline__ int64_t ray_offset(const int64_t shape[4], const int64_t stride[4], int mode, int64_t r) {
    if (mode == kPacked) return 3 * r;
    if (mode == kConstant) return 0;
    if (mode == kGeneral32) {   // fewer than 2^31 rays: 32-bit divisions
        const uint32_t s2 = (uint32_t)shape[2], s1 = (uint32_t)shape[1], rr = (uint32_t)r;
        const uint32_t q = rr / s2, i2 = rr - q * s2;
        const uint32_t i0 = q / s1, i1 = q - i0 * s1;
        return (int64_t)i0 * stride[0] + (int64_t)i1 * stride[1] + (int64_t)i2 * stride[2];
    }
    const int64_t i2 = r % shape[2];
    const int64_t q = r / shape[2];
    const int64_t i1 = q % shape[1];
    const int64_t i0 = q / shape[1];
    return i0 * stride[0] + i1 * stride[1] + i2 * stride[2];
}

// Origin and direction of ray r: strided fetch (reference getRay, shaders.cu:35-63), the fixed direction
// of contains_points, or a pinhole camera ray generated in registers (reference gen_rays,
// test/performance_test.py:10-20: d = normalize(x - (w-1)/2, y - (h-1)/2, -f) @ cam_mat^T).
template <int MODE>
__device__ __forceinline__ void load_ray(const TraceParams& p, int64_t r_local, float& ox, float& oy, float& oz, float& dx,
                                         float& dy, float& dz) {
    const int64_t r = r_local + p.ray_first;     // index in the descriptor's space (rt_trace_opts::ray_first)
    if (p.o_mode == kPinhole) {
        const long long y = r / p.cam_w, x = r - y * p.cam_w;
        const float px = (float)x - p.cam_half_w, py = (float)y - p.cam_half_h, pz = -p.cam_f;
        const float n = sqrtf(px * px + py * py + pz * pz);
        const float cx = px / n, cy = py / n, cz = pz / n;
        dx = cx * p.cam_mat[0] + cy * p.cam_mat[1] + cz * p.cam_mat[2];
        dy = cx * p.cam_mat[3] + cy * p.cam_mat[4] + cz * p.cam_mat[5];
        dz = cx * p.cam_mat[6] + cy * p.cam_mat[7] + cz * p.cam_mat[8];
        ox = p.cam_origin[0]; oy = p.cam_origin[1]; oz = p.cam_origin[2];
        return;
    }
    const int64_t oo = ray_offset(p.rays.shape, p.rays.o_stride, p.o_mode, r);
    const int64_t os = p.rays.o_stride[3];
    ox = p.rays.origins[oo]; oy = p.rays.origins[oo + os]; oz = p.rays.origins[oo + 2 * os];
    if (MODE == kContains) {
        dx = p.dir[0]; dy = p.dir[1]; dz = p.dir[2];
    } else {
        const int64_t dd = ray_offset(p.rays.shape, p.rays.d_stride, p.d_mode, r);
        const int64_t ds = p.rays.d_stride[3];
        dx = p.rays.directions[dd]; dy = p.rays.directions[dd + ds]; dz = p.rays.directions[dd + 2 * ds];
    }
}

// records up to max_hits (tri, loc) per ray in traversal order, like the reference's
// __anyhit__intersectsLocation (shaders.cu:207-224), while counting every hit
template <class S>
struct AllHitsVisitor : S {
    float tmax;
    int32_t count = 0;
    int max_hits = 0;
    uint4* out = nullptr;
    const uint8_t* tris = nullptr;
    __device__ __forceinline__ explicit AllHitsVisitor(float tmax0) : tmax(tmax0) {}
    __device__ __forceinline__ bool hit(const Ray&, const TriHit& h, int32_t prim, uint32_t slot) {
        if (h.t > 0.0f && h.t < tmax) {
            if (count < max_hits) {
                const uint8_t* tp = tris + (size_t)slot * 48u;
                const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
                const HitAttr at = tri_attr(h, as_float(a.x), as_float(a.y), as_float(a.z), as_float(b.x),
                                            as_float(b.y), as_float(b.z), as_float(c.x), as_float(c.y), as_float(c.z));
                out[count] = make_uint4((uint32_t)prim, __float_as_uint(at.lx), __float_as_uint(at.ly),
                                        __float_as_uint(at.lz));
            }
            ++count;
        }
        return false;
    }
};

template <int MODE, class S>
struct VisitorOf {
    using type = typename std::conditional<
        MODE == kClosest || MODE == kFirst, ClosestVisitor<S>,
        typename std::conditional<MODE == kAny, AnyVisitor<S>,
                                  typename std::conditional<MODE == kAllHits, AllHitsVisitor<S>, CountVisitor<S>>::type>::type>::type;
};

// A warp re-fills its finished lanes from the global ray counter as soon as fewer than
// `refill_threshold` lanes are still busy (defaults below; TRIRO_REFILL_THRESHOLD overrides).
constexpr int kRefillThresholdCoopIncoherent = 26;   // sweep r: heightfields best at 24-26, soup at 26-28 (profiles/r2_sweeps.md)
constexpr int kRefillThresholdDirect = 8;
// warp-cooperative schedules (rt_trace_coop.cuh): pairs listed before the warp tests them
constexpr int kPairThresholdCoherent = 16;
constexpr int kPairThresholdIncoherent = 24;
constexpr int kPoolWords = 13;   // prepared ray: o, S, o permuted, 1/d, packed (kzf | octinv << 8)

// Per-lane schedule (direct): the triangles of a hit leaf slot are tested inside the node step by the lane that found
// them.  The host simulation (tests/hostsim) reproduces this kernel node for node.
#ifndef RT_TRACE_MIN_BLOCKS
#define RT_TRACE_MIN_BLOCKS 7
#endif
#ifndef RT_TRACE_MIN_BLOCKS_LIGHT      // cooperative kernels other than pooled closest-hit: 64 registers, 8 CTAs per SM
#define RT_TRACE_MIN_BLOCKS_LIGHT 8
#endif
template <int MODE, bool STATS>
__global__ void __launch_bounds__(kTraceThreads, RT_TRACE_MIN_BLOCKS) k_trace(const __grid_constant__ TraceParams p) {
    using S = typename std::conditional<STATS, Stats, NoStats>::type;
    using Vis = typename VisitorOf<MODE, S>::type;
    init_mask_luts();
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(p.blob);
    const uint8_t* tris = p.blob + hdr->tris_offset;
    const uint8_t* nodes = p.blob + hdr->nodes_offset;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t nray = p.nray;
    PairStack stack;
    unsigned long long st_nodes = 0, st_tris = 0, st_rays = 0, st_hits = 0;
    bool any_inside = false, any_broken = false;

    Vis vis(p.tmax);
    Trav tv;
    Ray ray;
    int64_t r = -1;
    bool active = false, exhausted = false;
    bool nodes_done = true;          // this lane's ray has no node work left
    int phase = 0;
    int32_t count_plus = 0;
    trav_init(tv);

    for (;;) {
        // ---- 1. retire finished rays, re-fill free lanes
        const bool finished = active && nodes_done;
        const unsigned free_lanes = __ballot_sync(0xffffffffu, !active || finished);
        const int busy = 32 - __popc(free_lanes);
        if (free_lanes != 0u && busy < (exhausted ? 1 : p.refill_threshold)) {
            if (finished) {
                if (STATS) { st_nodes += vis.n_nodes(); st_tris += vis.n_tris(); ++st_rays; }
                if constexpr (MODE == kClosest || MODE == kFirst) {
                    if (STATS) st_hits += vis.prim >= 0;
                    if (MODE == kFirst) {
                        if (p.tri) p.tri[r] = vis.prim;
                    } else if (p.hit) {
                        if (vis.prim >= 0) {
                            const uint8_t* tp = tris + (size_t)vis.slot * 48u;
                            const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
                            const float v0x = as_float(a.x), v0y = as_float(a.y), v0z = as_float(a.z);
                            const float v1x = as_float(b.x), v1y = as_float(b.y), v1z = as_float(b.z);
                            const float v2x = as_float(c.x), v2y = as_float(c.y), v2z = as_float(c.z);
                            TriHit h;
                            tri_test(ray, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z, h);
                            const HitAttr at = tri_attr(h, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z);
                            p.hit[r] = 1; p.front[r] = tri_front(ray, h) ? 1 : 0; p.tri[r] = vis.prim;
                            p.loc[3 * r] = at.lx; p.loc[3 * r + 1] = at.ly; p.loc[3 * r + 2] = at.lz;
                            p.uv[2 * r] = at.uv0; p.uv[2 * r + 1] = at.uv1;
                        } else {
                            // reference miss program: shaders.cu:128-135
                            p.hit[r] = 0; p.front[r] = 0; p.tri[r] = -1;
                            p.loc[3 * r] = 0.f; p.loc[3 * r + 1] = 0.f; p.loc[3 * r + 2] = 0.f;
                            p.uv[2 * r] = 0.f; p.uv[2 * r + 1] = 0.f;
                        }
                    }
                    active = false;
                } else if constexpr (MODE == kAny) {
                    if (STATS) st_hits += vis.found;
                    if (p.hit) p.hit[r] = vis.found ? 1 : 0;
                    active = false;
                } else if constexpr (MODE == kCount) {
                    if (STATS) st_hits += vis.count > 0;
                    if (p.count) p.count[r] = vis.count;
                    active = false;
                } else if constexpr (MODE == kAllHits) {
                    p.count[r] = vis.count < p.max_hits ? vis.count : p.max_hits;
                    active = false;
                } else if constexpr (MODE == kContains) {
                    // reference: ray_optix.py:238-267 — count along +dir, then along -dir
                    if (phase == 0) {
                        count_plus = vis.count;
                        const float ox = ray.ox, oy = ray.oy, oz = ray.oz;
                        ray_setup(ray, ox, oy, oz, -p.dir[0], -p.dir[1], -p.dir[2]);
                        ray.magic = p.byte_magic;
                        trav_init(tv);
                        vis = Vis(p.tmax);
                        nodes_done = false;
                        phase = 1;
                    } else {
                        const bool inside = ray.ox > p.aabb_lo[0] && ray.oy > p.aabb_lo[1] && ray.oz > p.aabb_lo[2] &&
                                            ray.ox < p.aabb_hi[0] && ray.oy < p.aabb_hi[1] && ray.oz < p.aabb_hi[2];
                        const bool agree = (count_plus & 1) && (vis.count & 1);
                        const bool brk = !agree && (count_plus == 0 || vis.count == 0);
                        p.contain[r] = (inside && agree) ? 1 : 0;
                        p.broken[r] = brk ? 1 : 0;
                        any_inside |= inside;
                        any_broken |= brk;
                        active = false;
                    }
                }
            }
            // re-fill late (most lanes at once): fetch and set up in place
            const unsigned idle = __ballot_sync(0xffffffffu, !active);
            if (idle != 0u && !exhausted) {
                const int n_idle = __popc(idle);
                const int leader = __ffs((int)idle) - 1;
                unsigned long long base = 0;
                if (lane == leader) base = atomicAdd(p.ray_counter, (unsigned long long)n_idle);
                base = __shfl_sync(0xffffffffu, base, leader);
                if ((int64_t)base + n_idle >= nray) exhausted = true;
                if (!active) {
                    r = (int64_t)base + __popc(idle & lt_mask);
                    if (r < nray) {
                        float ox, oy, oz, dx, dy, dz;
                        load_ray<MODE>(p, r, ox, oy, oz, dx, dy, dz);
                        ray_setup(ray, ox, oy, oz, dx, dy, dz);
                        ray.magic = p.byte_magic;
                        trav_init(tv);
                        vis = Vis(p.tmax);
                        if constexpr (MODE == kAllHits) {
                            vis.max_hits = p.max_hits; vis.out = p.staging + (size_t)r * p.max_hits; vis.tris = tris;
                        }
                        phase = 0;
                        nodes_done = false;
                        active = true;
                        if constexpr (MODE == kContains) { if (p.active && !p.active[r]) active = false; }
                    }
                }
            }
            if (!__any_sync(0xffffffffu, active)) {
                if (exhausted) break;
                continue;      // every lane drew a masked-out point (contains with `active`): draw again
            }
        }

        // ---- 2. one wide node per lane including its triangles
        if (active && !nodes_done) nodes_done = trav_step(nodes, tris, ray, vis, stack, tv);
    }
    if (MODE == kContains) {
        if (__any_sync(0xffffffffu, any_inside) && lane == 0) atomicOr(&p.flags[0], 1);
        if (__any_sync(0xffffffffu, any_broken) && lane == 0) atomicOr(&p.flags[1], 1);
    }
    if (STATS) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            st_nodes += __shfl_xor_sync(0xffffffffu, st_nodes, o);
            st_tris += __shfl_xor_sync(0xffffffffu, st_tris, o);
            st_rays += __shfl_xor_sync(0xffffffffu, st_rays, o);
            st_hits += __shfl_xor_sync(0xffffffffu, st_hits, o);
        }
        if (lane == 0) {
            atomicAdd(&p.counters[0], st_nodes);
            atomicAdd(&p.counters[1], st_tris);
            atomicAdd(&p.counters[2], st_rays);
            atomicAdd(&p.counters[3], st_hits);
        }
    }
    release_scratch(p);
}

__device__ __forceinline__ void release_scratch(const TraceParams& p) {
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int* done = reinterpret_cast<unsigned int*>(p.ray_counter + 1);
        __threadfence();
        if (atomicAdd(done, 1u) == gridDim.x - 1u) {
            atomicExch(p.ray_counter, 0ull);
            atomicExch(done, 0u);
        }
    }
}

}  // namespace rt
#include "rt_trace_coop.cuh"
namespace rt {

static int fetch_mode(const int64_t shape[4], const int64_t stride[4], int64_t nray) {
    if (batch_packed(shape, stride)) return kPacked;
    bool constant = true;
    for (int i = 0; i < 3; ++i) if (shape[i] != 1 && stride[i] != 0) constant = false;
    if (constant) return kConstant;                    // stride-0 broadcast of one vector
    return nray < ((int64_t)1 << 31) ? kGeneral32 : kGeneral;
}

// resident CTAs per SM of every kernel variant, per device (filled on first use; benign race: same value)
constexpr int kMaxDevices = 64;
constexpr int64_t kShareMaxRaysCoherentClosest = 1 << 20;   // coherent closest hit: launches up to this many rays share work in the tail
static int g_per_sm[kMaxDevices][5][2][8];

template <int MODE, bool STATS>
static int occupancy(int sched, int* per_sm) {
    switch (sched) {
        case RT_SCHED_DIRECT: return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k_trace<MODE, STATS>, kTraceThreads, 0);
        case RT_SCHED_COOP_COHERENT:
            return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k_trace_coop<MODE, STATS, false, true>, kTraceThreads, 0);
        default: return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k_trace_coop<MODE, STATS, true, true>, kTraceThreads, 0);
    }
}

template <int MODE, bool STATS>
static int launch(const char* fn, TraceParams& p, const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts,
                  void* scratch, cudaStream_t stream) {
    RT_REQUIRE(blob != nullptr && ((uintptr_t)blob & 15) == 0, RT_ERR_INVALID, "%s: blob null or not 16-byte aligned", fn);
    RT_REQUIRE(scratch != nullptr && ((uintptr_t)scratch & 7) == 0, RT_ERR_INVALID, "%s: scratch null or misaligned", fn);
    int64_t first = 0, count = 0;
    const int rc = batch_window(fn, rays, opts, &first, &count);
    if (rc != RT_OK) return rc;
    const bool pinhole = p.o_mode == kPinhole;     // preset by rt_trace_closest_pinhole: rays are generated, not fetched
    if (!pinhole && rays->nray > 0) {               // NULL data of a non-empty batch is an error even for an empty window
        RT_REQUIRE(rays->origins != nullptr, RT_ERR_INVALID, "%s: null origins", fn);
        RT_REQUIRE(MODE == kContains || rays->directions != nullptr, RT_ERR_INVALID, "%s: null directions", fn);
    }
    if (count == 0) return RT_OK;
    static const rt_trace_opts kDefaults = {};
    const rt_trace_opts& o = opts ? *opts : kDefaults;
    DeviceInfo dev;
    RT_REQUIRE(device_info(&dev) == RT_OK && dev.sm_count > 0, RT_ERR_CUDA, "%s: no CUDA device", fn);
    p.blob = reinterpret_cast<const uint8_t*>(blob);
    p.rays = *rays;
    p.ray_first = first;
    p.nray = count;
    if (!pinhole) {
        p.o_mode = fetch_mode(rays->shape, rays->o_stride, rays->nray);
        p.d_mode = MODE != kContains ? fetch_mode(rays->shape, rays->d_stride, rays->nray) : kConstant;
    }
    p.tmax = o.tmax > 0.0f ? o.tmax : RT_TMAX_DEFAULT;     // NaN and <= 0 select the reference's 1e7
    p.stop_on_broken = (MODE == kContains && (o.flags & RT_OPT_STOP_WHEN_BROKEN)) ? 1 : 0;
    p.share_lanes = (o.flags & RT_OPT_NO_LANE_SHARING) ? 0 : 1;
    p.byte_magic = kByteMagic;
    p.ray_counter = reinterpret_cast<unsigned long long*>(scratch);
    if (!(o.flags & RT_OPT_SCRATCH_ZEROED)) RT_CUDA_TRY(cudaMemsetAsync(scratch, 0, RT_TRACE_SCRATCH_BYTES, stream));
    // Scheduling: rays that share one origin (a stride-0 broadcast, i.e. camera / primary rays, reference
    // README.md:38 and test/performance_test.py:36-41) are coherent and mostly short: lanes re-fill late.
    // Anything else is treated as incoherent: rays prepared 32 at a time into a pool, early re-fill.  Both use
    // the warp-cooperative triangle tests of rt_trace_coop.cuh.
    const bool coherent = MODE != kContains && (p.o_mode == kConstant || pinhole);
    p.tile_per_row = 0u;
    if (coherent && !(o.flags & RT_OPT_NO_TILE_ORDER) && first == 0 && count == rays->nray) {
        const int64_t h = rays->shape[1], w = rays->shape[2];
        if (h > 0 && w > 0 && h % kTileH == 0 && w % kTileW == 0 && h * w < ((int64_t)1 << 31) && rays->nray == h * w) {
            p.tile_per_row = (uint32_t)(w / kTileW); p.tile_w = (uint32_t)w;
        }
    }
    int sched = o.schedule;
    RT_REQUIRE(sched >= RT_SCHED_AUTO && sched <= RT_SCHED_SLOTS, RT_ERR_INVALID, "%s: unknown schedule %d", fn, sched);
    if (sched == RT_SCHED_AUTO) sched = coherent ? RT_SCHED_COOP_COHERENT : RT_SCHED_COOP_INCOHERENT;
    if (sched == RT_SCHED_QUEUED || sched == RT_SCHED_SLOTS) sched = RT_SCHED_COOP_INCOHERENT;   // removed schedules (ABI v2 aliases)
    const bool coop = sched != RT_SCHED_DIRECT;
    auto clampi = [](int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); };
    p.refill_threshold = o.refill_threshold > 0 ? clampi(o.refill_threshold, 1, 32)
                                                : (sched == RT_SCHED_COOP_INCOHERENT ? kRefillThresholdCoopIncoherent : kRefillThresholdDirect);
    // the per-lane kernel tests triangles in the node step and does not read tri_threshold
    p.tri_threshold = !coop ? 0
                      : o.tri_threshold > 0 ? clampi(o.tri_threshold, 1, kPairCap - 32)
                                            : (sched == RT_SCHED_COOP_INCOHERENT ? kPairThresholdIncoherent : kPairThresholdCoherent);
    RT_REQUIRE(dev.device >= 0 && dev.device < kMaxDevices, RT_ERR_CUDA, "%s: device index %d not supported", fn, dev.device);
    int& per_sm = g_per_sm[dev.device][sched - 1][STATS ? 1 : 0][MODE];
    if (per_sm == 0) {
        int v = 0;
        const int oc = occupancy<MODE, STATS>(sched, &v);
        RT_REQUIRE(oc == (int)cudaSuccess && v > 0, RT_ERR_CUDA, "%s: kernel does not fit an SM", fn);
        per_sm = v;
    }
    int64_t grid = (int64_t)dev.sm_count * per_sm;
    const int64_t rays_per_cta = (int64_t)kTraceThreads * clampi(o.grid_div > 0 ? o.grid_div : 1, 1, 64);
    const int64_t need = (count + rays_per_cta - 1) / rays_per_cta;
    if (grid > need) grid = need;
    switch (sched) {
        case RT_SCHED_DIRECT: k_trace<MODE, STATS><<<(unsigned)grid, kTraceThreads, 0, stream>>>(p); break;
        default:
            // Work sharing between the lanes of a draining warp (rt_trace_coop.cuh, step 1b) is compiled into every
            // cooperative kernel; coherent closest hit exists a second time without it, for big launches: there the
            // tail is a small part of the launch and the leaner loop is worth 1-3 % (profiles/r2_sweeps.md "p").
            if (sched == RT_SCHED_COOP_COHERENT) {
                if (MODE == kClosest && !STATS && count > kShareMaxRaysCoherentClosest)
                    k_trace_coop<MODE, STATS, false, MODE != kClosest || STATS><<<(unsigned)grid, kTraceThreads, 0, stream>>>(p);
                else
                    k_trace_coop<MODE, STATS, false, true><<<(unsigned)grid, kTraceThreads, 0, stream>>>(p);
            } else {
                k_trace_coop<MODE, STATS, true, true><<<(unsigned)grid, kTraceThreads, 0, stream>>>(p);
            }
    }
    RT_CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

}  // namespace rt

using namespace rt;

extern "C" int rt_trace_any(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, uint8_t* hit, void* scratch,
                            void* stream) {
    RT_REQUIRE(hit || (rays && rays->nray == 0), RT_ERR_INVALID, "rt_trace_any: null output");
    TraceParams p = {};
    p.hit = hit;
    return launch<kAny, false>("rt_trace_any", p, blob, rays, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_trace_first(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int32_t* tri_idx,
                              void* scratch, void* stream) {
    RT_REQUIRE(tri_idx || (rays && rays->nray == 0), RT_ERR_INVALID, "rt_trace_first: null output");
    TraceParams p = {};
    p.tri = tri_idx;
    return launch<kFirst, false>("rt_trace_first", p, blob, rays, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_trace_closest(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, uint8_t* hit,
                                uint8_t* front, int32_t* tri_idx, float* loc, float* uv, void* scratch, void* stream) {
    RT_REQUIRE((hit && front && tri_idx && loc && uv) || (rays && rays->nray == 0), RT_ERR_INVALID,
               "rt_trace_closest: null output");
    TraceParams p = {};
    p.hit = hit; p.front = front; p.tri = tri_idx; p.loc = loc; p.uv = uv;
    return launch<kClosest, false>("rt_trace_closest", p, blob, rays, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_trace_closest_pinhole(const void* blob, const rt_pinhole* cam, const rt_trace_opts* opts, uint8_t* hit,
                                        uint8_t* front, int32_t* tri_idx, float* loc, float* uv, void* scratch,
                                        void* stream) {
    RT_REQUIRE(cam != nullptr && cam->width > 0 && cam->height > 0 && cam->focal > 0.0f, RT_ERR_INVALID,
               "rt_trace_closest_pinhole: bad camera");
    RT_REQUIRE(hit && front && tri_idx && loc && uv, RT_ERR_INVALID, "rt_trace_closest_pinhole: null output");
    TraceParams p = {};
    p.hit = hit; p.front = front; p.tri = tri_idx; p.loc = loc; p.uv = uv;
    p.o_mode = kPinhole; p.d_mode = kPinhole;
    p.cam_w = cam->width;
    p.cam_half_w = (float)(cam->width - 1) / 2.0f; p.cam_half_h = (float)(cam->height - 1) / 2.0f; p.cam_f = cam->focal;
    for (int i = 0; i < 9; ++i) p.cam_mat[i] = cam->cam_mat[i];
    for (int i = 0; i < 3; ++i) p.cam_origin[i] = cam->origin[i];
    rt_ray_desc rd = {};
    rd.nray = cam->width * cam->height;
    rd.shape[0] = 1; rd.shape[1] = cam->height; rd.shape[2] = cam->width; rd.shape[3] = 3;
    return launch<kClosest, false>("rt_trace_closest_pinhole", p, blob, &rd, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_trace_count(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int32_t* count,
                              void* scratch, void* stream) {
    RT_REQUIRE(count || (rays && rays->nray == 0), RT_ERR_INVALID, "rt_trace_count: null output");
    TraceParams p = {};
    p.count = count;
    return launch<kCount, false>("rt_trace_count", p, blob, rays, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_contains_parity(const void* blob, const rt_ray_desc* points, const rt_trace_opts* opts, const float dir[3],
                                  const float aabb_lo[3], const float aabb_hi[3], const uint8_t* active, uint8_t* contain,
                                  uint8_t* broken, int32_t* flags_dev, void* scratch, void* stream) {
    RT_REQUIRE(dir && aabb_lo && aabb_hi && flags_dev, RT_ERR_INVALID, "rt_contains_parity: null argument");
    RT_REQUIRE((contain && broken) || (points && points->nray == 0), RT_ERR_INVALID,
               "rt_contains_parity: null output");
    TraceParams p = {};
    for (int a = 0; a < 3; ++a) { p.dir[a] = dir[a]; p.aabb_lo[a] = aabb_lo[a]; p.aabb_hi[a] = aabb_hi[a]; }
    p.active = active; p.contain = contain; p.broken = broken; p.flags = flags_dev;
    RT_CUDA_TRY(cudaMemsetAsync(flags_dev, 0, 2 * sizeof(int32_t), (cudaStream_t)stream));
    return launch<kContains, false>("rt_contains_parity", p, blob, points, opts, scratch, (cudaStream_t)stream);
}

extern "C" int rt_trace_stats(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int mode,
                              uint64_t* counters_dev, void* scratch, void* stream) {
    RT_REQUIRE(counters_dev != nullptr, RT_ERR_INVALID, "rt_trace_stats: null counters");
    RT_CUDA_TRY(cudaMemsetAsync(counters_dev, 0, 4 * sizeof(uint64_t), (cudaStream_t)stream));
    TraceParams p = {};
    p.counters = reinterpret_cast<unsigned long long*>(counters_dev);
    switch (mode) {
        case 0: return launch<kClosest, true>("rt_trace_stats", p, blob, rays, opts, scratch, (cudaStream_t)stream);
        case 1: return launch<kAny, true>("rt_trace_stats", p, blob, rays, opts, scratch, (cudaStream_t)stream);
        case 2: return launch<kCount, true>("rt_trace_stats", p, blob, rays, opts, scratch, (cudaStream_t)stream);
        default: return set_error(RT_ERR_INVALID, "rt_trace_stats: mode must be 0 (closest), 1 (any) or 2 (count)");
    }
}

// all-hits trace lives here (kernel), its scan + scatter in rt_compact.cu
namespace rt {
int scan_counts_i32(const int32_t* counts, int64_t n, void* workspace, size_t workspace_bytes, int64_t* total_dev,
                    cudaStream_t stream);
size_t scan_workspace_bytes(int64_t n);
}

extern "C" int rt_allhits_sizes(int64_t nray, int max_hits, size_t* staging_bytes, size_t* workspace_bytes) {
    RT_REQUIRE(nray >= 0 && max_hits >= 1 && max_hits <= RT_MAX_HITS_LIMIT && staging_bytes && workspace_bytes,
               RT_ERR_INVALID, "rt_allhits_sizes: bad arguments");
    *staging_bytes = (size_t)nray * (size_t)max_hits * 16u;
    *workspace_bytes = scan_workspace_bytes(nray);
    return RT_OK;
}

extern "C" int rt_allhits_trace(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int max_hits,
                                int32_t* count_clamped, void* staging, void* workspace, size_t workspace_bytes,
                                int64_t* total_dev, void* scratch, void* stream) {
    RT_REQUIRE(max_hits >= 1 && max_hits <= RT_MAX_HITS_LIMIT, RT_ERR_INVALID, "rt_allhits_trace: max_hits out of range");
    RT_REQUIRE(total_dev != nullptr, RT_ERR_INVALID, "rt_allhits_trace: null total");
    RT_REQUIRE((count_clamped && staging && workspace) || (rays && rays->nray == 0), RT_ERR_INVALID,
               "rt_allhits_trace: null buffer");
    TraceParams p = {};
    p.count = count_clamped; p.max_hits = max_hits; p.staging = reinterpret_cast<uint4*>(staging);
    const int rc = launch<kAllHits, false>("rt_allhits_trace", p, blob, rays, opts, scratch, (cudaStream_t)stream);
    if (rc != RT_OK) return rc;
    return scan_counts_i32(count_clamped, p.nray, workspace, workspace_bytes, total_dev, (cudaStream_t)stream);
}
