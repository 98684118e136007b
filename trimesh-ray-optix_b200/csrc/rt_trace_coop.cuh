// rt_trace_coop.cuh — traversal kernel with WARP-COOPERATIVE triangle tests (included by rt_trace.cu).
//
// Same role as k_trace (rt_trace.cu): replaces optixTrace + the closest/first/any/count/all-hits programs of the
// reference (triro/backend/shaders.cu:67-246) and the two count launches of contains_points
// (triro/ray/ray_optix.py:254-260).  What differs from k_trace is WHO tests a triangle:
//
//   * every lane still owns one ray and walks the BVH8 one wide node per step, but a hit leaf slot is
//     not tested by the lane that found it.  The lane appends (lane, triangle record) pairs to a list
//     shared by the warp; when the list is long enough (or lanes wait to retire) ALL 32 lanes test
//     pairs, whichever ray they belong to.  The part of the ray the triangle test needs (shear S,
//     permuted origin, kz) lives in shared memory, column = lane, so any lane can read any ray
//     without bank conflicts;
//   * results merge through shared memory: closest hit is a 64-bit atomicMin on
//     (float bits of t << 32 | primitive index << 1 | front flag) — t > 0, so the bit pattern orders like the
//     value and equal t resolves to the smaller primitive index, exactly the rule of ClosestVisitor — count is a
//     32-bit atomicAdd, any-hit a flag;
//   * the lane whose pair wins computes location / uv right there, at the width of the pair
//     batch, and parks them in shared memory; retiring a ray is then a plain copy (k_trace re-fetches
//     and re-tests the winning triangle with the few lanes that retire together);
//   * pooled (incoherent) kernels test every ray against the box around the root's child slots while they prepare
//     32 rays with all lanes busy; a ray that misses it has its miss written there and never takes a lane
//     (fill_pool_frame below, rt_core.cuh frame_missed);
//   * contains_points walks the second direction only as far as the first count leaves the answer open (retirement);
//   * once a warp can draw no more rays (the tail of a launch; all of a small launch), lanes without a ray take
//     over part of a busy neighbour's traversal stack (step 1b, template parameter SHARE): possible because
//     everything a triangle test or a hit touches is addressed by the ray's shared-memory column, not by the lane.
//
// ncu of k_trace on config 2 (profiles/r1_ncu_regions_config2_v4.txt): the in-step triangle test was
// 27.8 % of all warp instructions at 8.17 of 32 active lanes.  Results are bit-identical to k_trace
// (tests/test_gpu_round2.py::test_all_schedules_give_identical_results).
#pragma once

namespace rt {

#ifndef RT_PAIR_CAP
#define RT_PAIR_CAP 128
#endif
constexpr int kPairCap = RT_PAIR_CAP;  // pairs a warp can list before it must test them
#ifndef RT_TAIL_LANES
#define RT_TAIL_LANES 4
#endif
constexpr int kTailLanes = RT_TAIL_LANES;          // <= this many lanes with node work: test listed pairs every step
// Pool fill with the root-frame test (see the call site).  The ORDER inside matters for the whole kernel: with the full
// ray set-up before the frame test (or with the whole root node tested here) the register peak of this code made ptxas
// keep traversal state in local memory around every node step (soup -9...-16 %); a __noinline__ call still left one such
// spill.  Testing on (origin, 1/d) first and setting up only the survivors needs no spill at all.
template <int MODE>
__device__ __forceinline__ unsigned fill_pool_frame(const TraceParams& p, int64_t base, int n, float (*s_pool)[kTraceThreads],
                                                   const RootFrame& s_root, int col0, int lane) {
    // the frame test needs the origin and 1/d only: it runs before the (register-hungry) rest of the set-up
    bool live = false;
    float ox = 0.f, oy = 0.f, oz = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
    if (lane < n) {
        load_ray<MODE>(p, base + lane, ox, oy, oz, dx, dy, dz);
        float idx, idy, idz;
        ray_inverse(dx, dy, dz, idx, idy, idz);
        live = !frame_missed(ox, oy, oz, idx, idy, idz, s_root, p.tmax);
        if (!live) {
            const int64_t q = base + lane;
            if constexpr (MODE == kClosest) {
                if (p.hit) {      // miss: reference miss program shaders.cu:128-135
                    p.hit[q] = 0; p.front[q] = 0; p.tri[q] = -1;
                    p.loc[3 * q] = 0.f; p.loc[3 * q + 1] = 0.f; p.loc[3 * q + 2] = 0.f;
                    p.uv[2 * q] = 0.f; p.uv[2 * q + 1] = 0.f;
                }
            } else if constexpr (MODE == kFirst) {
                if (p.tri) p.tri[q] = -1;
            } else if constexpr (MODE == kAny) {
                if (p.hit) p.hit[q] = 0;
            } else {
                if (p.count) p.count[q] = 0;     // count, all hits
            }
        }
    }
    const unsigned alive = __ballot_sync(0xffffffffu, live);
    if (live) {
        Ray t;
        ray_setup(t, ox, oy, oz, dx, dy, dz);
        const int col = col0 + __popc(alive & ((1u << lane) - 1u));
        s_pool[0][col] = t.ox; s_pool[1][col] = t.oy; s_pool[2][col] = t.oz;
        s_pool[3][col] = t.Sx; s_pool[4][col] = t.Sy; s_pool[5][col] = t.Sz;
        s_pool[6][col] = t.okx; s_pool[7][col] = t.oky; s_pool[8][col] = t.okz;
        s_pool[9][col] = t.idx; s_pool[10][col] = t.idy; s_pool[11][col] = t.idz;
        s_pool[12][col] = __int_as_float(t.kzf | (int)(t.octinv << 8) | (lane << 20));
    }
    return alive;
}

constexpr uint32_t kContainsAnyBit = 0x80000000u;   // contains: s_cnt bit 31 = "this walk only has to find one hit"
constexpr int kRayWords = 7;           // resident part of a ray in shared memory: S(3), permuted origin(3), kzf

// POOL = incoherent batches: rays are prepared 32 at a time into a shared-memory pool and lanes re-fill early;
// otherwise lanes re-fill late and set their ray up in place (coherent batches).
template <int MODE, bool STATS, bool POOL, bool SHARE>
__global__ void __launch_bounds__(kTraceThreads, (MODE == kClosest && POOL) ? RT_TRACE_MIN_BLOCKS : RT_TRACE_MIN_BLOCKS_LIGHT)
k_trace_coop(const __grid_constant__ TraceParams p) {
    constexpr bool kKey = MODE == kClosest || MODE == kFirst;
    __shared__ float s_ray[kRayWords][kTraceThreads];
    // Shared memory is L1 taken away (one 256 KB array per SM, carve-out steps 100 / 132 / 164 KB): the arrays below are
    // sized so that 7 resident CTAs of the pooled closest-hit kernel stay under 132 KB and 8 CTAs of the others under
    // 100 / 132 KB (1 KB per CTA is reserved by the system).
    __shared__ unsigned long long s_best[kKey ? kTraceThreads : 1];      // (t bits << 32) | prim  (closest: prim << 1 | front)
    __shared__ uint32_t s_cnt[kKey ? 1 : kTraceThreads];                 // count / any flag
    __shared__ float s_attr[MODE == kClosest ? 5 : 1][kTraceThreads];    // loc(3), uv(2)
    // ray index of the column's ray (all hits: where the owner's records go).  The pooled 64-register kernels keep the
    // lane's ray index here instead of in two registers: their loop sits at the register edge, and a value spilled around
    // every node step costs the L1TEX-bound soup 10 %; it is touched when a ray starts and retires only.  (The pooled
    // closest-hit kernel has 72 registers and keeps it there: measured equal or better.)
    constexpr bool kRInSmem = POOL && MODE != kClosest;
    __shared__ long long s_rayidx[(MODE == kAllHits || kRInSmem) ? kTraceThreads : 1];
    __shared__ uint2 s_pair[kTraceThreads / 32][kPairCap];               // (triangle record, owner lane)
    constexpr bool kRootFirst = POOL && MODE != kContains;     // contains fills its pool without the frame test
    __shared__ float s_pool[POOL ? kPoolWords : 1][POOL ? kTraceThreads : 1];
    __shared__ RootFrame s_root;
    __shared__ long long s_pool_base[POOL ? kTraceThreads / 32 : 1];     // ray index of the pool's first ray, per warp (not a register: the loop is at the 64-register edge)
    if (kRootFirst && threadIdx.x == 0) {
        const uint8_t* np = p.blob + reinterpret_cast<const rt_blob_header*>(p.blob)->nodes_offset;
        s_root = root_frame(ldg128(np), ldg128(np + 32), ldg128(np + 48), ldg128(np + 64));
    }
    init_mask_luts();     // ends with __syncthreads()
    const rt_blob_header* hdr = reinterpret_cast<const rt_blob_header*>(p.blob);
    const uint8_t* tris = p.blob + hdr->tris_offset;
    const uint8_t* nodes = p.blob + hdr->nodes_offset;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col0 = (int)(threadIdx.x & ~31u), mycol = (int)threadIdx.x;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t nray = p.nray;
    const unsigned long long key_init = (unsigned long long)__float_as_uint(p.tmax) << 32;
    PairStack stack;
    unsigned long long st_nodes = 0, st_tris = 0, st_rays = 0, st_hits = 0;
    bool any_inside = false, any_broken = false;

    Trav tv;
    Ray ray;                          // only o, 1/d, octinv, magic stay live across iterations
    float tmax = p.tmax;
    int64_t r_reg = -1;
    auto ray_index = [&]() -> int64_t { if constexpr (kRInSmem) return (int64_t)s_rayidx[mycol]; else return r_reg; };
    auto set_ray_index = [&](int64_t v) { if constexpr (kRInSmem) s_rayidx[mycol] = (long long)v; else r_reg = v; };
    set_ray_index(0);                 // a lane without a ray must not read as a helper (negative index, see owner_col)
    bool active = false, exhausted = false, nodes_done = true;
    int phase = 0;
    uint32_t count_plus = 0;
    int n_pend = 0;                   // pairs in the warp's list (warp-uniform)
    int my_pend = 0;                  // != 0: some of them belong to this lane's ray
    int pool_head = 0, pool_count = 0;
    uint32_t ty = 0u, tx = 0u, tmask = 0u;      // triangles of this lane's last node step not yet listed
    // column of the ray this lane walks for: its own, or (work sharing, SHARE) a neighbour's - a helper keeps
    // ~column in r, which it does not need (no extra register in the loop)
    auto owner_col = [&]() -> int { const int64_t r = ray_index(); return r < 0 ? (int)(~r) : mycol; };
    trav_init(tv);

    // ---- test every listed pair with the whole warp
    auto flush = [&](auto drain_tag) {
        constexpr bool DRAIN = decltype(drain_tag)::value;
        __syncwarp();
        for (int base = 0; base < n_pend; base += 32) {
            const int i = base + lane;
            bool won = false;
            unsigned long long key = 0;
            int col = 0;
            TriHit h;
            Ray t;
            float v0x = 0, v0y = 0, v0z = 0, v1x = 0, v1y = 0, v1z = 0, v2x = 0, v2y = 0, v2z = 0;
            if (i < n_pend) {
                const uint2 pr = s_pair[warp][i];
                const uint32_t slot = pr.x;
                col = col0 + (int)pr.y;
                t.Sx = s_ray[0][col]; t.Sy = s_ray[1][col]; t.Sz = s_ray[2][col];
                t.okx = s_ray[3][col]; t.oky = s_ray[4][col]; t.okz = s_ray[5][col];
                t.kzf = __float_as_int(s_ray[6][col]);
                const uint8_t* tp = tris + (size_t)slot * 48u;
                const U4 a = ldg128(tp), b = ldg128(tp + 16), c = ldg128(tp + 32);
                v0x = as_float(a.x); v0y = as_float(a.y); v0z = as_float(a.z);
                v1x = as_float(b.x); v1y = as_float(b.y); v1z = as_float(b.z);
                v2x = as_float(c.x); v2y = as_float(c.y); v2z = as_float(c.z);
                if (STATS) ++st_tris;
                if (tri_test(t, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z, h) && h.t > 0.0f) {
                    if constexpr (kKey) {
                        // equal t resolves to the smaller primitive index; closest hit carries the front flag in bit 0
                        // (one word of shared memory per ray less), primitive indices are < 2^31 (int32 outputs)
                        uint32_t low = (uint32_t)a.w;
                        if constexpr (MODE == kClosest) low = (low << 1) | (tri_front(t, h) ? 1u : 0u);
                        key = ((unsigned long long)__float_as_uint(h.t) << 32) | (unsigned long long)low;
                        if (key < s_best[col]) { atomicMin(&s_best[col], key); won = true; }
                    } else if constexpr (MODE == kAny) {
                        if (h.t < p.tmax) s_cnt[col] = 1u;
                    } else if constexpr (MODE == kAllHits) {
                        // reference __anyhit__intersectsLocation (shaders.cu:207-224): the first max_hits hits found are
                        // recorded (which ones, beyond max_hits, is traversal order there and test order here), all counted
                        if (h.t < p.tmax) {
                            const uint32_t k = atomicAdd(&s_cnt[col], 1u);
                            if (k < (uint32_t)p.max_hits) {
                                const HitAttr at = tri_attr(h, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z);
                                p.staging[(size_t)s_rayidx[col] * (size_t)p.max_hits + k] =
                                    make_uint4(a.w, __float_as_uint(at.lx), __float_as_uint(at.ly), __float_as_uint(at.lz));
                            }
                        }
                    } else {
                        if (h.t < p.tmax) atomicAdd(&s_cnt[col], 1u);
                    }
                }
            }
            if constexpr (MODE == kClosest) {
                __syncwarp();
                if (won && s_best[col] == key) {     // this pair is the ray's nearest so far: its lane computes the attributes
                    const HitAttr at = tri_attr(h, v0x, v0y, v0z, v1x, v1y, v1z, v2x, v2y, v2z);
                    s_attr[0][col] = at.lx; s_attr[1][col] = at.ly; s_attr[2][col] = at.lz;
                    s_attr[3][col] = at.uv0; s_attr[4][col] = at.uv1;
                }
            }
        }
        __syncwarp();
        n_pend = 0; my_pend = 0;
        const int oc = (DRAIN && active) ? owner_col() : mycol;
        if constexpr (kKey) tmax = __uint_as_float((uint32_t)(s_best[oc] >> 32));
        if constexpr (MODE == kAny) { if (active && s_cnt[oc]) { nodes_done = true; ty = 0u; } }   // early exit
        if constexpr (MODE == kContains) { if (active && s_cnt[oc] > kContainsAnyBit) { nodes_done = true; ty = 0u; } }   // any-hit second walk: found
    };

    // ---- start ray r on this lane from a prepared set-up
    auto start_ray = [&](const Ray& t) {
        s_ray[0][mycol] = t.Sx; s_ray[1][mycol] = t.Sy; s_ray[2][mycol] = t.Sz;
        s_ray[3][mycol] = t.okx; s_ray[4][mycol] = t.oky; s_ray[5][mycol] = t.okz;
        s_ray[6][mycol] = __int_as_float(t.kzf);
        if constexpr (kKey) s_best[mycol] = key_init; else s_cnt[mycol] = 0u;
        if constexpr (MODE == kAllHits && !kRInSmem) s_rayidx[mycol] = (long long)r_reg;
        tmax = p.tmax;
        trav_init(tv);
        nodes_done = false;
        active = true;
    };

    // One iteration of the traversal loop; returns 1 when the warp is finished, 2 to switch to the DRAIN instance.  Instantiated twice: DRAIN = false is
    // the loop proper; DRAIN = true runs once this warp can draw no more rays and adds work sharing between its lanes
    // (a separate instance, so that the hot loop's code is exactly what it is without sharing: folding the two cost 3-4 %
    // on config 2, profiles/r2_sweeps.md "p").
    auto step = [&](auto drain_tag) -> int {
        constexpr bool DRAIN = decltype(drain_tag)::value;
        // ---- 1. flush policy (the ONE place pairs are tested), retirement, re-fill
        const unsigned done_mask = __ballot_sync(0xffffffffu, !active || nodes_done);
        const int busy = 32 - __popc(done_mask);
        const bool want_refill = done_mask != 0u && busy < ((exhausted && pool_count == 0) ? 1 : p.refill_threshold);
        if (n_pend > 0) {
            // few lanes left with node work (the tail of a launch, or a lone long ray): test at once, so that tmax shrinks
            // before the next node step instead of after tri_threshold pairs have trickled in
            bool go = n_pend >= p.tri_threshold || busy <= kTailLanes;
            if (!go && n_pend == kPairCap) go = true;                                                      // list full (triangles may be waiting in ty)
            if (!go && want_refill) go = __any_sync(0xffffffffu, active && nodes_done && my_pend != 0);   // rays wait to retire
            if (go) flush(drain_tag);
        }
        if (want_refill) {
            if constexpr (MODE == kContains) {
                // RT_OPT_STOP_WHEN_BROKEN (the retry of ray_optix.py:272-277): once any point is broken again the caller
                // discards the whole launch, so stop drawing points
                if (p.stop_on_broken && !(exhausted && pool_count == 0)) {
                    int f = 0;
                    if (lane == 0) f = *reinterpret_cast<volatile int32_t*>(&p.flags[1]);
                    if (__shfl_sync(0xffffffffu, f, 0)) { exhausted = true; pool_count = 0; }
                }
            }
            bool retire = active && nodes_done && my_pend == 0 && ty == 0u;
            if constexpr (DRAIN) {
                // work sharing (below): a helper that has listed everything simply becomes idle; a ray retires once no
                // helper still walks or holds unlisted triangles for it (the list itself is empty here: the flush above
                // ran, because no lane has node work left)
                bool helper = active && ray_index() < 0;
                if (retire && helper) { active = false; set_ray_index(0); retire = false; helper = false; }
                const unsigned helped = __reduce_or_sync(0xffffffffu, helper ? 1u << ((int)(~ray_index()) & 31) : 0u);
                if ((helped >> lane) & 1u) retire = false;
            }
            if (retire) {
                const int64_t r = ray_index();
                if constexpr (MODE == kClosest || MODE == kFirst) {
                    const unsigned long long best = s_best[mycol];
                    const bool hit = best != key_init;
                    if (STATS) { ++st_rays; st_hits += hit; }
                    if (MODE == kFirst) {
                        if (p.tri) p.tri[r] = hit ? (int32_t)(uint32_t)best : -1;
                    } else if (p.hit) {
                        // miss: reference miss program shaders.cu:128-135
                        p.hit[r] = hit ? 1 : 0;
                        p.front[r] = hit ? (uint8_t)((uint32_t)best & 1u) : 0;
                        p.tri[r] = hit ? (int32_t)((uint32_t)best >> 1) : -1;
                        p.loc[3 * r] = hit ? s_attr[0][mycol] : 0.f; p.loc[3 * r + 1] = hit ? s_attr[1][mycol] : 0.f;
                        p.loc[3 * r + 2] = hit ? s_attr[2][mycol] : 0.f;
                        p.uv[2 * r] = hit ? s_attr[3][mycol] : 0.f; p.uv[2 * r + 1] = hit ? s_attr[4][mycol] : 0.f;
                    }
                    active = false;
                } else if constexpr (MODE == kAny) {
                    const bool found = s_cnt[mycol] != 0u;
                    if (STATS) { ++st_rays; st_hits += found; }
                    if (p.hit) p.hit[r] = found ? 1 : 0;
                    active = false;
                } else if constexpr (MODE == kCount) {
                    const uint32_t c = s_cnt[mycol];
                    if (STATS) { ++st_rays; st_hits += c > 0u; }
                    if (p.count) p.count[r] = (int32_t)c;
                    active = false;
                } else if constexpr (MODE == kAllHits) {
                    const uint32_t c = s_cnt[mycol];
                    p.count[r] = (int32_t)(c < (uint32_t)p.max_hits ? c : (uint32_t)p.max_hits);     // ray.cpp:334-335
                    active = false;
                } else if constexpr (MODE == kContains) {
                    // reference: ray_optix.py:238-267 — count along +dir, then along -dir; contain = inside the AABB and
                    // both counts odd, broken = they disagree on "odd" and one of them is 0 (symmetric in the two counts:
                    // which walk comes first is free, see the pool fill).  What the second walk has to find out depends
                    // on the first count c+ (same outputs, less work):
                    //   c+ == 0      nothing: contain = 0, broken = 1 whatever c- is
                    //   c+ even > 0  only whether c- == 0: an any-hit walk (kContainsAnyBit in s_cnt ends it at the first hit)
                    //   c+ odd       the parity of c-: the full count
                    const uint32_t c = s_cnt[mycol] & ~kContainsAnyBit;
                    if (!(phase & 1) && c != 0u) {
                        count_plus = c;
                        Ray t;
                        const float sg = (phase & 4) ? 1.0f : -1.0f;     // the second walk goes the other way
                        ray_setup(t, ray.ox, ray.oy, ray.oz, sg * p.dir[0], sg * p.dir[1], sg * p.dir[2]);
                        ray.idx = t.idx; ray.idy = t.idy; ray.idz = t.idz; ray.octinv = t.octinv;
                        start_ray(t);
                        if (!(c & 1u)) s_cnt[mycol] = kContainsAnyBit;
                        phase |= 1;
                    } else {
                        if (!(phase & 1)) count_plus = 0u;         // first count 0: c (= 0) stands in for the second
                        const bool inside = ray.ox > p.aabb_lo[0] && ray.oy > p.aabb_lo[1] && ray.oz > p.aabb_lo[2] &&
                                            ray.ox < p.aabb_hi[0] && ray.oy < p.aabb_hi[1] && ray.oz < p.aabb_hi[2];
                        const bool agree = (count_plus & 1u) && (c & 1u);
                        const bool brk = !agree && (count_plus == 0u || c == 0u);
                        p.contain[r] = (inside && agree) ? 1 : 0;
                        p.broken[r] = brk ? 1 : 0;
                        any_inside |= inside;
                        if (brk && !any_broken && p.stop_on_broken) atomicOr(&p.flags[1], 1);     // tell the other warps now
                        any_broken |= brk;
                        active = false;
                    }
                }
            }
            if constexpr (POOL) {
                for (;;) {
                    const unsigned idle = __ballot_sync(0xffffffffu, !active);
                    if (idle == 0u) break;
                    if (pool_count == 0) {
                        if (exhausted) break;
                        unsigned long long base = 0;
                        if (lane == 0) base = atomicAdd(p.ray_counter, 32ull);
                        base = __shfl_sync(0xffffffffu, base, 0);
                        int64_t n = nray - (int64_t)base;
                        if (n <= 32) exhausted = true;
                        if (n <= 0) break;
                        if (n > 32) n = 32;
                        if constexpr (kRootFirst) {
                            // Rays are tested here, with all 32 lanes busy, against the box that bounds the root's children
                            // in the root's own quantised frame (frame_missed: the arithmetic of node_test, so a ray it
                            // rejects is rejected by every child slot of the root as well).  Such a ray gets its miss
                            // written on the spot (32 consecutive rays: coalesced) and never takes a lane; the others
                            // enter the pool, compacted.  Heightfields with 74 % missing rays: +8...12 %.  Testing the
                            // whole root node here was tried: its registers made ptxas keep the lanes' ray registers in
                            // local memory across the loop (soup -14 %).
                            const unsigned alive = fill_pool_frame<MODE>(p, (int64_t)base, (int)n, s_pool, s_root, col0, lane);
                            if (STATS && lane == 0) { st_rays += (unsigned)n - __popc(alive); st_nodes += (unsigned)n - __popc(alive); }
                            if (lane == 0) s_pool_base[warp] = (long long)base;
                            __syncwarp();
                            pool_head = 0; pool_count = __popc(alive);
                            continue;
                        }
                        if (lane < n) {
                            float ox, oy, oz, dx, dy, dz;
                            load_ray<MODE>(p, (int64_t)base + lane, ox, oy, oz, dx, dy, dz);
                            int skip = 0, flip = 0;
                            if constexpr (MODE == kContains) {
                                if (p.active && !p.active[(int64_t)base + lane]) skip = 1;
                                // contain / broken are symmetric in the two counts, so a point inside the AABB walks FIRST
                                // towards the side where it leaves the AABB sooner: the short walk is cheap and most
                                // likely to count 0, which settles the point without the long walk (see the retirement)
                                float tp = 3.0e38f, tm = 3.0e38f;
                                const float o3[3] = {ox, oy, oz};
                                bool in = true;
#pragma unroll
                                for (int a = 0; a < 3; ++a) {
                                    const float d = p.dir[a], lo = p.aabb_lo[a] - o3[a], hi = p.aabb_hi[a] - o3[a];
                                    in = in && lo < 0.0f && hi > 0.0f;
                                    if (d != 0.0f) {
                                        const float inv = __frcp_rn(d);
                                        tp = fminf(tp, (d > 0.0f ? hi : lo) * inv);
                                        tm = fminf(tm, (d > 0.0f ? lo : hi) * -inv);
                                    }
                                }
                                if (in && tm < tp) { flip = 1; dx = -dx; dy = -dy; dz = -dz; }
                            }
                            Ray t;
                            ray_setup(t, ox, oy, oz, dx, dy, dz);
                            const int col = col0 + lane;
                            s_pool[0][col] = t.ox; s_pool[1][col] = t.oy; s_pool[2][col] = t.oz;
                            s_pool[3][col] = t.Sx; s_pool[4][col] = t.Sy; s_pool[5][col] = t.Sz;
                            s_pool[6][col] = t.okx; s_pool[7][col] = t.oky; s_pool[8][col] = t.okz;
                            s_pool[9][col] = t.idx; s_pool[10][col] = t.idy; s_pool[11][col] = t.idz;
                            s_pool[12][col] = __int_as_float(t.kzf | (int)(t.octinv << 8) | (skip << 16) | (flip << 17));
                        }
                        if (lane == 0) s_pool_base[warp] = (long long)base;
                        __syncwarp();
                        pool_head = 0; pool_count = (int)n;
                    }
                    const int n_idle = __popc(idle);
                    const int take = n_idle < pool_count ? n_idle : pool_count;
                    const int my = __popc(idle & lt_mask);
                    if (!active && my < take) {
                        const int col = col0 + pool_head + my;
                        const int packed = __float_as_int(s_pool[12][col]);
                        if (kRootFirst || !((packed >> 16) & 1)) {
                            set_ray_index((int64_t)s_pool_base[warp] + (kRootFirst ? ((packed >> 20) & 31) : pool_head + my));
                            Ray t;
                            ray.ox = s_pool[0][col]; ray.oy = s_pool[1][col]; ray.oz = s_pool[2][col];
                            t.Sx = s_pool[3][col]; t.Sy = s_pool[4][col]; t.Sz = s_pool[5][col];
                            t.okx = s_pool[6][col]; t.oky = s_pool[7][col]; t.okz = s_pool[8][col];
                            ray.idx = s_pool[9][col]; ray.idy = s_pool[10][col]; ray.idz = s_pool[11][col];
                            t.kzf = packed & 0xff; ray.octinv = ((uint32_t)packed >> 8) & 0xffu;
                            ray.magic = p.byte_magic;
                            phase = (MODE == kContains && ((packed >> 17) & 1)) ? 4 : 0;     // bit 2: the first walk goes along -dir
                            start_ray(t);
                        }
                    }
                    __syncwarp();
                    pool_head += take; pool_count -= take;
                }
            } else {
                const unsigned idle = __ballot_sync(0xffffffffu, !active);
                if (idle != 0u && !exhausted) {
                    const int n_idle = __popc(idle);
                    const int leader = __ffs((int)idle) - 1;
                    unsigned long long base = 0;
                    if (lane == leader) base = atomicAdd(p.ray_counter, (unsigned long long)n_idle);
                    base = __shfl_sync(0xffffffffu, base, leader);
                    if ((int64_t)base + n_idle >= nray) exhausted = true;
                    if (!active) {
                        int64_t r = (int64_t)base + __popc(idle & lt_mask);
                        bool take = r < nray;
                        if (take) r = tile_order(p, r);
                        if constexpr (MODE == kContains) { if (take && p.active && !p.active[r]) take = false; }
                        set_ray_index(r);
                        if (take) {
                            float ox, oy, oz, dx, dy, dz;
                            load_ray<MODE>(p, r, ox, oy, oz, dx, dy, dz);
                            Ray t;
                            ray_setup(t, ox, oy, oz, dx, dy, dz);
                            ray.ox = t.ox; ray.oy = t.oy; ray.oz = t.oz;
                            ray.idx = t.idx; ray.idy = t.idy; ray.idz = t.idz; ray.octinv = t.octinv;
                            ray.magic = p.byte_magic;
                            phase = 0;
                            start_ray(t);
                        }
                    }
                }
            }
            if (!__any_sync(0xffffffffu, active)) return (exhausted && pool_count == 0) ? 1 : 0;   // 0: every lane drew a masked-out point, draw again
            if constexpr (!DRAIN && SHARE) { if (exhausted && pool_count == 0 && p.share_lanes) return 2; }
        }

        // ---- 1b. work sharing once this warp can draw no more rays: a lane without a ray takes the top stack entry (the
        //          nearest untested sibling group) of a lane that still walks, together with that ray's node-test registers,
        //          and walks it as a HELPER.  Everything a triangle test or a hit needs is indexed by the ray's shared-memory
        //          column (s_ray / s_best / s_cnt / s_attr / s_rayidx), pairs carry the owner's column, and the closest hit is
        //          an order-independent atomicMin, so results do not depend on who walked which subtree; only the owner
        //          retires the ray.  Cuts the tail of a launch: a silhouette ray's 60 node steps spread over the warp.
        if constexpr (DRAIN) {
            if (active && nodes_done && ty == 0u && ray_index() < 0) { active = false; set_ray_index(0); }      // helper finished
            const unsigned idle = __ballot_sync(0xffffffffu, !active);
            const unsigned rich = __ballot_sync(0xffffffffu, active && !nodes_done && tv.sp > 0);
            if (idle != 0u && rich != 0u) {
                const int n_idle = __popc(idle), n_rich = __popc(rich);
                const int take = n_idle < n_rich ? n_idle : n_rich;
                uint32_t sgx = 0u, sgy = 0u;
                if (((rich >> lane) & 1u) && __popc(rich & lt_mask) < take) { --tv.sp; stack.pop(tv.sp, sgx, sgy); }
                const int my = __popc(idle & lt_mask);
                const bool get = !active && my < take;
                const int src = get ? (int)__fns(rich, 0u, my + 1) : lane;
                sgx = __shfl_sync(0xffffffffu, sgx, src); sgy = __shfl_sync(0xffffffffu, sgy, src);
                const float hox = __shfl_sync(0xffffffffu, ray.ox, src), hoy = __shfl_sync(0xffffffffu, ray.oy, src),
                            hoz = __shfl_sync(0xffffffffu, ray.oz, src);
                const float hix = __shfl_sync(0xffffffffu, ray.idx, src), hiy = __shfl_sync(0xffffffffu, ray.idy, src),
                            hiz = __shfl_sync(0xffffffffu, ray.idz, src);
                const uint32_t hoct = __shfl_sync(0xffffffffu, ray.octinv, src);
                const int hcol = __shfl_sync(0xffffffffu, owner_col(), src);
                if (get) {
                    ray.ox = hox; ray.oy = hoy; ray.oz = hoz; ray.idx = hix; ray.idy = hiy; ray.idz = hiz;
                    ray.octinv = hoct; ray.magic = p.byte_magic;
                    set_ray_index(~(int64_t)hcol);
                    tmax = p.tmax;
                    if constexpr (kKey) tmax = __uint_as_float((uint32_t)(s_best[hcol] >> 32));
                    trav_init(tv);
                    tv.gx = sgx; tv.gy = sgy;
                    ty = 0u;
                    nodes_done = false; active = true;
                }
            }
        }

        // ---- 2. node phase: one wide node per lane; hit leaf slots yield a 24-bit triangle mask
        if (active && !nodes_done && ty == 0u) {
            if (tv.gy & 0xff000000u) {
                const uint32_t hits = tv.gy;
                const int bit = 31 - clz32(hits);
                tv.gy &= ~(1u << bit);
                if (tv.gy & 0xff000000u) { stack.push(tv.sp, tv.gx, tv.gy); ++tv.sp; }
                const uint32_t slot = (uint32_t)(bit - 24) ^ ray.octinv;
                const uint32_t rel = (uint32_t)popc32(hits & ~(0xffffffffu << slot));
                const uint8_t* np = nodes + (size_t)(tv.gx + rel) * 80u;
                const U4 n0 = ldg128(np), n1 = ldg128(np + 16), n2 = ldg128(np + 32), n3 = ldg128(np + 48),
                         n4 = ldg128(np + 64);
                if (STATS) ++st_nodes;
                const uint32_t hm = node_test(ray, n0, n1, n2, n3, n4, 0.0f, tmax);
                tv.gx = n1.x;
                tv.gy = (hm & 0xff000000u) | (n0.w >> 24);
                ty = hm & 0x00ffffffu; tx = n1.y; tmask = n1.z;
            }
            if (!(tv.gy & 0xff000000u)) {
                if (tv.sp == 0) nodes_done = true;
                else { --tv.sp; stack.pop(tv.sp, tv.gx, tv.gy); }
            }
        }

        // ---- 3. append this step's (triangle, lane) pairs to the warp's list: one warp scan of the per-lane counts gives
        //         every lane its first position; what does not fit stays in ty and is listed after the next flush (such a
        //         lane takes no node step meanwhile)
        if (__any_sync(0xffffffffu, ty != 0u)) {
            const int c = __popc(ty);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            int pos = n_pend + incl - c;
            if (ty != 0u && pos < kPairCap) my_pend = 1;
            while (ty != 0u && pos < kPairCap) {
                const int b = ffs32(ty) - 1;
                ty &= ty - 1u;
                s_pair[warp][pos] = make_uint2(tx + (uint32_t)popc32(tmask & ~(0xffffffffu << b)), (uint32_t)(DRAIN ? owner_col() & 31 : lane));
                ++pos;
            }
            n_pend = n_pend + total < kPairCap ? n_pend + total : kPairCap;
        }
        return 0;
    };
    int rc;
    do { rc = step(std::false_type{}); } while (rc == 0);
    if constexpr (SHARE) {
        if (rc == 2) {
            while (step(std::true_type{}) == 0) {}
        }
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

}  // namespace rt
