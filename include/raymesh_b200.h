/*
 * raymesh_b200.h — C ABI of the B200-native ray/mesh intersector (libtriro_b200.so).
 *
 * This is the drop-in boundary for the hot path of lcp29/trimesh-ray-optix ("Triro").
 * Every entry point replaces one piece of the reference's native interface
 * (pybind11 module `triro`, triro/backend/binding.cpp:31-59).  Citations below are
 * relative to the reference tree.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types in any signature;
 *   - every function returns 0 on success, a negative rt_status on failure; the
 *     message is available through rt_last_error() (thread-local).  Nothing here
 *     throws or calls exit() (the reference exits the interpreter on OptiX errors,
 *     triro/backend/optix8.h:41-49);
 *   - all pointers except where noted are DEVICE pointers on the current CUDA device;
 *     memory is owned by the caller (the Python host allocates it with torch);
 *   - `stream` is a cudaStream_t passed as void* (the caller's current stream);
 *     all work is asynchronous on that stream, there is no hidden synchronisation;
 *   - no CPU fallback exists: without a CUDA device every compute entry point fails.
 */
#ifndef RAYMESH_B200_H
#define RAYMESH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 2

/* reference: LaunchParams.h:8-9 */
#define RT_MAX_ANYHIT_SIZE 8
/* the all-hits entry points accept max_hits up to this limit (the reference's cap of 8 is the default) */
#define RT_MAX_HITS_LIMIT 64
#define RT_MAX_SIZE_LENGTH 4
/* reference: tmin = 0, tmax = 1e7 on every optixTrace, shaders.cu:86,112,163,191,238 */
#define RT_TMAX_DEFAULT 1.0e7f

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, misalignment) */
    RT_ERR_CUDA = -2,      /* a CUDA runtime call failed */
    RT_ERR_SIZE = -3,      /* caller buffer too small */
    RT_ERR_BLOB = -4,      /* not a BVH blob of this ABI version */
    RT_ERR_DEPTH = -5      /* BVH deeper than the traversal stack (degenerate mesh) */
} rt_status;

/*
 * Strided ray batch.  Mirrors `RayInput` (LaunchParams.h:11-28) as filled by
 * `fillArray` (ray.cpp:151-159): the tensor shape [*b, 3] is right-aligned into
 * 4 slots; strides are in ELEMENTS (floats), any value including 0 (broadcast) and
 * negative.  Missing leading dimensions have shape 1 / stride 0.  As in the
 * reference (ray.cpp:177-179) the shape of `origins` is used for both tensors.
 * Ray r (row-major over shape[0..2]) reads component k of its origin at
 *   origins[i0*o_stride[0] + i1*o_stride[1] + i2*o_stride[2] + k*o_stride[3]].
 * (shaders.cu:27-63; the reference's 32-bit `idx*3` overflow is not reproduced:
 * indices are 64-bit.)
 */
typedef struct rt_ray_desc {
    int64_t nray;
    int64_t shape[RT_MAX_SIZE_LENGTH];
    const float* origins;
    int64_t o_stride[RT_MAX_SIZE_LENGTH];
    const float* directions;
    int64_t d_stride[RT_MAX_SIZE_LENGTH];
} rt_ray_desc;

/* Host-readable copy of the blob header (first RT_BLOB_HEADER_BYTES of a blob). */
#define RT_BLOB_HEADER_BYTES 256
#define RT_BLOB_MAGIC 0x38485642u /* "BVH8" */
typedef struct rt_blob_header {
    uint32_t magic;
    uint32_t abi_version;
    uint32_t n_tris;
    uint32_t n_nodes;       /* 80-byte BVH8 nodes in use */
    uint32_t depth;         /* wide-tree levels (traversal stack bound) */
    uint32_t n_nodes_cap;
    uint64_t tris_offset;   /* byte offset of the 48-byte triangle records */
    uint64_t nodes_offset;  /* byte offset of the node array */
    uint64_t used_bytes;    /* prefix of the blob that must travel (NCCL broadcast / save) */
    float aabb_lo[3];
    float aabb_hi[3];
    uint32_t bad_index_faces;  /* faces whose vertex indices were out of range (build error) */
    uint32_t node_overflow;    /* node pool overflow (internal error, must be 0) */
    uint64_t parents_offset;   /* byte offset of the per-node (parent << 3 | slot) array used by rt_bvh_refit */
    uint32_t reserved[40];
} rt_blob_header;

/* Size of the scratch buffer every trace call needs (zeroed by the call itself unless
 * RT_OPT_SCRATCH_ZEROED is set, see rt_trace_opts). */
#define RT_TRACE_SCRATCH_BYTES 256

/*
 * Per-call options of every trace entry point (NULL = all defaults).  Replaces what the reference
 * hard-codes: tmin = 0 / tmax = 1e7 on every optixTrace (shaders.cu:86,112,163,191,238).  There is no
 * per-thread or per-process state behind the trace calls: everything a launch depends on is in its
 * arguments.
 *   tmax        far end of the open ray interval (0, tmax); <= 0 selects RT_TMAX_DEFAULT.
 *   ray_first / ray_count
 *               trace only rays [ray_first, ray_first + ray_count) of the descriptor's flattened
 *               (row-major) index space; ray_count <= 0 = up to the end, so a zero-initialised struct
 *               means the whole batch (a caller with an empty window simply does not call).  Outputs are indexed by
 *               (ray - ray_first), i.e. the output pointers belong to the window.  Lets a caller
 *               chunk or shard an arbitrarily strided batch without copying it.
 *   schedule    RT_SCHED_AUTO picks by ray coherence (one shared origin = coherent); the others
 *               force a traversal schedule (all give bit-identical results).
 *   refill_threshold, tri_threshold, grid_div
 *               scheduling knobs for experiments, 0 = default.
 *   flags       RT_OPT_SCRATCH_ZEROED: the caller guarantees that `scratch` is all zero on entry
 *               (stream-ordered); the kernel then restores it to zero before it exits, so a launch
 *               is exactly one kernel and the same scratch can be reused by the next call on the
 *               same stream without a memset.  RT_OPT_STOP_WHEN_BROKEN, RT_OPT_NO_LANE_SHARING,
 *               RT_OPT_NO_TILE_ORDER: see below (the last two switch off scheduling refinements that never
 *               change a result; they exist for A/B measurements and tests).
 */
#define RT_SCHED_AUTO 0
#define RT_SCHED_DIRECT 1       /* triangles tested inside the node step, per lane (round-1 coherent schedule) */
#define RT_SCHED_QUEUED 2       /* per-lane triangle queues (round-1 incoherent schedule) */
#define RT_SCHED_COOP_COHERENT 3   /* warp-shared (ray, triangle) pair list tested by all 32 lanes, late re-fill */
#define RT_SCHED_COOP_INCOHERENT 4 /* same, early re-fill from a pool of prepared rays */
#define RT_SCHED_SLOTS 5           /* rays live in per-warp slots handed around by queues: lanes never wait for triangle
                                      tests, results are written 32 rays at a time (closest / first / any / count) */
#define RT_OPT_SCRATCH_ZEROED 1u
#define RT_OPT_STOP_WHEN_BROKEN 2u /* rt_contains_parity only: the launch may stop as soon as flags_dev[1] (any broken) is
                                      known to be 1; contain / broken entries are then unspecified for the points it skipped.
                                      For callers that discard the per-point results in that case, like the retry of
                                      ray_optix.py:272-279 (a retry with broken points yields all False for the subset). */
#define RT_OPT_NO_LANE_SHARING 4u  /* cooperative schedules: lanes of a warp that can draw no more rays normally take over
                                      part of a neighbour's traversal stack (results are identical either way); this
                                      switches that off (experiments) */
#define RT_OPT_NO_TILE_ORDER 8u    /* coherent image batches [.., H, W, 3] (H % 4 == 0, W % 8 == 0) are normally traced in
                                      8x4-pixel tiles per warp instead of 32-pixel row segments (same results, indexed
                                      by ray); this keeps the row order (experiments) */
typedef struct rt_trace_opts {
    float tmax;
    int32_t schedule;
    int64_t ray_first;
    int64_t ray_count;
    uint32_t flags;
    int32_t refill_threshold;
    int32_t tri_threshold;
    int32_t grid_div;
    int32_t reserved[4];
} rt_trace_opts;

const char* rt_last_error(void);
int rt_abi_version(void);
/* number of SMs of the current device (0 when there is no device) */
int rt_device_sm_count(void);

/* ---- BVH build: replaces OptixAccelStructureWrapperCPP::buildAccelStructure
 *      (ray.cpp:27-100) = optixAccelComputeMemoryUsage + optixAccelBuild + optixAccelCompact.
 *      Morton codes -> onesweep radix sort -> Karras LBVH -> refit -> 8-wide quantised nodes. */
int rt_bvh_sizes(int64_t n_verts, int64_t n_faces, size_t* workspace_bytes, size_t* blob_bytes);
int rt_bvh_build(const float* vertices, int64_t n_verts,   /* [n_verts,3] f32 contiguous */
                 const int32_t* faces, int64_t n_faces,    /* [n_faces,3] i32 contiguous */
                 void* workspace, size_t workspace_bytes,
                 void* blob, size_t blob_bytes, void* stream);
/* Same topology, new vertex positions: rewrites the triangle records and re-fits every node box
 * bottom-up in the existing blob (SURVEY 8f rank 1; the reference rebuilds from scratch in
 * update_raw, ray_optix.py:55-69).  `blob` must be the complete blob rt_bvh_build produced (not just
 * its used prefix).  workspace: rt_bvh_refit_sizes() bytes. */
int rt_bvh_refit_sizes(int64_t n_faces, size_t* workspace_bytes);
int rt_bvh_refit(const float* vertices, int64_t n_verts, const int32_t* faces, int64_t n_faces,
                 void* workspace, size_t workspace_bytes, void* blob, size_t blob_bytes, void* stream);

/* ---- Radix sort exposed for testing (the builder's onesweep sort, 64-bit key + 32-bit value). */
int rt_sort_sizes(int64_t n, size_t* workspace_bytes);
int rt_sort_pairs_u64(uint64_t* keys, uint32_t* vals, int64_t n, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ---- Trace entry points.  `scratch` = RT_TRACE_SCRATCH_BYTES device bytes private to the call. */
/* replaces intersectsAny (ray.cpp:161-189; programs shaders.cu:67-89): hit[r] = 1 iff some triangle
 * is hit with 0 < t < 1e7. */
int rt_trace_any(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, uint8_t* hit, void* scratch,
                 void* stream);
/* replaces intersectsFirst (ray.cpp:191-219; shaders.cu:93-116): nearest-hit triangle index or -1. */
int rt_trace_first(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int32_t* tri_idx, void* scratch,
                   void* stream);
/* replaces intersectsClosest (ray.cpp:231-289; shaders.cu:120-172).  Outputs dense in ray order:
 * hit u8, front u8, tri i32 (-1 on miss), loc f32x3 (0 on miss), uv f32x2 = (w0, w1) (0 on miss). */
int rt_trace_closest(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, uint8_t* hit, uint8_t* front,
                     int32_t* tri_idx, float* loc, float* uv, void* scratch, void* stream);
/* Fused ray generation + closest hit (SURVEY 8f rank 3): the pinhole rays of the reference's benchmark
 * (gen_rays, test/performance_test.py:10-20: d = normalize(x-(w-1)/2, y-(h-1)/2, -f) @ cam_mat^T, all rays
 * from `origin`) are generated in registers, so no ray tensor is read.  Outputs are [height, width] dense. */
typedef struct rt_pinhole {
    int64_t width, height;
    float focal;
    float cam_mat[9];   /* row-major 3x3 */
    float origin[3];
} rt_pinhole;
int rt_trace_closest_pinhole(const void* blob, const rt_pinhole* cam, const rt_trace_opts* opts, uint8_t* hit,
                             uint8_t* front, int32_t* tri_idx, float* loc, float* uv, void* scratch, void* stream);
/* replaces intersectsCount (ray.cpp:291-322; shaders.cu:176-194): exact number of triangles hit. */
int rt_trace_count(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int32_t* count, void* scratch,
                   void* stream);

/* ---- Stream compaction: replaces the boolean-mask indexing of ray_optix.py:142-144 / :219-223.
 *      Step 1 scans the hit mask (decoupled look-back), writing one exclusive prefix per
 *      RT_COMPACT_TILE rays and the total; the host reads `total` to size the outputs
 *      (the only sync the reference API makes unavoidable); step 2 scatters. */
#define RT_COMPACT_TILE 2048
int rt_compact_sizes(int64_t nray, size_t* workspace_bytes);
int rt_compact_scan(const uint8_t* hit, int64_t nray, void* workspace, size_t workspace_bytes,
                    int64_t* total_dev, void* stream);
int rt_compact_scatter(const uint8_t* hit, int64_t nray, const void* workspace,
                       const uint8_t* front, const int32_t* tri_idx, const float* loc, const float* uv,
                       uint8_t* front_out, int32_t* ray_idx_out, int32_t* tri_idx_out, float* loc_out,
                       float* uv_out, void* stream);

/* Sharded variant (no counterpart in the single-GPU reference): the same scatter, but every ray index is
 * written as ray_base + local index, as int32 (ray_idx_bytes 4) or int64 (8, for jobs of more than 2^31 rays), and the
 * *_out pointers are taken as given - they may point into ANOTHER GPU's memory (NVLink peer mapping), already offset
 * to this rank's first packed row, so that the ranks of a ray-sharded job pack their hits straight into one tensor
 * on the root (triro/distributed.py). */
int rt_compact_scatter_at(const uint8_t* hit, int64_t nray, const void* workspace,
                          const uint8_t* front, const int32_t* tri_idx, const float* loc, const float* uv,
                          int64_t ray_base, int ray_idx_bytes, uint8_t* front_out, void* ray_idx_out,
                          int32_t* tri_idx_out, float* loc_out, float* uv_out, void* stream);

/* ---- All hits: replaces intersectsLocation (ray.cpp:324-378; shaders.cu:196-246), i.e. the
 *      reference's count pass + clamp/cumsum (ray.cpp:333-342) + second traversal, in ONE traversal:
 *      step 1 traces once, storing up to max_hits (<= RT_MAX_HITS_LIMIT, reference: 8) hits per ray into
 *      `staging` (nray * max_hits * 16 bytes: tri, x, y, z) and the clamped count per ray, then
 *      scans the counts; step 2 packs them by ray.  nray here is the size of the traced WINDOW
 *      (opts->ray_count): a caller bounds the staging memory by tracing a large batch window by
 *      window (the Python host does, see ops.intersects_location). */
int rt_allhits_sizes(int64_t nray, int max_hits, size_t* staging_bytes, size_t* workspace_bytes);
int rt_allhits_trace(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int max_hits,
                     int32_t* count_clamped, void* staging, void* workspace, size_t workspace_bytes,
                     int64_t* total_dev, void* scratch, void* stream);
int rt_allhits_scatter(int64_t nray, int max_hits, const int32_t* count_clamped, const void* staging,
                       const void* workspace, float* loc_out, int32_t* ray_idx_out, int32_t* tri_idx_out,
                       void* stream);

/* Sharded / windowed variant of rt_allhits_scatter, see rt_compact_scatter_at. */
int rt_allhits_scatter_at(int64_t nray, int max_hits, const int32_t* count_clamped, const void* staging,
                          const void* workspace, int64_t ray_base, int ray_idx_bytes, float* loc_out,
                          void* ray_idx_out, int32_t* tri_idx_out, void* stream);

/* ---- contains_points core: replaces the two intersectsCount launches + ~15 torch kernels of
 *      ray_optix.py:236-267.  For each point traces +dir and -dir exhaustively and writes
 *        contain[i] = inside_aabb & odd(+) & odd(-)
 *        broken[i]  = !(odd(+) & odd(-)) & (count(+)==0 | count(-)==0)
 *      flags_dev[0] = any(inside_aabb), flags_dev[1] = any(broken).  `points` describes
 *      the point batch through the origins fields of rt_ray_desc (directions ignored).
 *      `active` (may be NULL) is a per-point mask: only points with active[i] != 0 are traced and
 *      written, the others keep their contain/broken bytes.  `active` may alias `broken`: the retry of
 *      ray_optix.py:272-277 (`contains[broken] = contains_points(points[broken], new_dir)`) is then one
 *      in-place launch with no gather or scatter. */
int rt_contains_parity(const void* blob, const rt_ray_desc* points, const rt_trace_opts* opts, const float dir[3],
                       const float aabb_lo[3], const float aabb_hi[3], const uint8_t* active, uint8_t* contain,
                       uint8_t* broken, int32_t* flags_dev, void* scratch, void* stream);

/* ---- Instrumented traversal (same code path, counters compiled in): feeds the
 *      bytes-per-ray figure of the roofline.  mode: 0 closest, 1 any, 2 count.
 *      counters_dev[0] = BVH8 nodes fetched, [1] = triangles fetched, [2] = rays, [3] = hits. */
int rt_trace_stats(const void* blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int mode,
                   uint64_t* counters_dev, void* scratch, void* stream);

/* ---- Closest point on the mesh (trimesh.proximity.closest_point; no counterpart in the reference).
 *      Outputs dense over the point batch/window: closest f32x3, distance f32, tri i32, uv f32x2 = (w0, w1).
 *      max_distance: +inf = unbounded; NaN or negative -> RT_ERR_INVALID. counters_dev: NULL or u64[4].
 *      `points` describes the batch through the origins fields of rt_ray_desc (directions ignored), opts supplies
 *      the window (ray_first / ray_count); tmax and schedule are ignored.  tri_idx[i] is the triangle minimising
 *      (d2, tri) over all triangles with d2 <= fl(max_distance * max_distance), d2 being the binary32 squared
 *      distance of the closest point rt_point.cuh computes; ties go to the smaller index, so the result does not
 *      depend on the BVH or the launch.  distance = correctly rounded sqrt(d2).  uv are the weights of the
 *      triangle's vertices 0 and 1 (the convention of rt_trace_closest).  No triangle within reach (empty mesh,
 *      non-finite point, everything beyond max_distance): tri -1, distance +inf, closest 0, uv 0.
 *      counters_dev (instrumented kernel when not NULL): [0] BVH8 nodes fetched, [1] triangles tested, [2] points,
 *      [3] points with an answer.  `scratch` is accepted like every trace call's and left untouched. */
int rt_closest_point(const void* blob, const rt_ray_desc* points, const rt_trace_opts* opts, float max_distance,
                     float* closest, float* distance, int32_t* tri_idx, float* uv, uint64_t* counters_dev,
                     void* scratch, void* stream);

/* ---- Host-buffer entry points (end-to-end path): rays and results live in (pinned) HOST memory.
 *      Copies ray chunks H2D, traces and copies results D2H on internal streams, overlapping
 *      the three; `dev_work` is caller-provided device memory of rt_host_closest_sizes() bytes.
 *      Synchronous: returns when the results are in the host buffers. */
int rt_host_closest_sizes(int64_t nray, size_t* dev_work_bytes);
int rt_host_trace_closest(const void* blob, int64_t nray, const float* h_origins /* [nray,3] or [1,3] */,
                          int origins_broadcast, const float* h_directions /* [nray,3] */,
                          const rt_trace_opts* opts, uint8_t* h_hit, uint8_t* h_front, int32_t* h_tri_idx,
                          float* h_loc, float* h_uv, void* dev_work, size_t dev_work_bytes);
/* Same with stream compaction on the device (intersects_closest(stream_compaction=True), ray_optix.py:139-146):
 * the dense hit mask h_hit[nray] plus the packed rows of the rays that hit, in ascending ray order:
 * h_front[h], h_ray_idx[h], h_tri_idx[h], h_loc[h,3], h_uv[h,2]; *n_hit_out = h.  The packed host buffers must
 * hold nray rows (worst case).  D2H traffic is 1 + 29 * hit_fraction bytes per ray instead of 26. */
int rt_host_trace_closest_compact(const void* blob, int64_t nray, const float* h_origins, int origins_broadcast,
                                  const float* h_directions, const rt_trace_opts* opts, uint8_t* h_hit,
                                  uint8_t* h_front, int32_t* h_ray_idx, int32_t* h_tri_idx, float* h_loc, float* h_uv,
                                  int64_t* n_hit_out, void* dev_work, size_t dev_work_bytes);

#ifdef __cplusplus
}
#endif
#endif /* RAYMESH_B200_H */
