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
#define RT_SCHED_QUEUED 2       /* removed schedule (per-lane triangle queues): accepted as RT_SCHED_COOP_INCOHERENT,
                                   the number is not reused */
#define RT_SCHED_COOP_COHERENT 3   /* warp-shared (ray, triangle) pair list tested by all 32 lanes, late re-fill */
#define RT_SCHED_COOP_INCOHERENT 4 /* same, early re-fill from a pool of prepared rays */
#define RT_SCHED_SLOTS 5           /* removed schedule (rays in per-warp slots): accepted as RT_SCHED_COOP_INCOHERENT,
                                      the number is not reused */
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

/* ---- Generalized winding number (Jacobson, Kavan, Sorkine-Hornung 2013; libigl's fast_winding_number, Barill et al.
 *      2018; no counterpart in the reference): w(q) = sum over triangles of the signed solid angle / 4 pi, orientation
 *      from the face order.  ~1 inside and ~0 outside a closed outward-facing mesh; meaningful for open meshes, soups
 *      and self-intersecting meshes too (nested shells add up, open surfaces give fractions).
 *
 *      rt_winding_moments fills the per-node moment array (64 bytes per node: area-weighted centroid, radius bound,
 *      sum of area vectors, first-moment tensor) bottom-up from any valid blob: built, re-fitted, broadcast or loaded.
 *      It is a side array, not part of the blob: recompute it after rt_bvh_refit.  Sizes: rt_winding_moments_sizes
 *      bounds them from the triangle count (for any leaf size); a caller that knows the blob's node count (header
 *      n_nodes) may pass exactly n_nodes * 64 moment bytes and a workspace of two 256-byte aligned arrays of
 *      n_nodes * 4 bytes.  Moments 16-byte and workspace 256-byte aligned.  A blob with more nodes than the buffers
 *      can hold is left without moments (nothing is written).
 *
 *      rt_winding_number: winding[i] for every point of the batch/window (`points` through the origins fields of
 *      rt_ray_desc, opts for ray_first / ray_count only).  Triangles in leaf slots are summed exactly; an inner child
 *      whose moment ball is far (|p~ - q| > beta * radius) adds its two-term far-field expansion instead of being
 *      visited.  beta >= 1 (libigl's default is 2); beta = +inf sums every triangle exactly; beta < 1 or NaN ->
 *      RT_ERR_INVALID.  A triangle with a non-finite vertex or a zero computed determinant contributes 0; a
 *      non-finite point gives NaN; an empty mesh gives +0.  The result is a function of (blob, moments, point, beta)
 *      only.  counters_dev (instrumented kernel when not NULL): [0] BVH8 nodes visited, [1] triangles summed exactly,
 *      [2] points, [3] far-field terms.  `scratch` is accepted like every trace call's and left untouched. */
int rt_winding_moments_sizes(int64_t n_faces, size_t* moments_bytes, size_t* workspace_bytes);
int rt_winding_moments(const void* blob, void* moments, size_t moments_bytes, void* workspace, size_t workspace_bytes,
                       void* stream);
int rt_winding_number(const void* blob, const void* moments, const rt_ray_desc* points, const rt_trace_opts* opts,
                      float beta, float* winding, uint64_t* counters_dev, void* scratch, void* stream);

/* ---- Pseudo-normal signed distance (Baerentzen & Aanaes 2005, "Signed distance computation using the angle weighted
 *      pseudonormal"; no counterpart in the reference): the sign of the closest point's feature normal, exact for a
 *      closed, manifold, consistently oriented mesh, with one closest-point walk per point.
 *
 *      rt_pseudonormals fills the side array of 96 bytes per triangle record (6 x f32x4: the angle-weighted normals of
 *      vertices a, b, c and the normals of edges ab, ac, bc) from any valid blob: built, re-fitted, broadcast or loaded.
 *      Corners are welded by exact equality of their coordinates (-0 = +0), not by the face indices, so an unwelded
 *      soup of a closed surface gets the normals of the welded mesh; a triangle with a non-finite vertex takes part in
 *      nothing.  It is a side array, not part of the blob: recompute it after rt_bvh_refit.  normals_bytes / 96 is the
 *      capacity in triangles (at most 2^30 / 3, else RT_ERR_INVALID); a blob with more triangles than that is left
 *      without normals.  Normals 16-byte and workspace 256-byte aligned; rt_pseudonormals_sizes gives both sizes for
 *      n_faces triangles.  edge_counts_dev (u64[3], zeroed by the call): [0] boundary edges (one face), [1]
 *      non-manifold edges (more than two faces), [2] inconsistent edges (two faces that traverse it the same way), on
 *      the welded surface.  The sign below is an inside/outside answer when all three are 0.
 *
 *      rt_signed_distance: signed_distance[i] for every point of the batch/window (`points` through the origins fields
 *      of rt_ray_desc, opts for ray_first / ray_count only).  |signed_distance| is bit for bit the distance of
 *      rt_closest_point (max_distance = +inf) and the closest triangle is the one it picks; the value is +d when
 *      (p - c) . n < 0 for the pseudo-normal n of the Voronoi region of c (face, edge or vertex), else -d; an exact
 *      d = 0 gives +0; a non-finite point or an empty mesh gives -inf.  A function of (blob, normals, point) only.
 *      counters_dev: NULL or u64[4] as for rt_closest_point.  `scratch` is accepted and left untouched. */
int rt_pseudonormals_sizes(int64_t n_faces, size_t* normals_bytes, size_t* workspace_bytes);
int rt_pseudonormals(const void* blob, void* normals, size_t normals_bytes, void* workspace, size_t workspace_bytes,
                     uint64_t* edge_counts_dev, void* stream);
int rt_signed_distance(const void* blob, const void* normals, const rt_ray_desc* points, const rt_trace_opts* opts,
                       float* signed_distance, uint64_t* counters_dev, void* scratch, void* stream);
/*      rt_signed_distance_closest: rt_signed_distance (the same signed_distance bits) that also writes closest [n,3],
 *      tri_idx [n] and uv [n,2] exactly as rt_closest_point does (tri -1, closest 0, uv 0 where there is no
 *      triangle).  All three outputs are required. */
int rt_signed_distance_closest(const void* blob, const void* normals, const rt_ray_desc* points, const rt_trace_opts* opts,
                               float* signed_distance, float* closest, int32_t* tri_idx, float* uv, uint64_t* counters_dev,
                               void* scratch, void* stream);

/* ---- Gradient of the distance (DESIGN.md §4.9): the backward of rt_closest_point's distance and of the signed
 *      distances, from the forward's outputs alone (no BVH walk).  With g = grad_out[i], s = -1 when value[i] has its
 *      sign bit set else +1, c = closest[i], (w0, w1, w2) = (uv0, uv1, 1 - uv0 - uv1):
 *        grad_points[i]              = g * s * (p - c) / |value|                      (= q_i)
 *        grad_vertices[faces[t][k]] += -w_k * q_i       for k = 0, 1, 2, t = tri_idx[i]
 *      A point with value +-0, +-inf or NaN, tri_idx outside [0, n_faces), or a vertex index outside [0, n_verts)
 *      contributes 0 (its grad_points row is +0).  `points`, opts (ray_first / ray_count) and the outputs of the
 *      forward are laid out as in rt_closest_point: value, closest, tri_idx and uv indexed by the position in the
 *      window, faces int32 [n_faces, 3].  grad_points (dense [n,3]) and grad_vertices ([n_verts,3], overwritten) may
 *      each be NULL.  Deterministic: the vertex sums are stably sorted by vertex and reduced in a fixed tree over
 *      each vertex's contributions in point order (groups of 32, left to right, then groups of 32 of those sums),
 *      independent of the launch.  The batch runs as consecutive point windows of the size that fits
 *      workspace_bytes (at most 2^30 / 3 points); grad_vertices starts at +0 and each window's sums are added in
 *      window order.  rt_distance_grad_sizes: workspace for one window of n_points (the whole batch when it fits one
 *      window); none is needed when grad_vertices is NULL.  Workspace 256-byte aligned. */
int rt_distance_grad_sizes(int64_t n_points, int64_t n_verts, size_t* workspace_bytes);
int rt_distance_grad(const rt_ray_desc* points, const rt_trace_opts* opts, const float* grad_out, const float* value,
                     const float* closest, const int32_t* tri_idx, const float* uv, const int32_t* faces, int64_t n_faces,
                     int64_t n_verts, float* grad_points, float* grad_vertices, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ---- Gradient of the hit locations and barycentrics (DESIGN.md §4.10): the backward of rt_trace_closest's loc and uv
 *      (dense or compacted) and of the all-hits loc, with respect to the rays and the mesh vertices, without a BVH
 *      walk.  Row i is the hit of triangle t = tri_idx[i] by ray r = row_ray[i] of the window (row_ray NULL: r = i,
 *      and n_rows must equal the window's ray count unless it is 0); g_L = grad_loc[i] (NULL: 0) and
 *      g_U = grad_uv[i] (NULL: 0).
 *      With v0, v1, v2 = vertices[faces[t]], e1 = v1 - v0, e2 = v2 - v0, the hit is recomputed in binary32 with one
 *      fixed Moeller-Trumbore sequence:
 *        s = o - v0, p = d x e2, det = e1.p, b1 = s.p / det, r = s x e1, b2 = d.r / det, t = e2.r / det
 *        gb1 = g_L.e1 - g_U0 + g_U1, gb2 = g_L.e2 - g_U0, lambda = (gb1 p + gb2 (e1 x d)) / det
 *        grad_origins[r] += lambda, grad_directions[r] += t lambda,
 *        grad_vertices[faces[t][k]] += -w_k (lambda - g_L),   w = (1 - b1 - b2, b1, 1 - w0 - w1)
 *      A row whose triangle is outside [0, n_faces), with a vertex index outside [0, n_verts), a row_ray outside
 *      the window, det = 0, or any non-finite value among lambda, t lambda, lambda - g_L and w contributes 0.  The
 *      rows of one ray must be contiguous (row_ray non-decreasing, as rt_compact_scatter and rt_allhits_scatter
 *      write it); each ray's sums run over its rows left to right from +0, and rays without rows get +0 (with
 *      n_rows = 0 every ray and vertex does, whatever row_ray is).  The vertex sums are those of rt_distance_grad: a
 *      stable sort by vertex and the fixed 32-ary tree per vertex, in row windows of the size that fits
 *      workspace_bytes (at most 2^30 / 3 rows), added in window order.  The zero rules are per row: finite rows can
 *      still overflow in a product or a sum, as in rt_distance_grad.
 *      `rays` and opts (ray_first / ray_count only) are those of the forward; vertices float32 [n_verts, 3], faces
 *      int32 [n_faces, 3].  grad_origins and grad_directions (dense [window, 3]) and grad_vertices ([n_verts, 3],
 *      overwritten) may each be NULL.  rt_ray_grad_sizes: workspace for one window of n_rows (the whole batch when it
 *      fits one window); none is needed when grad_vertices is NULL.  Workspace 256-byte aligned. */
int rt_ray_grad_sizes(int64_t n_rows, int64_t n_verts, size_t* workspace_bytes);
int rt_ray_grad(const rt_ray_desc* rays, const rt_trace_opts* opts, int64_t n_rows, const int32_t* row_ray,
                const int32_t* tri_idx, const float* grad_loc, const float* grad_uv, const float* vertices, int64_t n_verts,
                const int32_t* faces, int64_t n_faces, float* grad_origins, float* grad_directions, float* grad_vertices,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- Instanced scenes (DESIGN.md §4.11; the reference's OptiX instance acceleration structures were never exposed):
 *      M meshes (BVH8 blobs from rt_bvh_build) and I instances, instance i = (mesh m_i, affine object->world transform
 *      (A_i | b_i) as a row-major binary32 3x4).  The world ray (o, d) meets instance i as o' = A_i^-1 (o - b_i),
 *      d' = A_i^-1 d, with the same t.
 *
 *      rt_scene_prepare_sizes: bytes of the scene table (256-byte aligned device memory) for M meshes and I instances.
 *      rt_scene_prepare: `blobs` (HOST array of M device addresses, each a blob of the current device), `inst_mesh`
 *      (HOST int32 [I]) and `transforms` (HOST f32 [I,3,4]) are checked on the host: a mesh index outside [0, M), a
 *      non-finite transform, det(A) = 0 in binary64, or an inverse that overflows binary32 -> RT_ERR_INVALID, and
 *      nothing is written.  Then one kernel reads each mesh's header box from the device, computes A^-1 and the
 *      object-space offset -A^-1 b in binary64, rounds them to binary32 once, and writes the instance table plus the
 *      top-level geometry: tlas_vertices f32 [2I,3] = the padded world boxes (lo_i, hi_i), tlas_faces i32 [I,3] =
 *      (2i, 2i+1, 2i).  Build the top-level tree from those with rt_bvh_build (its records' prim is the instance).  An
 *      instance of a mesh without triangles gets a point box and is never entered.  Asynchronous on `stream`; the
 *      host arrays may be released when it returns.  Rebuilding or re-fitting a member blob makes the table stale:
 *      prepare again.
 *
 *      rt_scene_trace: one query for the batch/window (rays, opts: tmax, ray_first / ray_count) against the table and
 *      the top-level blob.  mode RT_SCENE_CLOSEST: the hit minimising (t, inst, prim) over every instance in
 *      (0, tmax); hit u8, front u8 (object-space front face XOR det(A) < 0), inst_idx i32, tri_idx i32 (row of the
 *      instance's mesh faces), loc f32x3 (the world point A loc_obj + b), uv f32x2 (object-space weights of v0, v1);
 *      a miss gives inst_idx = tri_idx = -1 and 0 elsewhere.  RT_SCENE_ANY: hit.  RT_SCENE_COUNT: count i32 = the sum
 *      over instances of the crossings in (0, tmax).  Outputs the mode does not write may be NULL.  One identity
 *      instance gives the bits of rt_trace_closest / _any / _count on its mesh. */
#define RT_SCENE_CLOSEST 0
#define RT_SCENE_ANY 1
#define RT_SCENE_COUNT 2
int rt_scene_prepare_sizes(int64_t n_meshes, int64_t n_inst, size_t* table_bytes);
int rt_scene_prepare(int64_t n_meshes, const void* const* blobs, int64_t n_inst, const int32_t* inst_mesh,
                     const float* transforms, void* table, size_t table_bytes, float* tlas_vertices, int32_t* tlas_faces,
                     void* stream);
int rt_scene_trace(const void* table, const void* tlas_blob, const rt_ray_desc* rays, const rt_trace_opts* opts, int mode,
                   uint8_t* hit, uint8_t* front, int32_t* inst_idx, int32_t* tri_idx, float* loc, float* uv, int32_t* count,
                   void* stream);

/* ---- Point queries on instanced scenes (DESIGN.md §4.12), on a table and top-level blob from rt_scene_prepare.
 *      The world triangle t of instance i has the vertices W_k = affine_row(A_i row, b_i (0 as -0), v_k) in binary32,
 *      the sequence rt_scene_trace uses for loc.
 *
 *      rt_scene_point_sizes: bytes of the side array (16-byte aligned device memory) for I instances.
 *      rt_scene_point_prepare: one kernel writes the side array (per instance a lower bound on the smallest singular
 *      value of A_i and the margins of the instance walk's bound) from the table and its meshes' header boxes.  A
 *      function of those alone; prepare again after rt_scene_prepare.  Asynchronous on `stream`.
 *
 *      rt_scene_closest_point: for each point of the batch/window (points, opts: ray_first / ray_count) the (inst, prim)
 *      minimising the key (d2, inst, prim) over every non-empty instance and triangle with d2 <= fl(max_distance^2),
 *      d2 = the single-mesh point/triangle distance of rt_closest_point on the world triangle.  closest f32x3 (world),
 *      distance f32 = sqrt(d2), inst_idx i32, tri_idx i32 (row of the instance's mesh faces), uv f32x2 (weights of
 *      v0, v1).  A point with none (nothing in reach, non-finite point, empty scene): inst = tri = -1, distance +inf,
 *      closest and uv 0.  max_distance must be >= 0 or +inf (NaN or negative -> RT_ERR_INVALID).  The result equals
 *      rt_closest_point on the mesh of every instance's affine_row world vertices, faces in instance order, bit for bit.
 *
 *      rt_scene_signed_distance: the same walk with max_distance +inf, then the pseudo-normal sign of rt_signed_distance
 *      with the normal carried to world space as A^-T n (from the stored binary32 inverse): +d when (p - c) . n_w < 0,
 *      -d otherwise, +0 for d = 0, -inf for a point without answer.  `normals_table`: DEVICE array of M addresses, the
 *      rt_pseudonormals rows of each mesh (any 16-byte aligned address for a mesh without triangles); NULL or misaligned
 *      -> RT_ERR_INVALID.  closest, inst_idx, tri_idx and uv are all NULL or all set (then written as by
 *      rt_scene_closest_point).  The sign is that of inside/outside when every mesh is closed, manifold and consistently
 *      oriented, every A_i is a similarity (mirrors allowed) and the instances do not overlap. */
int rt_scene_point_sizes(int64_t n_inst, size_t* side_bytes);
int rt_scene_point_prepare(const void* table, int64_t n_inst, void* side, size_t side_bytes, void* stream);
int rt_scene_closest_point(const void* table, const void* tlas_blob, const void* side, const rt_ray_desc* points,
                           const rt_trace_opts* opts, float max_distance, float* closest, float* distance, int32_t* inst_idx,
                           int32_t* tri_idx, float* uv, void* stream);
int rt_scene_signed_distance(const void* table, const void* tlas_blob, const void* side, const void* normals_table,
                             const rt_ray_desc* points, const rt_trace_opts* opts, float* signed_distance, float* closest,
                             int32_t* inst_idx, int32_t* tri_idx, float* uv, void* stream);

/* ---- Gradients of instanced-scene queries (DESIGN.md §4.13): the backward of rt_scene_trace's closest-hit loc and uv
 *      (dense or compacted) and of rt_scene_closest_point's distance / rt_scene_signed_distance's value, with respect
 *      to the rays or points, the instance transforms and the member vertices, without a walk.
 *      `members`: DEVICE array of one rt_scene_member per mesh of the table: the member's vertices f32 [n_verts, 3] and
 *      faces i32 [n_faces, 3] as of the forward, and vertex_base, the row of its vertex 0 in grad_vertices
 *      ([n_verts_total, 3]).  `n_inst` and `n_meshes` bound what the rows may index (the table's own counts when
 *      smaller).  Row j is (instance i = inst_idx[j], triangle t = tri_idx[j]); with A | b the table's transform of i,
 *      v_k the member's vertices of face t and w its barycentrics:
 *        hit rows: the hit is recomputed as rt_ray_grad does on the WORLD triangle W_k = affine_row(A row, b (0 as -0),
 *          v_k); lambda, t lambda, q = lambda - g_L and w are rt_ray_grad's, and so are the per-ray sums into
 *          grad_origins / grad_directions (rows of one ray contiguous, row_ray NULL: row j is ray j).
 *        point rows: q = rt_distance_grad's grad_points row (from grad_out, value, closest), w = (uv0, uv1).
 *        Then, with w2 = (1 - w0) - w1, x = (w0 v0 + w1 v1) + w2 v2 and q_obj_j = affine_row(A column j, -0, q):
 *          grad_transforms[i][r][j] += -x_j q_r (j < 3),  grad_transforms[i][r][3] += -q_r,
 *          grad_vertices[vertex_base + faces[t][k]] += -w_k q_obj.
 *      A row contributes 0 everywhere (its own grad_points row included) when inst is outside [0, n_inst), its mesh
 *      outside [0, n_meshes), t outside the member's faces, a vertex index outside its vertices or vertex_base + index
 *      outside [0, n_verts_total), det = 0 (hit rows), value +-0, +-inf or NaN (point rows), a hit row's ray outside
 *      the window, or when any of lambda, t lambda, q, w, x, q_obj is not finite.  The transform columns and the vertices
 *      are summed as rt_distance_grad sums vertices: one stable sort of (key, pair) over the joint key space
 *      [member vertices | 4 I transform columns], the fixed 32-ary tree per key in ascending (row, corner) order, in
 *      row windows of the size that fits workspace_bytes (at most 2^30 / 7 rows), added in window order from +0.
 *      grad_origins / grad_directions / grad_points (dense [window, 3]), grad_transforms (f32 [n_inst, 3, 4],
 *      overwritten) and grad_vertices ([n_verts_total, 3], overwritten) may each be NULL.  n_verts_total + 4 n_inst
 *      must stay below 2^32 - 1.  rt_scene_grad_sizes: workspace for one window of n_rows, `outputs` =
 *      RT_SCENE_GRAD_TRANSFORMS | RT_SCENE_GRAD_VERTICES as the call will request (0 bytes when neither: none is needed
 *      then).  Workspace 256-byte aligned. */
typedef struct rt_scene_member {
    const float* vertices;
    const int32_t* faces;
    int64_t n_verts, n_faces;
    int64_t vertex_base;
} rt_scene_member;
#define RT_SCENE_GRAD_TRANSFORMS 1
#define RT_SCENE_GRAD_VERTICES 2
int rt_scene_grad_sizes(int64_t n_rows, int64_t n_inst, int64_t n_verts_total, int outputs, size_t* workspace_bytes);
int rt_scene_ray_grad(const void* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                      int64_t n_verts_total, const rt_ray_desc* rays, const rt_trace_opts* opts, int64_t n_rows,
                      const int32_t* row_ray, const int32_t* inst_idx, const int32_t* tri_idx, const float* grad_loc,
                      const float* grad_uv, float* grad_origins, float* grad_directions, float* grad_transforms,
                      float* grad_vertices, void* workspace, size_t workspace_bytes, void* stream);
int rt_scene_distance_grad(const void* table, int64_t n_inst, const rt_scene_member* members, int64_t n_meshes,
                           int64_t n_verts_total, const rt_ray_desc* points, const rt_trace_opts* opts,
                           const float* grad_out, const float* value, const float* closest, const int32_t* inst_idx,
                           const int32_t* tri_idx, const float* uv, float* grad_points, float* grad_transforms,
                           float* grad_vertices, void* workspace, size_t workspace_bytes, void* stream);

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
