/* contourist_b200 -- C ABI of the B200-native isosurface engine (libcontourist_b200.so).
 *
 * The reference (AaronWatters/contourist) is pure Python and has NO plugin / FFI / operator
 * interface (SURVEY.md section 8(b)); its boundary is the public Python class API.  This header is
 * therefore the boundary a maintainer binds with ctypes (INTEGRATION.md shows the stub); every entry
 * point names the reference function(s) whose work it replaces (paths are under
 * /root/reference/contourist/).
 *
 * Conventions
 *   - All entry points return 0 on success or a negative ctr_status; ctr_last_error() gives text.
 *   - The caller owns every host buffer; the context owns all device memory and reuses it.
 *   - Two-phase: *_run() computes on the device and reports sizes, *_fetch() copies the results
 *     into caller buffers of exactly those sizes (any pointer may be NULL = "not wanted").
 *   - A context is bound to one device and one stream; it is not thread-safe.  Calls are
 *     synchronous on return.
 *   - field[i][j][k] (C order, last axis contiguous) is the sample at grid point (i,j,k): exactly
 *     the f(i,j,k) the reference's grid-level engines call (tetrahedral.py:129-130).
 *   - Linear point index lin = (i*n1 + j)*n2 + k.  An edge key names a grid edge by its
 *     component-wise-min endpoint and direction: 3D key = lin*8 + d, d = di*4+dj*2+dk in 1..7;
 *     4D key = lin*16 + d, d in 1..15; 2D key = lin*4 + d, d = di*2+dj in 1..3.  This is the
 *     reference's dict key (p_low, p_high) (tetrahedral.py:184-188) made canonical; `lowmin`
 *     says which endpoint is the low one.
 */
#ifndef CONTOURIST_B200_H
#define CONTOURIST_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define CTR_API __attribute__((visibility("default")))
#else
#define CTR_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ctr_ctx ctr_ctx;

typedef enum {
  CTR_OK = 0,
  CTR_ERR_BAD_ARG = -1,
  CTR_ERR_CUDA = -2,
  CTR_ERR_OOM = -3,
  CTR_ERR_UNSUPPORTED = -4,
  CTR_ERR_STATE = -5,
  CTR_ERR_OVERFLOW = -6
} ctr_status;

/* Sample types.  Every entry point takes CTR_F32 and CTR_F64.  The integer types are accepted by the 3D extraction
 * only (ctr_mt3d_run, ctr_mt3d_enqueue and, through the run it selects from, ctr_mt3d_select_seeded); the 2D and 4D
 * runs reject them with CTR_ERR_BAD_ARG.  An integer field gives exactly the result of the same field widened to
 * float64 (every uint8 / int16 / uint16 is exact in fp32 and fp64), so with fp32 geometry it also equals the float32
 * run; stage 1 reads 1 or 2 bytes a sample instead of 4 or 8.  One known exception, in the float path: with
 * CTR_WANT_MINMAX, a float32 / float64 field whose size in bytes is not a multiple of 16 KiB and that takes the TMA
 * stage-1 kernel reports fmax = +inf (the padding of its partial last chunk enters the max); an integer field reports
 * its true maximum. */
typedef enum { CTR_F32 = 0, CTR_F64 = 1, CTR_U8 = 2, CTR_I16 = 3, CTR_U16 = 4 } ctr_dtype;

/* flags */
#define CTR_FIELD_ON_DEVICE 1u /* `field` is a device pointer (no H2D copy)                          */
#define CTR_GEOM_F64 2u        /* positions / normals computed and returned in fp64 (else fp32)      */
#define CTR_WANT_NORMALS 4u    /* gradient normals (engine extension; the reference computes none)   */
#define CTR_WANT_KEYS 8u       /* per-vertex edge key + orientation (parity / dedup across slabs)    */
#define CTR_WANT_CODES 16u     /* compact (cell, 30-bit case code) list of emitting cells            */
#define CTR_NO_GEOMETRY 32u    /* classification, counts and offsets only                            */
#define CTR_WANT_MINMAX 64u    /* field min / max (grid_field.py:79-80); NaN in the counts otherwise   */
#define CTR_MORPH 128u         /* 4D only: run the morph stage (time binning, filtering, slicing)     */

/* ---- context ----------------------------------------------------------------------------------- */
CTR_API int ctr_create(int device, ctr_ctx** out);
CTR_API void ctr_destroy(ctr_ctx* ctx);
/* ctx may be NULL: last error of a failed ctr_create. The pointer stays valid until the next call. */
CTR_API const char* ctr_last_error(const ctr_ctx* ctx);
/* Launch on an existing CUDA stream (a cudaStream_t passed as void*), e.g. torch's current stream. */
CTR_API int ctr_set_stream(ctr_ctx* ctx, void* cuda_stream);
/* Per-stage device times (ms, CUDA events) of the last *_run when timing is enabled.
 * 3D stages: 0 H2D, 1 bitplane (classify), 2 count+scan, 3 emit vertices, 4 emit triangles, 5 codes. */
CTR_API int ctr_set_timing(ctr_ctx* ctx, int enabled);
CTR_API int ctr_stage_times(ctr_ctx* ctx, float* ms, int n);
/* Number of kernels launched by this context since creation (bench.py's gpu_launches). */
CTR_API int64_t ctr_kernel_launches(const ctr_ctx* ctx);

/* Page-locked host memory for the caller's input / output arrays: cudaMemcpyAsync to or from it runs at full PCIe
 * rate (pageable memory is staged through a bounce buffer, ~3x slower for the 0.2-0.5 GB arrays of a 512^3 run). */
CTR_API int ctr_host_alloc(ctr_ctx* ctx, uint64_t bytes, void** out);
CTR_API int ctr_host_free(ctr_ctx* ctx, void* p);

/* Pipelines that span contexts (engine.py: mt3d_extract_host uploads a host volume ONCE on an upload context while
 * two extraction contexts work through its slabs, instead of re-sending each slab's halo planes).
 * ctr_stage_upload: queue, on ctx's stream, the copy of `bytes` from host memory to byte offset `dst_offset` of the
 *   context's staging buffer, which is first grown to `total_bytes` (growing waits for the stream and discards the
 *   content: pass the final size with the first piece).  *device_base receives the buffer's device address; it is
 *   valid until the buffer grows or the context is destroyed.  Returns without waiting for the copy.
 * ctr_wait_for: whatever is queued on ctx after this call starts only when everything queued on `other` so far has
 *   finished (event record + stream wait on the device; the host does not wait).  Both contexts on the same device. */
CTR_API int ctr_stage_upload(ctr_ctx* ctx, const void* host, uint64_t dst_offset, uint64_t bytes, uint64_t total_bytes,
                             void** device_base);
CTR_API int ctr_wait_for(ctr_ctx* ctx, ctr_ctx* other);

/* ---- 3D marching tetrahedra ---------------------------------------------------------------------
 * Replaces, for an array-backed field, the reference's
 *   grid_field.py:64-84     FunctionGrid.find_contour_crossing_grid_segments  (n_crossings, fmin, fmax)
 *   tetrahedral.py:383-469  border_voxel / find_initial_voxels / expand_voxels (full scan instead of flood fill)
 *   tetrahedral.py:554-595  enumerate_voxel_triangles / enumerate_tetrahedron_triangles (case codes, triangles)
 *   tetrahedral.py:176-188,471-512  add_simplex / interpolate_pair / contour_pair_interpolation (keys, positions)
 *   tetrahedral.py:604-614  extract_surface_geometry vertex numbering (deterministic: by 32-sample word of the owner
 *                           point, then edge direction, then k; sort by key for the canonical order)
 *   tetrahedral.py:83-87 + grid_field.py:89-93  grid -> world coordinates
 */
typedef struct {
  const void* field;    /* n0*n1*n2 samples, host or device (CTR_FIELD_ON_DEVICE)                     */
  int32_t dtype;        /* ctr_dtype of field (all five types)                                       */
  uint32_t flags;
  int64_t n0, n1, n2;   /* SAMPLES per axis; voxels have origins in [0, n-2]                          */
  double isovalue;
  double origin[3];     /* world = grid*delta + origin (grid_field.py:89-93); use 0 / 1 for grid units */
  double delta[3];
  /* z-slab sharding (SURVEY.md 8(e)); single GPU: i_lo = 0, i_hi = n0, plane_offset = 0.
   * Voxel layers and owner planes i in [i_lo, i_hi) are emitted; planes outside are halo (needed:
   * 1 below for normals, 2 above for the ids of the next shard's first plane).  plane_offset is the
   * global index of array plane 0; keys and positions are global.                                   */
  int64_t i_lo, i_hi, plane_offset;
  /* added to every vertex id written into the triangles: the number of vertices of the shards before this one, when
   * the caller already knows it (slab-by-slab runs on one device: contourist_b200/engine.py mt3d_extract_host).     */
  int64_t vert_id_base;
} ctr_mt3d_params;

typedef struct {
  int64_t n_verts;        /* vertices emitted by this call (= number of distinct edge keys)           */
  int64_t n_tris;
  int64_t n_active_cells; /* voxels that emit at least one triangle                                   */
  int64_t n_crossings;    /* strictly crossing grid segments, grid_field.py:81                        */
  int64_t n_codes;        /* entries of the (cell, code) list (CTR_WANT_CODES)                        */
  double fmin, fmax;      /* grid_field.py:79-80                                                      */
} ctr_mt3d_counts;

CTR_API int ctr_mt3d_run(ctr_ctx* ctx, const ctr_mt3d_params* p, ctr_mt3d_counts* out);
/* The same extraction split in two: _enqueue returns as soon as every stage is queued on the stream (the field must
 * stay valid), _finish waits for it and reports the counts.  The host can work in between -- e.g. all-gather the
 * counts of the previous volume (bench.py, N > 1).  Not with CTR_WANT_CODES.                                         */
CTR_API int ctr_mt3d_enqueue(ctr_ctx* ctx, const ctr_mt3d_params* p);
CTR_API int ctr_mt3d_finish(ctr_ctx* ctx, ctr_mt3d_counts* out);
/* Device-side copy of the counts (SURVEY.md 8(e): the all-gather of per-rank counts -> vertex / triangle offsets needs
 * no host round trip): from now on every ctr_mt3d_run / _enqueue also stores {n_verts, n_tris} as two int64 at
 * `device_counts` (caller-owned device memory, 16 bytes, valid until replaced) behind its last kernel, on the context's
 * stream -- a collective queued after an event on that stream can send them straight from there.  NULL turns it off. */
CTR_API int ctr_mt3d_publish_counts(ctr_ctx* ctx, void* device_counts);
/* Adds `base` to every vertex id of the last run's device triangles (stream-ordered, no wait): what vert_id_base does,
 * for a base that was not known yet when the run was queued -- slab k+1 of a pipelined host-array extraction is queued
 * (its upload overlapping the kernels of slab k) before slab k's vertex count exists.  Not part of the reference.  */
CTR_API int ctr_mt3d_offset_ids(ctr_ctx* ctx, int64_t base);
/* verts/normals: [n_verts][3] float or double (CTR_GEOM_F64); tris: [n_tris][3] vertex ids, local to
 * this call (0 = first emitted vertex; ids >= n_verts refer to the next shard's vertices; vertices are numbered
 * by owner word (plane-major), then edge direction, then k -- not by key);
 * keys/lowmin: [n_verts]; cells/codes: [n_codes] linear voxel index ((i*(n1-1)+j)*(n2-1)+k, i global)
 * and 30-bit case code (6 tets x (4-bit low mask | 16 if skipped by allclose)), unordered.            */
CTR_API int ctr_mt3d_fetch(ctr_ctx* ctx, void* verts, void* normals, int32_t* tris, uint64_t* keys,
                   uint8_t* lowmin, int64_t* cells, uint32_t* codes);
/* Device pointers of the last run's outputs (valid until the next *_run on this context).          */
CTR_API int ctr_mt3d_device_ptrs(ctr_ctx* ctx, void** verts, void** normals, int32_t** tris);

/* Stage 4b, orientation (SURVEY.md 8(f1)): rewinds the LAST run's device triangles like the reference's
 *   surface_geometry.py:52-140  SurfaceGeometry.orient_triangles
 * does: per edge-connected component, the triangle with the largest |cross.x| at the component's max-x vertex faces +x
 * ("outward" for closed sheets).  The engine's triangles are wound towards the high side of the field, so this is one
 * keep / reverse decision per component.  Fetch afterwards to get the rewound triangles.                            */
CTR_API int ctr_mt3d_orient_reference(ctr_ctx* ctx, int64_t* n_components, int64_t* n_flipped);

/* Connected components of the mesh with their size and topology (engine extension; the reference has none --
 * oracle/mt3d_components.py:components is the definition).  Works on the LAST 3D run's device mesh as it stands now
 * (after ctr_mt3d_select_seeded, ctr_mt3d_clean or ctr_mt3d_orient_reference too); it does not edit the mesh and may be
 * called any number of times.  Synchronous on return.
 *   - Components are EDGE-connected: two triangles are joined when they share an undirected vertex-id edge (the rule of
 *     ctr_mt3d_orient_reference, whose n_components is the same number on every mesh).  Two sheets touching in one
 *     vertex stay apart.
 *   - Numbering: 0..C-1 in ascending order of each component's smallest triangle index (first_tri); deterministic.
 *   - A vertex shared by k components counts in each of their n_verts, so n_verts - n_edges + n_tris is the
 *     component's Euler characteristic (2 for a sphere, 0 for a torus, 1 for a disc cut by the volume's edge).  A
 *     component is closed when n_boundary_edges == 0.
 *   - area and volume are fp64 sums over its triangles (positions widened from the geometry type first), volume
 *     relative to the component's box corner lo.  On the raw engine mesh (triangles wound towards the high side) a
 *     closed component has volume > 0 when the region it encloses is below the isovalue and < 0 when it is above (a
 *     blob brighter than its surroundings: negative).  After ctr_mt3d_orient_reference, or ctr_mt3d_clean with
 *     CTR_CLEAN_ORIENT, every closed component faces outward and its volume is >= 0.  For an open component the value
 *     is reported but is not an enclosed volume.  After ctr_mt3d_cap the components that the box cut are closed by
 *     their caps, so their volumes are enclosed volumes too.
 *   - The integer fields, first_tri and the box are exact.  area and volume are sums whose order may change between
 *     calls: their last bits may differ.
 *   - CTR_ERR_STATE: no 3D run or a CTR_NO_GEOMETRY run; a slab run (i_lo != 0 or i_hi != n0) or vert_id_base != 0; a
 *     triangle id outside [0, n_verts) (e.g. after ctr_mt3d_offset_ids); _fetch with no ctr_mt3d_components since the
 *     last run.  An empty mesh has 0 components.
 *   _components      : *n_components (may be NULL) receives C
 *   _components_fetch: tri_component [n_tris] (the component of every triangle, row for row with ctr_mt3d_fetch's
 *                      triangles) and components [C]; either may be NULL.  These are the results of the last call: a
 *                      later selection or clean-up does not update them (ctr_mt3d_keep_components does).             */
typedef struct {
  int64_t n_tris, n_verts, n_edges;          /* faces, distinct vertices, distinct undirected edges of the component  */
  int64_t n_boundary_edges;                  /* edges used by exactly one triangle                                     */
  int64_t n_nonmanifold_edges;               /* edges used by three or more triangles                                  */
  int64_t first_tri;                         /* smallest triangle index in the component (the numbering key)           */
  double area;                               /* sum of |cross(b-a, c-a)| / 2                                           */
  double volume;                             /* sum of (a-p) . ((b-p) x (c-p)) / 6, p = lo                             */
  double lo[3], hi[3];                       /* bounding box of its vertices                                           */
} ctr_mt3d_component;                        /* 112 bytes */
CTR_API int ctr_mt3d_components(ctr_ctx* ctx, int64_t* n_components);
CTR_API int ctr_mt3d_components_fetch(ctr_ctx* ctx, int32_t* tri_component, ctr_mt3d_component* components);

/* Keeps the components whose keep[c] is non-zero and drops the others, on the LAST 3D run's device mesh as the last
 * ctr_mt3d_components call measured it (engine extension, like VTK's vtkPolyDataConnectivityFilter with specified
 * regions; oracle/mt3d_filter.py:keep_components is the definition).  Synchronous on return.
 *   - keep: host array of n_keep == C bytes, indexed by the component numbers of the last ctr_mt3d_components call.
 *     *n_verts and *n_tris (either may be NULL) receive the new counts; fetch afterwards.
 *   - A triangle stays when its component is kept; kept triangles stay in their order.  A vertex stays when a kept
 *     triangle uses it (also one that a kept and a dropped component share); kept vertices stay in their order and the
 *     ids in the triangles are rewritten.  Positions, normals (CTR_WANT_NORMALS), keys / lowmin (CTR_WANT_KEYS) and the
 *     values of a ctr_mt3d_interpolate made on the current mesh are compacted in place, so _interpolate_fetch stays
 *     row for row with ctr_mt3d_fetch.  Cells and codes stay those of the full scan, as after a selection.
 *   - The component results are updated, not dropped: the kept components are renumbered 0..K-1 in their old order,
 *     tri_component is compacted and relabelled, the table rows are compacted with first_tri the compacted index (still
 *     the component's smallest triangle).  Every other field is carried over: a component is kept whole, so they stay
 *     true.  ctr_mt3d_components_fetch returns the filtered results; calling this again filters further.
 *   - The device buffers are rewritten in place: pointers from ctr_mt3d_device_ptrs and
 *     ctr_mt3d_interpolate_device_ptr stay valid.  The counts published by ctr_mt3d_publish_counts stay those of the
 *     run.
 *   - A seeded selection after this call returns CTR_ERR_STATE; ctr_mt3d_clean, ctr_mt3d_orient_reference,
 *     ctr_mt3d_components and ctr_mt3d_interpolate are accepted.
 *   - CTR_ERR_BAD_ARG: n_keep != C, or keep == NULL with C > 0.  CTR_ERR_STATE: no 3D run, a CTR_NO_GEOMETRY run or no
 *     ctr_mt3d_components since the last run; or the mesh was edited after that call by ctr_mt3d_select_seeded,
 *     ctr_mt3d_clean, ctr_mt3d_smooth or ctr_mt3d_offset_ids (ctr_mt3d_orient_reference only swaps corners inside
 *     triangles: the labels stay valid; after smoothing the areas and volumes are stale, so measure again).  An empty
 *     mesh (C = 0) is a valid no-op; keeping nothing leaves an empty mesh.                                             */
CTR_API int ctr_mt3d_keep_components(ctr_ctx* ctx, const uint8_t* keep, int64_t n_keep, int64_t* n_verts, int64_t* n_tris);

/* Taubin lambda|mu smoothing of the LAST 3D run's device mesh as it stands now (after a selection, clean-up, orientation
 * or component filter too), in place (engine extension, the smoothing step of VTK-style pipelines; the reference's
 * smooth_interpolations is not reproduced -- oracle/mt3d_smooth.py:smooth is the definition).  Synchronous on return.
 *   - An edge is {a, b}, a != b, of some triangle; its uses are the triangle edge slots on it.  A vertex on an edge used
 *     once (boundary) or three or more times (non-manifold), or on no edge, is FIXED: it never moves and keeps its
 *     position bit for bit -- a surface cut by the volume's box stays exactly on the box faces.
 *   - Every free vertex moves towards the average of its distinct edge neighbours (fixed ones included), summed in
 *     ascending id order: x' = x + w * (avg - x), multiply and add rounded apart.  A step is a Jacobi step (all vertices
 *     read the positions from before the step); one iteration is a step with w = lambda, then one with w = mu (skipped
 *     when mu == 0: plain Laplacian smoothing, which shrinks the surface; lambda 0.5 / mu -0.53 does not).  All in fp64
 *     on a copy widened from the geometry type, rounded back once at the end: the positions equal the definition bit for
 *     bit, and with CTR_GEOM_F64 n iterations followed by m equal n + m.
 *   - Normals (CTR_WANT_NORMALS) are recomputed: per vertex the sum of cross(b - a, c - a) over its triangles (fp64, in
 *     an unspecified order: equal to the definition within rounding), normalised, its sign chosen so that it does not
 *     point against the old gradient normal (up the field, whatever the winding); a zero sum keeps the old normal.
 *   - Nothing else changes: triangles, keys / lowmin, cells / codes, the counts, the counts published by
 *     ctr_mt3d_publish_counts and every device pointer handed out before.
 *   - After a call with iterations > 0 on a non-empty mesh: component results of an earlier ctr_mt3d_components are
 *     stale (ctr_mt3d_keep_components returns CTR_ERR_STATE until ctr_mt3d_components measures again); vertex values of
 *     an earlier ctr_mt3d_interpolate are not compacted by a later filter; ctr_mt3d_select_seeded and ctr_mt3d_clean
 *     return CTR_ERR_STATE (the clean-up is defined on the interpolated positions: clean up first).
 *     ctr_mt3d_orient_reference, ctr_mt3d_components, ctr_mt3d_interpolate and further smoothing are accepted; values
 *     interpolated afterwards are still those at each vertex's edge crossing (the keys did not move).
 *   - *out receives n_edges (distinct undirected edges, self-edges of degenerate triangles excluded) and n_fixed_verts,
 *     also for iterations == 0, which writes nothing.
 *   - CTR_ERR_BAD_ARG: a NULL argument, iterations outside [0, 1000], lambda outside (0, 1], mu outside [-1, 0], a NaN
 *     parameter, reserved != 0.  CTR_ERR_STATE: no 3D run or a CTR_NO_GEOMETRY run; a slab run (i_lo != 0 or i_hi != n0)
 *     or vert_id_base != 0; a triangle id outside [0, n_verts) (e.g. after ctr_mt3d_offset_ids), detected before
 *     anything is written.  An empty mesh is a valid no-op.                                                            */
typedef struct {
  int32_t iterations;   /* lambda|mu pairs, 0..1000 (0: nothing is written, the counts are reported) */
  uint32_t reserved;    /* 0 */
  double lambda;        /* (0, 1], e.g. 0.5   */
  double mu;            /* [-1, 0], e.g. -0.53; 0 = Laplacian (mu step skipped) */
} ctr_smooth_params;
typedef struct { int64_t n_edges, n_fixed_verts; } ctr_smooth_counts;
CTR_API int ctr_mt3d_smooth(ctr_ctx* ctx, const ctr_smooth_params* p, ctr_smooth_counts* out);

/* Quadric vertex-clustering decimation of the LAST 3D run's device mesh as it stands now (after a selection, clean-up,
 * orientation, component filter or smoothing too), in place (engine extension: Lindstrom's quadric clustering, as in
 * VTK's vtkQuadricClustering; the reference's flatten is not reproduced -- oracle/mt3d_decimate.py:decimate is the
 * definition).  Synchronous on return.  All arithmetic is fp64 on positions widened from the geometry type, each
 * operation rounded on its own (no fused multiply-add).
 *   - Cluster of a vertex: q[a] = floor((p[a] - origin[a]) / cell[a]) (subtract, then divide), which must lie in
 *     [-2^20, 2^20) on every axis; the cell corner is lo[a] = origin[a] + q[a] * cell[a] (multiply, then add).
 *   - Quadrics: every triangle (a, b, c) of the input, also one that collapses below, has n = cross(P_b - P_a, P_c - P_a)
 *     (unnormalised: the quadric is weighted by area squared).  For each corner, with k its cluster and
 *     d = -(n . (P_a - lo_k)), cluster k gets A_k += n n^T and g_k += d n (a triangle with two corners in k adds twice).
 *   - Position: m_k = mean of (P - lo_k) over the cluster's vertices, lambda_k = 1e-3 * trace(A_k); x = m_k when
 *     lambda_k == 0, else the solution of (A_k + lambda_k I) x = lambda_k m_k - g_k (the minimiser of
 *     sum (n . x + d)^2 + lambda |x - m|^2: exact on flat clusters, keeps a corner or ridge inside a cell, and pulled to
 *     the mean only along directions no plane constrains).  Each axis of x is clamped to [0, cell[a]]; the position is
 *     lo_k + x, rounded to the geometry type once.
 *   - Triangles map to the clusters of their corners.  One with fewer than three distinct clusters is dropped
 *     (n_collapsed); of triangles with the same set of three clusters (either winding) the first in triangle order stays
 *     (n_duplicate: the rules of the clean-up's quantize step).  Kept triangles keep their order and corner order.
 *   - Each cluster a kept triangle uses becomes one vertex.  Clusters are ordered by their smallest member vertex id,
 *     and that member is the cluster's representative: keys / lowmin (CTR_WANT_KEYS) are its rows, so a later
 *     ctr_mt3d_interpolate gives the value at the representative's edge crossing -- a sample of the cluster, not its
 *     average.  Normals (CTR_WANT_NORMALS) are recomputed as ctr_mt3d_smooth does, signed by the representative's old
 *     normal.
 *   - Counts, triangles, vertex order, keys and lowmin are exact; positions and normals equal the definition within
 *     rounding (the sums run in an unspecified order).  Cells and codes stay those of the full scan.
 *   - The device buffers are compacted in place: pointers from ctr_mt3d_device_ptrs stay valid.  The counts published
 *     by ctr_mt3d_publish_counts stay those of the run.
 *   - After a call on a non-empty mesh: component results of an earlier ctr_mt3d_components are stale
 *     (ctr_mt3d_keep_components returns CTR_ERR_STATE until ctr_mt3d_components measures again) and so are vertex values
 *     of an earlier ctr_mt3d_interpolate; ctr_mt3d_select_seeded and ctr_mt3d_clean return CTR_ERR_STATE (the clean-up
 *     is defined on the interpolated positions: clean up first).  ctr_mt3d_orient_reference, ctr_mt3d_components,
 *     ctr_mt3d_interpolate, ctr_mt3d_smooth and further decimation are accepted.
 *   - CTR_ERR_BAD_ARG: a NULL argument; a cell <= 0, NaN or infinite; an origin that is not finite; a cell index out of
 *     range.  CTR_ERR_STATE: no 3D run or a CTR_NO_GEOMETRY run; a slab run (i_lo != 0 or i_hi != n0) or
 *     vert_id_base != 0; a triangle id outside [0, n_verts) (e.g. after ctr_mt3d_offset_ids).  All are detected before
 *     anything is written.  An empty mesh is a valid no-op.                                                             */
typedef struct {
  double cell[3];     /* > 0 and finite: edge lengths of the clustering cells, in the units of the current positions */
  double origin[3];   /* finite: the corner of cell (0, 0, 0)                                                         */
} ctr_decimate_params;                       /* 48 bytes */
typedef struct {
  int64_t n_verts, n_tris;                   /* the decimated mesh                                                    */
  int64_t n_clusters;                        /* occupied cells: cells holding at least one vertex of the input        */
  int64_t n_collapsed;                       /* triangles dropped because two or three corners share a cluster        */
  int64_t n_duplicate;                       /* triangles dropped because an earlier kept triangle has the same three clusters */
} ctr_decimate_counts;                       /* 40 bytes */
CTR_API int ctr_mt3d_decimate(ctr_ctx* ctx, const ctr_decimate_params* p, ctr_decimate_counts* out);

/* Caps that close the LAST 3D run's device mesh at the faces of the volume's box (engine extension: a surface cut by the
 * box otherwise ends there in a rim of boundary edges; oracle/mt3d_cap.py:cap is the definition).  The mesh is
 * extended in place; synchronous on return.
 *   - side CTR_CAP_HIGH closes the region f >= isovalue (the side the triangles and normals face), CTR_CAP_LOW the
 *     region f < isovalue ("low" is the extraction's strict f < isovalue).
 *   - With the Kuhn decomposition each box face square with minimum corner m and in-face axes a < b is cut along its
 *     min -> max diagonal into the face triangles (m, m + e_a, m + e_a + e_b) and (m, m + e_b, m + e_a + e_b).  The cap
 *     is the part of every face triangle on the chosen side: the whole triangle, a corner and its two crossings, or a
 *     quad split by the fan from its first vertex (corners and crossings listed in the face triangle's corner order).
 *     Its rim vertices are the surface's own crossing vertices, found by edge key: the rim is shared exactly.
 *   - Cap triangles face into the box for CTR_CAP_HIGH and out of it for CTR_CAP_LOW (in grid coordinates), so every rim
 *     edge is crossed in opposite directions by its surface and cap triangles.
 *   - New vertices: one per box-surface grid point that some cap triangle uses (the faces share those on box edges and
 *     corners), appended after the existing vertices in ascending key order.  Key lin*8 + 0: d = 0 names the grid
 *     point itself, and ctr_mt3d_interpolate gives exactly the attribute's sample there.  lowmin 1 when the point is
 *     low.  Position grid*delta + origin, rounded per operation in the geometry type as the extraction's.  Normal
 *     (CTR_WANT_NORMALS) the normalised sum of the unit world normals of the cap triangles of the box faces the point
 *     lies on.  Existing vertices keep their rows.
 *   - New triangles are appended after the existing ones, by face (axis 0 lo, axis 0 hi, axis 1 lo, ..., axis 2 hi),
 *     then face square (row-major over (a, b)), then face triangle, then piece.
 *   - A face triangle whose crossing vertex is not in the mesh adds nothing and counts in n_missing: the surface has a
 *     gap there (a tetrahedron skipped by allclose).  Not watertight either: a face sample exactly equal to the
 *     isovalue gives a crossing vertex at ratio 1 that is not merged with the cap's grid vertex at the same position.
 *     Otherwise every edge of the capped mesh is used by exactly two triangles.
 *   - Accepted on the mesh as extracted and after ctr_mt3d_smooth, which keeps the triangles, the keys and the rim's
 *     positions bit for bit: smooth, then cap, gives flat caps.  Also after ctr_mt3d_interpolate and
 *     ctr_mt3d_components, whose results then become stale.
 *   - Afterwards: the published counts, cells and codes stay those of the run; the output buffers may have been
 *     reallocated, so take device pointers (ctr_mt3d_device_ptrs) again.  Component results and vertex values are
 *     stale.  ctr_mt3d_select_seeded and ctr_mt3d_clean return CTR_ERR_STATE; ctr_mt3d_components,
 *     ctr_mt3d_keep_components (after measuring again), ctr_mt3d_smooth (which then rounds the box edges),
 *     ctr_mt3d_decimate, ctr_mt3d_interpolate and ctr_mt3d_orient_reference are accepted.
 *   - CTR_ERR_BAD_ARG: a NULL argument, side not CTR_CAP_HIGH / CTR_CAP_LOW, reserved != 0.  CTR_ERR_STATE: no 3D run or
 *     a CTR_NO_GEOMETRY run; a run without CTR_WANT_KEYS; a slab run (i_lo != 0, i_hi != n0 or plane_offset != 0) or
 *     vert_id_base != 0; a triangle id outside [0, n_verts) (e.g. after ctr_mt3d_offset_ids); a mesh already selected
 *     from, cleaned, filtered, decimated, oriented or capped (the field no longer tells where its rim is or which way it
 *     faces: cap first).  CTR_ERR_OVERFLOW: 2^31 or more vertices or triangles after capping.  All are detected before
 *     anything is written.                                                                                              */
#define CTR_CAP_HIGH 0
#define CTR_CAP_LOW 1
typedef struct {
  int32_t side;       /* CTR_CAP_HIGH or CTR_CAP_LOW */
  uint32_t reserved;  /* 0 */
} ctr_cap_params;                            /* 8 bytes */
typedef struct {
  int64_t n_verts, n_tris;                   /* the capped mesh                                                       */
  int64_t n_cap_verts, n_cap_tris;           /* added by the caps                                                     */
  int64_t n_missing;                         /* face triangles left open because a crossing vertex is not in the mesh */
} ctr_cap_counts;                            /* 40 bytes */
CTR_API int ctr_mt3d_cap(ctr_ctx* ctx, const ctr_cap_params* p, ctr_cap_counts* out);

/* Seeded extraction (SURVEY.md 8(f3)): restricts the LAST full-volume run's mesh to what the reference's tracker
 *   tetrahedral.py:443-469  expand_voxels / in_range  (flood fill over the 26-neighbourhood of border voxels)
 * reaches from the given start voxels (the output of find_initial_voxels, tetrahedral.py:396-441, which the binding
 * evaluates on the host: a few samples per seed segment).  seed_voxels [n_seeds][3] voxel origins (i, j, k); origins
 * outside [0, n-2] are ignored (the reference's out-of-range "leak" voxels).  Triangles, vertices, normals and keys
 * are compacted in place (order kept, ids renumbered); case codes / cells stay those of the full scan.  Returns the
 * new counts and the number of emitting voxels selected; fetch afterwards.  With CTR_FIELD_ON_DEVICE the field must
 * still be resident.  ONE-SHOT: the run's mesh is rewritten, so a second call on the same run (or a call after
 * ctr_mt3d_clean, ctr_mt3d_keep_components or ctr_mt3d_smooth) returns CTR_ERR_STATE until the next ctr_mt3d_run.  */
CTR_API int ctr_mt3d_select_seeded(ctr_ctx* ctx, const int32_t* seed_voxels, int64_t n_seeds, int64_t* n_verts,
                                   int64_t* n_tris, int64_t* n_voxels);

/* Per-vertex values of another field (engine extension; the reference has none -- oracle/mt3d_values.py:vertex_values
 * is the definition): every vertex of the LAST 3D run, as its mesh stands now (after ctr_mt3d_select_seeded / ctr_mt3d_clean
 * too) and in the order ctr_mt3d_fetch returns it, gets
 *   value[id][c] = a_low[c] + ratio * (a_high[c] - a_low[c])      (IEEE multiply, then add; no fused multiply-add)
 * where low / high are the ends of the vertex's edge as its `lowmin` orders them, a = the attribute field's samples
 * widened to the run's geometry type, and ratio is the one the vertex's position was made with (the run's samples and
 * isovalue in the geometry type; 0.5 where |f_high - f_low| <= 1e-8; __fdividef in fp32 mode).  The world transform is
 * not applied to values.  In grid coordinates the field of point coordinates (component c = index along axis c, axis 0
 * global) gives the vertex positions bit for bit.
 * The pass is driven by the device keys: the run must have used CTR_WANT_KEYS (else CTR_ERR_STATE, as for no 3D run or
 * a CTR_NO_GEOMETRY run).  The run's field must still be valid when it was on the device.  The pass does not edit the
 * mesh and may be called any number of times per run, with different fields; values computed before a selection or
 * clean-up are NOT compacted with the mesh (interpolate after the last edit).  A host field is staged in a buffer of
 * its own (the run's staged samples stay).  Synchronous on return.
 *   _interpolate      : *n_verts (may be NULL) receives the number of vertices = rows of values
 *   _interpolate_fetch: values [n_verts][ncomp] in the run's geometry type (float / double with CTR_GEOM_F64)
 *   _interpolate_device_ptr: the same array on the device, valid until the next run or interpolation on this context */
typedef struct {
  const void* field;   /* the run's grid, component-last: [n0][n1][n2][ncomp], host or device (CTR_FIELD_ON_DEVICE);
                          n0..n2 those of the run's array (a slab's planes for a slab run)                          */
  int32_t dtype;       /* any ctr_dtype (F32, F64, U8, I16, U16), independent of the run's dtype                     */
  uint32_t flags;      /* CTR_FIELD_ON_DEVICE                                                                         */
  int32_t ncomp;       /* 1..4                                                                                        */
  int32_t reserved;
} ctr_attr_params;
CTR_API int ctr_mt3d_interpolate(ctr_ctx* ctx, const ctr_attr_params* p, int64_t* n_verts);
CTR_API int ctr_mt3d_interpolate_fetch(ctr_ctx* ctx, void* values);
CTR_API int ctr_mt3d_interpolate_device_ptr(ctr_ctx* ctx, void** values);

/* ---- multi-GPU: one process per GPU, z-slabs (SURVEY.md 8(e)) -----------------------------------------------------
 * Every rank runs ctr_mt3d_run on its slab (i_lo / i_hi / plane_offset) independently; NCCL carries only the counts and,
 * optionally, the mesh.  NCCL is bound at run time (the libnccl.so.2 already in the process, else the loader path).
 *   ctr_comm_unique_id    : rank 0 makes the 128-byte id (ncclGetUniqueId); the host distributes it by any means
 *   ctr_comm_init         : ncclCommInitRank on the context's device; from then on every 3D run of the context
 *                           publishes {n_verts, n_tris} on the device (as ctr_mt3d_publish_counts does)
 *   ctr_allgather_offsets : ncclAllGather of those device counts on the context's stream (no host round trip before the
 *                           collective) -> counts[nranks][2] (may be NULL), this rank's exclusive offsets [2], totals [2]
 *   ctr_gather_mesh       : after ctr_allgather_offsets: positions, normals (if computed) and triangles of every rank to
 *                           `root` by grouped ncclSend / ncclRecv of exactly the bytes each rank has; triangle ids are
 *                           made global on the root (local id + the rank's vertex offset).  Collective: every rank calls it.
 *   ctr_gathered_fetch    : root only: copy the gathered mesh to host buffers of total_verts x 3 (geometry type of the
 *                           runs) and total_tris x 3 int32.                                                          */
CTR_API int ctr_comm_unique_id(void* id128);
CTR_API int ctr_comm_init(ctr_ctx* ctx, const void* id128, int rank, int nranks);
CTR_API int ctr_comm_destroy(ctr_ctx* ctx);
CTR_API int ctr_allgather_offsets(ctr_ctx* ctx, int64_t* counts, int64_t* my_offsets, int64_t* totals);
CTR_API int ctr_gather_mesh(ctr_ctx* ctx, int root, int64_t* total_verts, int64_t* total_tris);
CTR_API int ctr_gathered_fetch(ctr_ctx* ctx, void* verts, void* normals, int32_t* tris);

/* The reference's mesh post-processing (SURVEY.md 8 a10 / a11 / a13, f1) on the device mesh of the LAST ctr_mt3d_run:
 *   tetrahedral.py:190-215     quantize_interpolations(divisions)   vertices in one cell of the divisions grid merge
 *   tetrahedral.py:353-375     remove_tiny_simplices(epsilon)       tiny simplices collapse to a point and go
 *   surface_geometry.py:14-50  clean_triangles                      zero-area triangles go, their coincident vertices merge
 *   surface_geometry.py:52-140 orient_triangles (CTR_CLEAN_ORIENT)  = ctr_mt3d_orient_reference, in grid coordinates
 *   grid_field.py:89-93        from_grid_coordinates                x * delta + origin, applied last (tetrahedral.py:86-90)
 * which is what GridContour3d.get_points_and_triangles(clean=True) returns (tetrahedral.py:541-552).  The run must have
 * been made in GRID coordinates (origin 0, delta 1), over the full volume, with vert_id_base 0.  Where the reference's
 * result depends on CPython dict / set order the vertex of smallest id survives (oracle/post3d.py states the rules).
 * Vertices, normals, keys and triangles are compacted in place (order kept); fetch afterwards.  One-shot per run, and
 * not after ctr_mt3d_smooth (CTR_ERR_STATE: quantizing and the tiny-simplex test are defined on interpolated
 * positions; clean up first, then smooth).                                                                           */
#define CTR_CLEAN_ORIENT 1u        /* run the orientation pass before the transform                         */
#define CTR_CLEAN_NO_TRIANGLES 2u  /* skip clean_triangles (get_points_and_triangles(clean=False))          */
typedef struct {
  int64_t corner[3];       /* grid dimensions N (voxels per axis) = n - 1: self.corner of the reference            */
  int32_t divisions;       /* 10000 in the reference; < 2^21                                                        */
  uint32_t flags;          /* CTR_CLEAN_ORIENT, CTR_CLEAN_NO_TRIANGLES                                              */
  double epsilon;          /* 1e-4 in the reference                                                                 */
  double origin[3], delta[3];
} ctr_clean_params;
typedef struct {
  int64_t n_verts, n_tris;           /* final mesh                                                                  */
  int64_t n_quantized, n_tiny, n_flat;   /* triangles removed by each pass                                          */
  int64_t n_components, n_flipped;   /* of the orientation pass (CTR_CLEAN_ORIENT)                                  */
} ctr_clean_counts;
CTR_API int ctr_mt3d_clean(ctr_ctx* ctx, const ctr_clean_params* params, ctr_clean_counts* out);

/* ---- 2D marching triangles, all levels in one pass ------------------------------------------------
 * Replaces, for an array-backed field, the reference's
 *   multiple_2d_contour.py:63-75 + :50-61  search_grid_for_crossings / classify_endpoint_values
 *   triangulated.py:198-213,307-378        search_grid / find_initial_contour_pairs / expand_contour_pairs /
 *                                          find_all_adjacent_contour_pairs / contour_pair_interpolation
 *   triangulated.py:66-77,295-305          adjacent_pairs / find_adjacencies   (segments = linked key pairs)
 *   multiple_2d_contour.py:100-108         Linear2DContour.get_values          (fmin / fmax)
 * field[i][j], points in range are 0 <= i < n0, 0 <= j < n1 (no extra sample, unlike 3D/4D).
 * Edge key = ((lin(min endpoint)*4 + d) << 1) | lowmin, d = di*2 + dj in {1,2,3}; the reference's key (p, q) has
 * lowmin = 1, (q, p) has lowmin = 0 (both exist when f(p) == f(q) == level).                        */
typedef struct {
  const void* field;
  int32_t dtype;        /* CTR_F32 or CTR_F64 */
  uint32_t flags;          /* CTR_FIELD_ON_DEVICE, CTR_GEOM_F64, CTR_NO_GEOMETRY, CTR_WANT_MINMAX            */
  int64_t n0, n1;
  const double* levels;    /* host array, strictly increasing                                                */
  int32_t nlevels;         /* 1..64                                                                          */
  int32_t reserved;
  double origin[2], delta[2];
  int64_t i_lo, i_hi, row_offset;   /* row-band sharding: squares of rows [i_lo, i_hi); single GPU 0, n0, 0    */
} ctr_mt2d_params;

typedef struct {
  int64_t n_segments;
  int64_t n_active_squares;
  double fmin, fmax;
} ctr_mt2d_counts;

CTR_API int ctr_mt2d_run(ctr_ctx* ctx, const ctr_mt2d_params* p, ctr_mt2d_counts* out);
/* seg_level [n_segments] index into levels; seg_keys [n_segments][2]; seg_pos [n_segments][2][2] float|double
 * (world coordinates of the two end points).  Order: by square, triangle, level.                          */
CTR_API int ctr_mt2d_fetch(ctr_ctx* ctx, uint8_t* seg_level, uint64_t* seg_keys, void* seg_pos);

/* Polylines of the LAST ctr_mt2d_run, on the device (SURVEY.md 8 a23 / f4).  Replaces
 *   triangulated.py:221-305  find_adjacencies / get_contour_sequences (the per-vertex chaining of contour pairs)
 *   triangulated.py:269      consecutive np.allclose points dropped
 * by list ranking over the segments' darts (pointer jumping).  Open contours start at their smaller end key, closed ones
 * at their smallest key towards the smaller neighbour (the reference's order follows CPython set iteration).  A level
 * in which some key lies on more than two segments (a sample exactly on the level) is reported in junction_levels and
 * nothing is chained: there the order of visits decides and the binding's fixed-order walk is the definition.
 * _fetch: per polyline its level index, closed flag (bit 0: a cycle of segments, bit 1: an open chain whose ends are
 * np.allclose), start key, first point and number of points; points [n_points][2]
 * in the run's geometry type.  Polylines come in no particular order (sort by level / closed / start key).           */
typedef struct {
  int64_t n_polylines, n_points;
  uint64_t junction_levels;      /* bit l set: level l has a key with more than two segments; nothing was chained     */
} ctr_poly_counts;
CTR_API int ctr_mt2d_polylines(ctr_ctx* ctx, ctr_poly_counts* out);
CTR_API int ctr_mt2d_polylines_fetch(ctr_ctx* ctx, int32_t* level, uint8_t* closed, uint64_t* start_key, uint32_t* offset,
                                     uint32_t* length, void* points);

/* ---- 4D marching pentatopes + morph triangles ---------------------------------------------------
 * Replaces, for an array-backed field f[i][j][k][l] (l = time, contiguous), the reference's
 *   pentatopes.py:101-106,216-291   find_tetrahedra (flood fill -> full scan), enumerate_voxel_tetrahedra,
 *                                   enumerate_pentatope_tetrahedra (24 Kuhn pentatopes, 1 or 3 tetrahedra each)
 *   tetrahedral.py:471-512          contour_pair_interpolation in 4D (keys, positions)
 * and, with CTR_MORPH (always in grid coordinates, fp64),
 *   pentatopes.py:162-169           bin_times(nbins)
 *   pentatopes.py:171-189           drop_instant_tetrahedra(1e-7)
 *   tetrahedral.py:353-375          remove_tiny_simplices(1e-3): the predicate (vertex merging: DESIGN.md)
 *   morph_geometry.py:145-237       triangulate_tetrahedron_at_midpoints / add_tetrahedron / interpolate_pair_3d
 *   pentatopes.py:336-348           removal of triangles with a zero-duration segment                    */
typedef struct {
  const void* field;
  int32_t dtype;        /* CTR_F32 or CTR_F64 */
  uint32_t flags;
  int64_t n0, n1, n2, n3;
  double isovalue;
  double origin[4], delta[4];
  int32_t nbins;            /* bin_times: 100 in the reference */
  int32_t reserved;
} ctr_mp4d_params;

typedef struct {
  int64_t n_verts, n_tets, n_active_cells, n_crossings, n_codes, n_morph_tris;
  double fmin, fmax;
  double t_min, t_max;      /* t range of the binned vertices (grid units); NaN without CTR_MORPH          */
} ctr_mp4d_counts;

CTR_API int ctr_mp4d_run(ctr_ctx* ctx, const ctr_mp4d_params* p, ctr_mp4d_counts* out);
/* verts [n_verts][4] float|double world coords; tets [n_tets][4] vertex ids; keys/lowmin [n_verts];
 * codes [n_codes][24] per-pentatope case codes (5-bit low mask | 32 if skipped) and cells [n_codes] packed
 * (word << 22 | bit << 17 | ...) hypervoxel ids of the emitting hypervoxels;
 * morph_verts [n_verts][4] fp64 grid coordinates after bin_times; keep [n_tets] 0/1 after the instant / tiny filter;
 * morph_tris [n_morph_tris][3][2]: three segments (low-t vertex id, high-t vertex id) per morph triangle,
 * duplicates not removed.                                                                                */
CTR_API int ctr_mp4d_fetch(ctr_ctx* ctx, void* verts, int32_t* tets, uint64_t* keys, uint8_t* lowmin, uint8_t* codes,
                           int64_t* cells, double* morph_verts, uint8_t* keep, int32_t* morph_tris);

/* ---- wire formats (SURVEY.md 8(f2)): the text the reference's emitters build with Python joins, by host threads
 *   html_demo.py:118-161       grid_html_page ("[[x, y, z],\n    [..]]"), emit_three_json ("[0,\ni,\nj,\nk,\n0,.."], flat vertices)
 *   morph_geometry.py:91-128   MorphTriangles.to_json / flatten_json_list ("[a,b,c,d,\ne,f,g,h]")
 * data [rows][cols] -> "[" row (row_sep row)* "]",  row = row_prefix value (col_sep value)* row_suffix.
 * Values are formatted exactly like Python's str(): integers in decimal; floats as repr(float) (shortest round-trip
 * digits, "1e-05" / "0.0001" / "1000000000000000.0" / "1e+16", float32 widened first like float(np.float32(x))).
 * *out is malloc'ed, NUL-terminated, *out_len bytes without the NUL; release with ctr_wire_free.  Host-only: needs no
 * context and no device.  n_threads <= 0 = all hardware threads.                                                    */
typedef enum { CTR_WIRE_I32 = 0, CTR_WIRE_I64 = 1, CTR_WIRE_U32 = 2, CTR_WIRE_F32 = 3, CTR_WIRE_F64 = 4 } ctr_wire_dtype;
CTR_API int ctr_wire_format(const void* data, int dtype, int64_t rows, int64_t cols, const char* row_prefix,
                            const char* col_sep, const char* row_suffix, const char* row_sep, int n_threads, char** out,
                            int64_t* out_len);
CTR_API void ctr_wire_free(char* p);

#ifdef __cplusplus
}
#endif
#endif
