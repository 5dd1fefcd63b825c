// Shared plumbing of the engine: context, grow-only device buffers, error handling, warp helpers,
// decoupled-lookback tile status.  Host language above this is Python (ctypes), see engine.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <utility>
#include <vector>

#include "../../include/contourist_b200.h"

#define CTR_NSTAGE 8

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct ctr_comm_state;                    // comm.cu: NCCL communicator + gathered mesh of a context

// The 3D slots of ctr_ctx::aux (the 2D and 4D paths number theirs in their own translation units).
enum Aux3 : int {
  // the extraction's work lists and flags, rewritten by every ctr_mt3d_run; the seeded selection reads them
  AUX_OWN_LIST = 0,          // (owner id, vertex offset) per active owner
  AUX_CELL_LIST = 2,         // id of every emitting voxel
  AUX_ROW_FLAGS = 4,         // per voxel row: some sample near the isovalue
  AUX_WORD_FLAGS = 32,       // per word: near flags
  AUX_WORD_RECS = 33,        // records of the listed interesting words
  AUX_TILE_WORDS = 34,       // (first entry, entries) of the word list per tile
  AUX_EXACT_FLAGS = 35,      // per word: "exact test differs" flags
  AUX_WORD_SLOTS = 41,       // first work-list slots of the listed words
  // scratch of the mesh passes: any pass may overwrite them
  AUX_SCRATCH0 = 27,
  AUX_SCRATCH1 = 28,
  AUX_SCRATCH2 = 29,
  AUX_SCRATCH3 = 30,
  AUX_SCRATCH4 = 31,
  AUX_ATTR_FIELD = 42,       // ctr_mt3d_interpolate's staged host field
  AUX_SMOOTH_X0 = 46,        // smoothing's two fp64 working copies
  AUX_SMOOTH_X1 = 47,
  // results that outlive the pass that made them: no pass uses them as scratch
  AUX_VALUES = 43,           // vertex values (ctr_mt3d_interpolate)
  AUX_LABELS = 44,           // component of every triangle (ctr_mt3d_components)
  AUX_COMPONENTS = 45,       // component table
  AUX_SECTION_SEGS = 1,      // plane sections (ctr_mt3d_section): segments and junction planes
  AUX_SECTION_POLYS = 3,     // ... polylines, their points and measures
  AUX_CLOSEST_RESULT = 48,   // closest points (ctr_mt3d_closest): distance, triangle, point per query point
  AUX_CLOSEST_TREE = 49,     // ... the tree of the last call (rebuilt by every call)
  AUX_CLOSEST_POINTS = 50,   // ... its host query points, staged
  AUX_RAY_RESULT = 51,       // ray casting (ctr_mt3d_raycast): t, weights, point, triangle, side per ray (its tree is
  AUX_RAY_INPUT = 52,        // ... its host rays, staged                      AUX_CLOSEST_TREE, rebuilt by every call)
};

// ctr_ctx::last3_edited: the passes that have rewritten the device mesh of the last 3D run
enum Edit3 : unsigned {
  EDIT_SELECT = 1u,          // seeded selection
  EDIT_CLEAN = 2u,           // clean-up
  EDIT_KEEP = 4u,            // component filter
  EDIT_SMOOTH = 8u,          // smoothing
  EDIT_DECIMATE = 16u,       // decimation
  EDIT_CAP = 32u,            // caps at the box faces
  EDIT_ORIENT = 64u,         // reference orientation (rewinds triangles only: the mesh generation stays)
  EDIT_CLIP = 128u,          // clipping by a plane or a vertex value
};

// What a pass on the device mesh of the last 3D run needs of that run, and which earlier passes refuse it: one row per
// pass, checked by check_pass.  Every pass needs a completed run with geometry (CTR_ERR_STATE).
// Slab conditions, each including the one before: i_lo == 0 and i_hi == n0; vert_id_base == 0; plane_offset == 0.
enum Slab3 : int { ANY_RUN, FULL, FULL_ID0, FULL_ID0_PLANE0 };

struct PassRule {
  const char* verb;          // ends "no completed ctr_mt3d_run with geometry<verb>"
  bool keys;                 // needs the run's CTR_WANT_KEYS outputs
  Slab3 slab;
  int slab_code;             // the error of a run that misses the slab condition
  const char* slab_msg;
  unsigned refused_after;    // Edit3 bits of the passes that must not have run before this one
  const char* order_msg;     // what to do instead, after the list of those passes
};

constexpr PassRule PASS_ORIENT = {" to orient", false, ANY_RUN, 0, nullptr, 0u, nullptr};
constexpr PassRule PASS_COMPONENTS = {" to measure", false, FULL_ID0, CTR_ERR_STATE,
                                      "components need a full-volume run with vert_id_base 0 (components cross slab faces)", 0u, nullptr};
constexpr PassRule PASS_SMOOTH = {" to smooth", false, FULL_ID0, CTR_ERR_STATE,
                                  "smoothing needs a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)", 0u, nullptr};
constexpr PassRule PASS_SECTION = {" to cut", false, FULL_ID0, CTR_ERR_STATE,
                                   "sections need a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)", 0u, nullptr};
constexpr PassRule PASS_DECIMATE = {" to decimate", false, FULL_ID0, CTR_ERR_STATE,
                                    "decimation needs a full-volume run with vert_id_base 0 (clusters cross slab faces)", 0u, nullptr};
// the selection compacts the run's mesh in place while the voxel work list keeps its per-voxel triangle offsets: it can
// be applied once per run, and before any other edit (an oriented mesh has the same rows)
constexpr PassRule PASS_SELECT = {" to select from", false, FULL, CTR_ERR_UNSUPPORTED,
                                  "seeded selection needs a full-volume run (components cross slab faces)",
                                  EDIT_SELECT | EDIT_CLEAN | EDIT_KEEP | EDIT_SMOOTH | EDIT_DECIMATE | EDIT_CAP | EDIT_CLIP,
                                  "run ctr_mt3d_run again"};
// the reference's clean-up (quantize, tiny simplices) is defined on the interpolated positions
constexpr PassRule PASS_CLEAN = {" to clean", false, FULL_ID0, CTR_ERR_UNSUPPORTED,
                                 "mesh clean-up needs a full-volume run (merges cross slab faces)",
                                 EDIT_CLEAN | EDIT_SMOOTH | EDIT_DECIMATE | EDIT_CAP | EDIT_CLIP,
                                 "clean it up once, before smoothing, decimating, capping or clipping"};
// after these passes the field no longer tells where the mesh's rim is or which way it faces
constexpr PassRule PASS_CAP = {" to cap", true, FULL_ID0_PLANE0, CTR_ERR_STATE,
                               "caps need a full-volume run with plane_offset 0 and vert_id_base 0 (the box of a slab is not the volume's)",
                               EDIT_SELECT | EDIT_CLEAN | EDIT_KEEP | EDIT_DECIMATE | EDIT_CAP | EDIT_ORIENT | EDIT_CLIP,
                               "cap it before those passes"};
// the clip keeps the part of the mesh on one side: any earlier pass, an earlier clip too (six clips make a box)
constexpr PassRule PASS_CLIP = {" to clip", false, FULL_ID0, CTR_ERR_STATE,
                                "clipping needs a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)", 0u, nullptr};
// the closest-point query reads the mesh as it stands after any pass
constexpr PassRule PASS_CLOSEST = {" to query", false, FULL_ID0, CTR_ERR_STATE,
                                   "closest points need a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)",
                                   0u, nullptr};
// the ray cast reads the mesh as it stands after any pass
constexpr PassRule PASS_RAYCAST = {" to cast rays at", false, FULL_ID0, CTR_ERR_STATE,
                                   "ray casting needs a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)",
                                   0u, nullptr};
constexpr PassRule PASS_INTERPOLATE = {" to interpolate on", true, ANY_RUN, 0, nullptr, 0u, nullptr};
constexpr PassRule PASS_OFFSET_IDS = {"", false, ANY_RUN, 0, nullptr, 0u, nullptr};

struct ctr_ctx {
  int device = 0;
  ctr_comm_state* comm = nullptr;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t ev_enqueued = nullptr;   // recorded behind everything ctr_mt3d_enqueue queued: ctr_mt3d_finish waits for it,
                                       // not for the stream (work queued later, e.g. a collective, is not its business)
  cudaEvent_t ev_tail = nullptr;       // ctr_wait_for(other context, this): marks this stream's tail for the other stream
  std::string err;
  int64_t launches = 0;
  bool timing = false;
  cudaEvent_t ev[CTR_NSTAGE + 1] = {};
  bool ev_set[CTR_NSTAGE + 1] = {};
  float stage_ms[CTR_NSTAGE] = {};
  int sm_count = 148;
  std::vector<const void*> smem_optin;   // kernels ctr_smem_optin has set up on this context's device

  // staging + shared scratch
  DevBuf field;              // device copy of a host field
  DevBuf bits, nbits;        // bitplanes: low (f < v) and near (conservative allclose hull)
  DevBuf vbase, tbase;       // per-word exclusive offsets (uint32)
  DevBuf list_v, list_t;     // compacted active word lists (uint32 word index)
  DevBuf tile_state;         // decoupled-lookback status words
  DevBuf counters;           // small block of device counters (see each path)
  DevBuf wmask;              // 3D: per-word (active-owner, emitting-voxel) masks
  DevBuf wdir;               // 3D: per-word direction prefix (dirpack) of the vertex numbering
  DevBuf vox_tab;            // 3D: corner bits -> triangle list of a voxel (256 x 12 words)
  void* counters_host = nullptr;  // pinned mirror

  // outputs (3D)
  DevBuf verts, normals, tris, keys, lowmin, cells, codes;
  // last-run descriptors
  int last_kind = 0;         // 0 none, 3 = mt3d, 2 = mt2d, 4 = mp4d
  uint32_t last_flags = 0;
  int64_t last_counts[8] = {};
  int64_t poly_counts[2] = {};            // 2D: polylines / points of the last ctr_mt2d_polylines
  unsigned char last3_params[160] = {};   // parameters of the last completed ctr_mt3d_run
  long long* publish3 = nullptr;          // ctr_mt3d_publish_counts: device {n_verts, n_tris} behind every 3D run
  unsigned last3_edited = 0;              // Edit3 bits of the passes that have rewritten the device mesh of that run
  // bumped by every 3D run and by mesh_edited (every pass that writes the mesh, orientation aside); the vertex values
  // and the components below record the generation they were computed on
  uint64_t mesh_gen = 0;
  // 3D: an extraction enqueued by ctr_mt3d_enqueue and not yet finished
  bool pending3 = false;
  alignas(8) unsigned char pending3_params[160] = {};
  // 3D: capacities of the output pools / work lists kept from earlier runs, last list lengths, launch coverage
  size_t spec_v = 0, spec_t = 0, spec_own = 0, spec_cell = 0, last_own = 0, last_cell = 0, cover_own = 0, cover_cell = 0;
  size_t spec_w = 0, last_w = 0, cover_w = 0;   // interesting-word list of the split stage 2
  DevBuf wlist;
  // 3D vertex values (ctr_mt3d_interpolate): rows and components of AUX_VALUES; 0 = none since the last 3D run
  size_t attr_rows = 0;
  int attr_ncomp = 0;
  uint64_t attr_gen = 0;
  // 3D connected components (ctr_mt3d_components): triangles and components of AUX_LABELS / AUX_COMPONENTS; -1 = none
  // since the last 3D run
  int64_t comp_tris = 0, comp_count = -1;
  uint64_t comp_gen = 0;
  // 3D plane sections (ctr_mt3d_section) in AUX_SECTION_SEGS / AUX_SECTION_POLYS: segments (-1 = none since the last 3D
  // run), polylines, points, junction planes; and the number of planes
  int64_t sect_count[4] = {-1, 0, 0, 0};
  int32_t sect_nplanes = 0;
  // 3D closest points (ctr_mt3d_closest) in AUX_CLOSEST_RESULT: query points of the last successful call; -1 = none since
  // the last 3D run (or the last call failed)
  int64_t closest_n = -1;
  // 3D ray casting (ctr_mt3d_raycast) in AUX_RAY_RESULT: rays of the last successful call; -1 = none since the last 3D run
  // (or the last call failed)
  int64_t ray_n = -1;

  // extra outputs and scratch in generic slots: 3D (Aux3 above); 5-10: 2D; 12-26: 4D; 36-40: 2D polylines
  DevBuf aux[53];
};

static inline int ctr_fail(ctr_ctx* ctx, int code, const char* what, const char* detail = "") {
  if (ctx) {
    ctx->err = std::string(what) + (detail && detail[0] ? ": " : "") + (detail ? detail : "");
  }
  return code;
}

#define CTR_CUDA(ctx, call)                                                                   \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      char b__[256];                                                                          \
      snprintf(b__, sizeof b__, "%s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__);  \
      return ctr_fail(ctx, e__ == cudaErrorMemoryAllocation ? CTR_ERR_OOM : CTR_ERR_CUDA,     \
                      "CUDA error", b__);                                                     \
    }                                                                                         \
  } while (0)

// grow-only allocation with 25% head-room so repeated runs of similar size never reallocate
static inline int ctr_ensure(ctr_ctx* ctx, DevBuf& b, size_t bytes, bool exact = false) {
  if (bytes <= b.cap && b.p) return 0;
  if (b.p) {
    cudaStreamSynchronize(ctx->stream);
    cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = exact ? bytes : bytes + bytes / 4;
  if (want < 256) want = 256;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess && want != bytes) {
    want = bytes < 256 ? 256 : bytes;
    e = cudaMalloc(&b.p, want);
  }
  if (e != cudaSuccess) {
    b.p = nullptr;
    cudaGetLastError();
    char m[128];
    snprintf(m, sizeof m, "cudaMalloc of %zu bytes failed", want);
    return ctr_fail(ctx, CTR_ERR_OOM, m);
  }
  b.cap = want;
  return 0;
}

// ctr_ensure for a buffer whose first `keep` bytes must survive: a larger buffer is allocated, the content copied over
// on the device and the old buffer freed.  The buffer's address changes when it grows.
static inline int ctr_grow_keep(ctr_ctx* ctx, DevBuf& b, size_t bytes, size_t keep) {
  if (bytes <= b.cap && b.p) return 0;
  DevBuf n;
  if (int rc = ctr_ensure(ctx, n, bytes)) return rc;
  cudaError_t e = keep ? cudaMemcpyAsync(n.p, b.p, keep, cudaMemcpyDeviceToDevice, ctx->stream) : cudaSuccess;
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    cudaFree(n.p);
    CTR_CUDA(ctx, e);
  }
  cudaFree(b.p);
  b = n;
  return 0;
}

// 256-byte-aligned pieces of one DevBuf.  `pieces` names each piece once, as carve(pointer, bytes); ctr_carve_buf calls
// it twice: to add up the size (the pointers stay null), then, after ctr_ensure, to point every piece into the buffer.
struct ctr_carve {
  char* base = nullptr;
  size_t off = 0;
  template <typename P>
  void operator()(P*& p, size_t bytes) {
    p = base ? reinterpret_cast<P*>(base + off) : nullptr;
    off += (bytes + 255) & ~(size_t)255;
  }
};

template <typename F>
static inline int ctr_carve_buf(ctr_ctx* ctx, DevBuf& b, F&& pieces) {
  ctr_carve c;
  pieces(c);
  if (int rc = ctr_ensure(ctx, b, c.off)) return rc;
  c = ctr_carve{(char*)b.p, 0};
  pieces(c);
  return 0;
}

// 0 when the last 3D run and the passes since allow the pass of row `r`, and the context's device is then current; else
// the error, with the message set
static inline int check_pass(ctr_ctx* ctx, const PassRule& r) {
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, (std::string("no completed ctr_mt3d_run with geometry") + r.verb).c_str());
  if (r.keys && !(ctx->last_flags & CTR_WANT_KEYS))
    return ctr_fail(ctx, CTR_ERR_STATE, "the run did not keep its keys: run with CTR_WANT_KEYS");
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  if ((r.slab >= FULL && (p->i_lo != 0 || p->i_hi != p->n0)) || (r.slab >= FULL_ID0 && p->vert_id_base != 0) ||
      (r.slab >= FULL_ID0_PLANE0 && p->plane_offset != 0))
    return ctr_fail(ctx, r.slab_code, r.slab_msg);
  if (const unsigned done = ctx->last3_edited & r.refused_after) {
    static const char* const names[] = {"selected from", "cleaned", "filtered", "smoothed", "decimated", "capped", "oriented",
                                              "clipped"};
    std::string list;
    for (int b = 0; b < 8; ++b)
      if (done & (1u << b)) list += std::string(list.empty() ? "" : ", ") + names[b];
    return ctr_fail(ctx, CTR_ERR_STATE, ("the mesh of this run has been " + list).c_str(), r.order_msg);
  }
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  return 0;
}

// A pass is about to write the device mesh of the last 3D run (a mesh buffer or its counts): results recorded against
// the mesh generation (components, vertex values) no longer describe it, and check_pass refuses the passes that must
// come before `edit` (0: a change no pass refuses, such as ctr_mt3d_offset_ids).
static inline void mesh_edited(ctr_ctx* ctx, unsigned edit) {
  ctx->mesh_gen++;
  ctx->last3_edited |= edit;
}

// f(T{}) for the sample type T of `dtype`
template <typename F>
static inline int with_sample_type(ctr_ctx* ctx, int dtype, F&& f) {
  switch (dtype) {
    case CTR_F32: return f(float{});
    case CTR_F64: return f(double{});
    case CTR_U8: return f(uint8_t{});
    case CTR_I16: return f(int16_t{});
    case CTR_U16: return f(uint16_t{});
  }
  return ctr_fail(ctx, CTR_ERR_BAD_ARG, "unknown dtype");
}

// f(G{}) for the geometry type G of the last run (double with CTR_GEOM_F64, else float)
template <typename F>
static inline int with_geom_type(ctr_ctx* ctx, F&& f) {
  if (ctx->last_flags & CTR_GEOM_F64) return f(double{});
  return f(float{});
}

static inline void ctr_stage_mark(ctr_ctx* ctx, int idx) {
  if (!ctx->timing) return;
  if (!ctx->ev[idx]) cudaEventCreate(&ctx->ev[idx]);
  cudaEventRecord(ctx->ev[idx], ctx->stream);
  ctx->ev_set[idx] = true;
}

// ------------------------------------------------------------------------------------------ device
#ifdef __CUDACC__

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }

struct Xform {
  double origin[3], delta[3], inv_delta[3];
};

// geometry-mode arithmetic: IEEE in fp64 mode (positions bit-exact vs the oracle); fast approximations in fp32 mode (1e-4 rel)
__device__ __forceinline__ double quot(double a, double b) { return a / b; }
__device__ __forceinline__ float quot(float a, float b) { return __fdividef(a, b); }
__device__ __forceinline__ double inv_sqrt(double a) { return 1.0 / sqrt(a); }
__device__ __forceinline__ float inv_sqrt(float a) { return rsqrtf(a); }

// Programmatic dependent launch.  The kernels of one extraction run back to back on one stream, several of them for a
// few microseconds only; launched with ctr_launch_dep a kernel's blocks may become resident (and run their prologue:
// shared-memory tables, mbarrier set-up) while the previous kernel drains.  Rules that keep this equal to plain stream
// order: (1) ctr_pdl_wait() -- returns when every earlier kernel has completed and its writes are visible -- precedes
// the first access to anything an earlier kernel of the stream writes or reads; (2) ctr_pdl_trigger() comes after the
// wait, so a kernel that has started implies that everything in front of its predecessor is complete.
#ifndef CTR_PDL
#define CTR_PDL 1
#endif
__device__ __forceinline__ void ctr_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void ctr_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void ctr_pdl_enter() {
  ctr_pdl_wait();
  ctr_pdl_trigger();
}

template <typename... KArgs, typename... Args>
static inline cudaError_t ctr_launch_dep(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = CTR_PDL;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// Lets `kernel` take `bytes` of dynamic shared memory (above the default 48 KiB), the first time this context launches
// it.  The attribute belongs to the device and to the kernel instance (a header's kernels are instantiated in every
// translation unit that includes it), so each context keeps its own list of the kernels it has set.
template <typename... KArgs>
static inline cudaError_t ctr_smem_optin(ctr_ctx* ctx, void (*kernel)(KArgs...), int bytes) {
  const void* k = reinterpret_cast<const void*>(kernel);
  for (const void* done : ctx->smem_optin)
    if (done == k) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) ctx->smem_optin.push_back(k);
  return e;
}

__device__ __forceinline__ unsigned long long warp_incl_scan_u64(unsigned long long v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane_id() >= (unsigned)o) v += n;
  }
  return v;
}

__device__ __forceinline__ unsigned warp_incl_scan_u32(unsigned v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned n = __shfl_up_sync(0xffffffffu, v, o);
    if (lane_id() >= (unsigned)o) v += n;
  }
  return v;
}

// Decoupled look-back (Merrill & Garland) over tiles handed out by ticket.  One 64-bit status word per
// tile per scan: bits 63..62 = state (0 invalid, 1 aggregate, 2 inclusive prefix), low 62 bits = value
// (two packed 31-bit sums).  A single word carries state and value, so no fence is needed between them.
#define CTR_LB_AGG (1ull << 62)
#define CTR_LB_INC (2ull << 62)
#define CTR_LB_VAL ((1ull << 62) - 1)

__device__ __forceinline__ unsigned long long lb_load(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void lb_store(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Called by one full warp.  Returns the exclusive prefix of `tile` (sum of aggregates of tiles < tile)
// and publishes the inclusive prefix.  status has one word per tile, zero-initialised.
// The two halves can be called apart: publish the aggregate as soon as it is known, do whatever does not need the
// prefix, then resolve it -- by then the predecessors have usually published theirs and nobody polls.
__device__ __forceinline__ void lb_publish(unsigned long long* status, int tile, unsigned long long aggregate) {
  if (lane_id() == 0) lb_store(&status[tile], (tile == 0 ? CTR_LB_INC : CTR_LB_AGG) | aggregate);
}

__device__ __forceinline__ unsigned long long lb_resolve(unsigned long long* status, int tile, unsigned long long aggregate) {
  const unsigned lane = lane_id();
  if (tile == 0) return 0ull;
  unsigned long long excl = 0;
  int idx = tile - 1;
  while (true) {
    int my = idx - (int)lane;
    unsigned long long s;
    if (my >= 0) {
      do {
        s = lb_load(&status[my]);
      } while ((s >> 62) == 0ull);
    } else {
      s = CTR_LB_INC;  // virtual tile before the first: inclusive prefix 0
    }
    unsigned inc = __ballot_sync(0xffffffffu, (s >> 62) == 2ull);
    unsigned long long v = s & CTR_LB_VAL;
    if (inc) {
      int first = __ffs(inc) - 1;
      if ((int)lane > first) v = 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    excl += v;
    if (inc) break;
    idx -= 32;
  }
  if (lane == 0) lb_store(&status[tile], CTR_LB_INC | (excl + aggregate));
  return excl;
}

__device__ __forceinline__ unsigned long long lb_lookback(unsigned long long* status, int tile,
                                                          unsigned long long aggregate) {
  lb_publish(status, tile, aggregate);
  return lb_resolve(status, tile, aggregate);
}

#endif  // __CUDACC__
