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
  unsigned last3_edited = 0;              // passes that have rewritten the device mesh of that run: 1 seeded selection, 2 clean-up,
                                          // 4 component filter, 8 smoothing
  // bumped by every 3D run and every pass that removes or renumbers mesh rows (selection, clean-up, offset_ids,
  // component filter) or moves vertices (smoothing); the vertex values and the components below record the generation
  // they were computed on
  uint64_t mesh_gen = 0;
  // 3D: an extraction enqueued by ctr_mt3d_enqueue and not yet finished
  bool pending3 = false;
  alignas(8) unsigned char pending3_params[160] = {};
  // 3D: capacities of the output pools / work lists kept from earlier runs, last list lengths, launch coverage
  size_t spec_v = 0, spec_t = 0, spec_own = 0, spec_cell = 0, last_own = 0, last_cell = 0, cover_own = 0, cover_cell = 0;
  size_t spec_w = 0, last_w = 0, cover_w = 0;   // interesting-word list of the split stage 2
  DevBuf wlist;
  // 3D vertex values (ctr_mt3d_interpolate): rows and components of aux[43]; 0 = none since the last 3D run
  size_t attr_rows = 0;
  int attr_ncomp = 0;
  uint64_t attr_gen = 0;
  // 3D connected components (ctr_mt3d_components): triangles and components of aux[44] / aux[45]; -1 = none since the
  // last 3D run
  int64_t comp_tris = 0, comp_count = -1;
  uint64_t comp_gen = 0;

  // 2D / 4D extra outputs are declared in their own translation units via these generic slots
  DevBuf aux[48];            // 0-4, 32-35, 41: 3D; 5-10: 2D; 12-26: 4D; 27-31: mesh passes; 36-40: 2D polylines;
                             // 42-43: 3D vertex values (staged attribute field, values);
                             // 44-45: 3D connected components (triangle labels, component table);
                             // 46-47: smoothing's fp64 working copies
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

static inline void ctr_stage_mark(ctr_ctx* ctx, int idx) {
  if (!ctx->timing) return;
  if (!ctx->ev[idx]) cudaEventCreate(&ctx->ev[idx]);
  cudaEventRecord(ctx->ev[idx], ctx->stream);
  ctx->ev_set[idx] = true;
}

// ------------------------------------------------------------------------------------------ device
#ifdef __CUDACC__

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

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
