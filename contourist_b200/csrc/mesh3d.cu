// Stage 4b (SURVEY.md 8(f1)): the reference's outward orientation of the indexed mesh, on the device.
//
// surface_geometry.py:52-140 orients every edge-connected component of the triangle mesh by a DFS seeded at the
// triangle with the largest |cross.x| at the component's max-x vertex, flipped so that cross.x > 0.  The engine's
// triangles are already wound consistently (normal towards the high side of the field), so only ONE decision per
// component is left: keep or reverse.  This file takes the last ctr_mt3d_run's device mesh and
//   k_o_edges   : inserts every undirected triangle edge into an open-addressing hash table, value = smallest id of
//                 the triangles that share it;
//   k_o_union   : unites each triangle with that triangle (lock-free union-find, path halving);
//   k_o_maxx    : root of every triangle, and per component the largest vertex x (atomicMax on an order-preserving key);
//   k_o_best / k_o_pick : per component the triangle at that x with the largest |cross.x| (ties: smallest index);
//   k_o_decide / k_o_flip : reverse the triangles of components whose seed has cross.x < 0.
// Components are joined through shared EDGES, as in the reference (two sheets touching in one vertex stay apart).
// components3d.cuh (ctr_mt3d_components) reuses the edge table and k_o_union to number and measure the components.
// smooth3d.cuh (ctr_mt3d_smooth) builds the same edge table with its use counts for the fixed vertices and neighbour lists.
// section3d.cuh (ctr_mt3d_section) names the crossing vertices of its plane sections by their slots in that table.
// clip3d.cuh (ctr_mt3d_clip) keeps the part of the mesh on one side of a plane or a vertex value, with the section's side
// test and crossing point, the caps' corner walk and one new vertex per crossed edge, found in the same kind of table.
// closest3d.cuh (ctr_mt3d_closest) finds the closest point of the mesh to query points through a tree it builds per call.
// raycast3d.cuh (ctr_mt3d_raycast) finds the first hit of rays on the mesh through the same tree, built the same way.
#include <math.h>
#include <string.h>

#include <algorithm>

#include <cub/device/device_radix_sort.cuh>             // header-only, with the toolkit: the sort of closest3d.cuh

#include "common.cuh"
#include "uf_hash.cuh"

namespace {

using ufh::EMPTY;
using ufh::uf_find;
using ufh::uf_union;
typedef ufh::Slot EdgeSlot;

__device__ __forceinline__ unsigned long long edge_key(int a, int b) {
  const unsigned lo = (unsigned)min(a, b), hi = (unsigned)max(a, b);
  return ((unsigned long long)hi << 32) | lo;
}

__device__ __forceinline__ EdgeSlot* edge_slot(EdgeSlot* tab, size_t mask, unsigned long long key, bool insert) {
  return ufh::hash_slot(tab, mask, key, insert);
}

// slots of the edge table of nt triangles: 1.5 nt distinct edges on closed sheets (3 nt at worst): load <= 3/8 (3/4)
static inline size_t edge_slots(unsigned nt) {
  size_t n = 1;
  while (n < (size_t)nt * 4) n <<= 1;
  return n;
}

// a pass found triangle ids outside [0, n_verts)
static inline int fail_shifted_ids(ctr_ctx* ctx) {
  return ctr_fail(ctx, CTR_ERR_STATE, "triangle ids outside [0, n_verts): the ids were shifted (ctr_mt3d_offset_ids)");
}

__global__ void k_o_init(EdgeSlot* tab, size_t nslots, int* parent, unsigned nt, unsigned long long* comp_key,
                         unsigned long long* comp_best) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t; q < nslots; q += n) reinterpret_cast<int4*>(tab)[q] = make_int4(-1, -1, 0x7fffffff, 0);
  for (size_t q = t; q < nt; q += n) {
    parent[q] = (int)q;
    comp_key[q] = 0ull;
    comp_best[q] = 0ull;
  }
}

__global__ void k_o_edges(const int* __restrict__ tris, unsigned nt, EdgeSlot* tab, size_t mask) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int a = tris[(size_t)t * 3], b = tris[(size_t)t * 3 + 1], c = tris[(size_t)t * 3 + 2];
  atomicMin(&edge_slot(tab, mask, edge_key(a, b), true)->tri, (int)t);
  atomicMin(&edge_slot(tab, mask, edge_key(b, c), true)->tri, (int)t);
  atomicMin(&edge_slot(tab, mask, edge_key(c, a), true)->tri, (int)t);
}

__global__ void k_o_union(const int* __restrict__ tris, unsigned nt, EdgeSlot* tab, size_t mask, int* parent) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int m = edge_slot(tab, mask, edge_key(v[e], v[(e + 1) % 3]), false)->tri;
    if (m != (int)t) uf_union(parent, (int)t, m);
  }
}

__device__ __forceinline__ unsigned long long okey(double x) {          // order-preserving, > 0 for every non-NaN
  unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

template <typename G>
__device__ __forceinline__ void tri_stats(const G* __restrict__ verts, const int* __restrict__ tris, unsigned t, double& maxx,
                                          double& cross_x) {
  const int a = tris[(size_t)t * 3], b = tris[(size_t)t * 3 + 1], c = tris[(size_t)t * 3 + 2];
  const double ax = verts[(size_t)a * 3], ay = verts[(size_t)a * 3 + 1], az = verts[(size_t)a * 3 + 2];
  const double bx = verts[(size_t)b * 3], by = verts[(size_t)b * 3 + 1], bz = verts[(size_t)b * 3 + 2];
  const double cx = verts[(size_t)c * 3], cy = verts[(size_t)c * 3 + 1], cz = verts[(size_t)c * 3 + 2];
  maxx = fmax(ax, fmax(bx, cx));
  // x component of cross(A - B, A - C)  (surface_geometry.py:93-95)
  cross_x = __dsub_rn(__dmul_rn(ay - by, az - cz), __dmul_rn(az - bz, ay - cy));
}

// atomicMax(&slot[r], k) for a whole warp: lanes with the same root combine first, and a slot that already holds at
// least k is left alone (the target only grows, so a stale read can only under-estimate it).  Without both, every
// triangle of a large component hits one address.
__device__ __forceinline__ void warp_max_to_root(unsigned long long* slot, int r, unsigned long long k, bool valid) {
  const unsigned act = __ballot_sync(0xffffffffu, valid);
  if (!valid) return;
  const unsigned peers = __match_any_sync(act, r);
  unsigned long long best = k;
  for (unsigned m = peers & (peers - 1) ? peers : 0u; m; m &= m - 1) {      // (skipped when alone in the group)
    const unsigned long long o = __shfl_sync(peers, k, __ffs(m) - 1);
    best = o > best ? o : best;
  }
  if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31) && *(volatile unsigned long long*)&slot[r] < best) atomicMax(&slot[r], best);
}

template <typename G>
__global__ void k_o_maxx(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt, int* parent, int* root,
                         unsigned long long* comp_key) {
  // blocks walk the triangle list from its end: the engine emits triangles by ascending x, so the running maximum is
  // found by the first wave and the remaining blocks only read it
  const unsigned t = (gridDim.x - 1 - blockIdx.x) * blockDim.x + threadIdx.x;
  const bool in = t < nt;
  int r = 0;
  double maxx = 0, cx;
  if (in) {
    r = (int)t;                                       // no unions any more: walk read-only, then one compressing write
    for (int q = parent[r]; q != r; q = parent[r]) r = q;
    if (r != (int)t) parent[t] = r;
    root[t] = r;                                      // a separate array: parent[] may still be rewritten by other walkers
    tri_stats(verts, tris, t, maxx, cx);
  }
  warp_max_to_root(comp_key, r, okey(maxx), in && maxx == maxx);
}

// largest |cross.x| among the triangles that reach the component's max x
template <typename G>
__global__ void k_o_best(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt, const int* __restrict__ parent,
                         const unsigned long long* __restrict__ comp_key, unsigned long long* comp_best) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int r = parent[t];
  double maxx, cx;
  tri_stats(verts, tris, t, maxx, cx);
  if (!(maxx == maxx) || okey(maxx) != comp_key[r]) return;
  const unsigned long long k = okey(fabs(cx));
  if (*(volatile unsigned long long*)&comp_best[r] < k) atomicMax(&comp_best[r], k);
}

// ... and the smallest index among those that attain it: the component's seed
template <typename G>
__global__ void k_o_pick(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt, const int* __restrict__ parent,
                         const unsigned long long* __restrict__ comp_key, const unsigned long long* __restrict__ comp_best,
                         int* comp_tri) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int r = parent[t];
  double maxx, cx;
  tri_stats(verts, tris, t, maxx, cx);
  if (!(maxx == maxx) || okey(maxx) != comp_key[r]) return;
  if (okey(fabs(cx)) == comp_best[r]) atomicMin(&comp_tri[r], (int)t);
}

// one decision per component (its root triangle takes it): reverse iff the seed faces -x (surface_geometry.py:100-103)
template <typename G>
__global__ void k_o_decide(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt, const int* __restrict__ parent,
                           int* comp_tri, unsigned* n_comp) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || parent[t] != (int)t) return;
  atomicAdd(n_comp, 1u);
  const int seed = comp_tri[t];
  int flip = 0;
  if (seed >= 0 && seed < (int)nt) {
    double maxx, cx;
    tri_stats(verts, tris, (unsigned)seed, maxx, cx);
    flip = cx < 0 ? 1 : 0;
  }
  comp_tri[t] = flip;                                 // reused as the component's flip flag
}

__global__ void k_o_flip(int* __restrict__ tris, unsigned nt, const int* __restrict__ parent, const int* __restrict__ comp_flip,
                         unsigned* n_flipped) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  if (comp_flip[parent[t]]) {
    const int a = tris[(size_t)t * 3], c = tris[(size_t)t * 3 + 2];
    tris[(size_t)t * 3] = c;
    tris[(size_t)t * 3 + 2] = a;
    atomicAdd(n_flipped, 1u);
  }
}

template <typename G>
int orient_typed(ctr_ctx* ctx, int64_t* n_components, int64_t* n_flipped) {
  const unsigned nt = (unsigned)ctx->last_counts[1];
  cudaStream_t st = ctx->stream;
  if (n_components) *n_components = 0;
  if (n_flipped) *n_flipped = 0;
  if (nt == 0) return 0;
  const size_t nslots = edge_slots(nt);
  int rc;
  DevBuf& b_tab = ctx->aux[AUX_SCRATCH0];
  DevBuf& b_par = ctx->aux[AUX_SCRATCH2];
  DevBuf& b_comp = ctx->aux[AUX_SCRATCH3];
  if ((rc = ctr_ensure(ctx, b_tab, nslots * sizeof(EdgeSlot)))) return rc;
  if ((rc = ctr_ensure(ctx, b_par, (size_t)nt * 8))) return rc;
  if ((rc = ctr_ensure(ctx, b_comp, (size_t)nt * (8 + 8 + 4) + 64))) return rc;
  EdgeSlot* tab = (EdgeSlot*)b_tab.p;
  int* parent = (int*)b_par.p;
  int* root = parent + nt;
  unsigned long long* comp_key = (unsigned long long*)b_comp.p;
  unsigned long long* comp_best = comp_key + nt;
  int* comp_tri = (int*)(comp_best + nt);
  unsigned* counters = (unsigned*)(comp_tri + nt);    // [0] flipped, [1] components
  const G* verts = (const G*)ctx->verts.p;
  int* tris = (int*)ctx->tris.p;
  const unsigned blocks = (nt + 255) / 256;
  k_o_init<<<ctx->sm_count * 8, 256, 0, st>>>(tab, nslots, parent, nt, comp_key, comp_best);
  CTR_CUDA(ctx, cudaMemsetAsync(comp_tri, 0x7f, (size_t)nt * 4, st));
  CTR_CUDA(ctx, cudaMemsetAsync(counters, 0, 8, st));
  k_o_edges<<<blocks, 256, 0, st>>>(tris, nt, tab, nslots - 1);
  k_o_union<<<blocks, 256, 0, st>>>(tris, nt, tab, nslots - 1, parent);
  k_o_maxx<G><<<blocks, 256, 0, st>>>(verts, tris, nt, parent, root, comp_key);
  k_o_best<G><<<blocks, 256, 0, st>>>(verts, tris, nt, root, comp_key, comp_best);
  k_o_pick<G><<<blocks, 256, 0, st>>>(verts, tris, nt, root, comp_key, comp_best, comp_tri);
  k_o_decide<G><<<blocks, 256, 0, st>>>(verts, tris, nt, root, comp_tri, counters + 1);
  k_o_flip<<<blocks, 256, 0, st>>>(tris, nt, root, comp_tri, counters);
  ctx->launches += 8;
  CTR_CUDA(ctx, cudaGetLastError());
  unsigned h[2] = {0, 0};
  CTR_CUDA(ctx, cudaMemcpyAsync(h, counters, 8, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (n_flipped) *n_flipped = h[0];
  if (n_components) *n_components = h[1];
  return 0;
}

#include "normals3d.cuh"
#include "components3d.cuh"
#include "smooth3d.cuh"
#include "section3d.cuh"
#include "compact3d.cuh"
#include "mt3d_keep.cuh"
#include "mt3d_clean.cuh"
#include "decimate3d.cuh"
#include "attr3d.cuh"
#include "cap3d.cuh"
#include "clip3d.cuh"
#include "closest3d.cuh"
#include "raycast3d.cuh"

}  // namespace

extern "C" int ctr_mt3d_orient_reference(ctr_ctx* ctx, int64_t* n_components, int64_t* n_flipped) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (int rc = check_pass(ctx, PASS_ORIENT)) return rc;
  ctx->last3_edited |= EDIT_ORIENT;                   // (also when the call fails below: it may have rewound a part)
  return with_geom_type(ctx, [&](auto g) { return orient_typed<decltype(g)>(ctx, n_components, n_flipped); });
}

extern "C" int ctr_mt3d_components(ctr_ctx* ctx, int64_t* n_components) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (n_components) *n_components = 0;
  ctx->comp_count = -1;                               // the buffers are rewritten: earlier results are gone
  if (int rc = check_pass(ctx, PASS_COMPONENTS)) return rc;
  return with_geom_type(ctx, [&](auto g) { return components_typed<decltype(g)>(ctx, n_components); });
}

extern "C" int ctr_mt3d_smooth(ctr_ctx* ctx, const ctr_smooth_params* sp, ctr_smooth_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!sp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (sp->iterations < 0 || sp->iterations > 1000) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "iterations must be in [0, 1000]");
  if (sp->reserved != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "reserved must be 0");
  if (!(sp->lambda > 0.0 && sp->lambda <= 1.0)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "lambda must be in (0, 1]");
  if (!(sp->mu >= -1.0 && sp->mu <= 0.0)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "mu must be in [-1, 0]");
  if (int rc = check_pass(ctx, PASS_SMOOTH)) return rc;
  return with_geom_type(ctx, [&](auto g) { return smooth_typed<decltype(g)>(ctx, sp, out); });
}

extern "C" int ctr_mt3d_components_fetch(ctr_ctx* ctx, int32_t* tri_component, ctr_mt3d_component* components) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->comp_count < 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_components since the last 3D run");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (tri_component && ctx->comp_tris)
    CTR_CUDA(ctx, cudaMemcpyAsync(tri_component, ctx->aux[AUX_LABELS].p, (size_t)ctx->comp_tris * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (components && ctx->comp_count)
    CTR_CUDA(ctx, cudaMemcpyAsync(components, ctx->aux[AUX_COMPONENTS].p, (size_t)ctx->comp_count * sizeof(ctr_mt3d_component),
                                  cudaMemcpyDeviceToHost, ctx->stream));
  CTR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int ctr_mt3d_section(ctr_ctx* ctx, const ctr_section_params* sp, ctr_section_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!sp || !out || !sp->offsets) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  const double* n = sp->normal;
  if (!(isfinite(n[0]) && isfinite(n[1]) && isfinite(n[2])) || (n[0] == 0.0 && n[1] == 0.0 && n[2] == 0.0))
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "normal must be finite and not zero");
  if (sp->nplanes < 1 || sp->nplanes > 65536) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "nplanes must be in [1, 65536]");
  if (sp->reserved != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "reserved must be 0");
  for (int32_t l = 0; l < sp->nplanes; ++l)
    if (!isfinite(sp->offsets[l]) || (l > 0 && !(sp->offsets[l] > sp->offsets[l - 1])))
      return ctr_fail(ctx, CTR_ERR_BAD_ARG, "offsets must be finite and strictly increasing");
  ctx->sect_count[0] = -1;                            // the buffers are rewritten: earlier results are gone
  if (int rc = check_pass(ctx, PASS_SECTION)) return rc;
  return with_geom_type(ctx, [&](auto g) { return section_typed<decltype(g)>(ctx, sp, out); });
}

extern "C" int ctr_mt3d_section_segments_fetch(ctr_ctx* ctx, int32_t* plane, int32_t* edges, void* points) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->sect_count[0] < 0) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_section since the last 3D run");
  const size_t S = (size_t)ctx->sect_count[0], gsz = (ctx->last_flags & CTR_GEOM_F64) ? 8 : 4;
  if (!S) return 0;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  SecSegs sg;
  ctr_carve c{(char*)ctx->aux[AUX_SECTION_SEGS].p, 0};
  sg.carve(c, S, gsz, (size_t)ctx->sect_nplanes);
  if (plane) CTR_CUDA(ctx, cudaMemcpyAsync(plane, sg.plane, S * 4, cudaMemcpyDeviceToHost, st));
  if (edges) CTR_CUDA(ctx, cudaMemcpyAsync(edges, sg.edges, S * 16, cudaMemcpyDeviceToHost, st));
  if (points) CTR_CUDA(ctx, cudaMemcpyAsync(points, sg.pts, S * 6 * gsz, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}

extern "C" int ctr_mt3d_section_polylines_fetch(ctr_ctx* ctx, int32_t* plane, uint8_t* flags, uint64_t* start_key, uint32_t* offset,
                                                uint32_t* length, double* measures, void* points, uint8_t* junction) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->sect_count[0] < 0) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_section since the last 3D run");
  const size_t S = (size_t)ctx->sect_count[0], P = (size_t)ctx->sect_count[1], N = (size_t)ctx->sect_count[2];
  const size_t np = (size_t)ctx->sect_nplanes, gsz = (ctx->last_flags & CTR_GEOM_F64) ? 8 : 4;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  std::vector<uint32_t> jp(junction ? np : 0);
  if (junction) {
    SecSegs sg;
    ctr_carve c{(char*)ctx->aux[AUX_SECTION_SEGS].p, 0};
    sg.carve(c, S, gsz, np);
    CTR_CUDA(ctx, cudaMemcpyAsync(jp.data(), sg.jplane, np * 4, cudaMemcpyDeviceToHost, st));
  }
  if (P) {
    SecPolys pg;
    ctr_carve c{(char*)ctx->aux[AUX_SECTION_POLYS].p, 0};
    pg.carve(c, P, N, gsz);
    if (plane) CTR_CUDA(ctx, cudaMemcpyAsync(plane, pg.plane, P * 4, cudaMemcpyDeviceToHost, st));
    if (flags) CTR_CUDA(ctx, cudaMemcpyAsync(flags, pg.flags, P, cudaMemcpyDeviceToHost, st));
    if (start_key) CTR_CUDA(ctx, cudaMemcpyAsync(start_key, pg.key, P * 8, cudaMemcpyDeviceToHost, st));
    if (offset) CTR_CUDA(ctx, cudaMemcpyAsync(offset, pg.off, P * 4, cudaMemcpyDeviceToHost, st));
    if (length) CTR_CUDA(ctx, cudaMemcpyAsync(length, pg.len, P * 4, cudaMemcpyDeviceToHost, st));
    if (measures) CTR_CUDA(ctx, cudaMemcpyAsync(measures, pg.meas, P * 16, cudaMemcpyDeviceToHost, st));
    if (points && N) CTR_CUDA(ctx, cudaMemcpyAsync(points, pg.pts, N * 3 * gsz, cudaMemcpyDeviceToHost, st));
  }
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  for (size_t l = 0; l < jp.size(); ++l) junction[l] = jp[l] ? 1 : 0;
  return 0;
}

extern "C" int ctr_mt3d_keep_components(ctr_ctx* ctx, const uint8_t* keep, int64_t n_keep, int64_t* n_verts, int64_t* n_tris) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->comp_count < 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_components since the last 3D run");
  if (ctx->comp_gen != ctx->mesh_gen)
    return ctr_fail(ctx, CTR_ERR_STATE, "the mesh was edited after ctr_mt3d_components (selection, clean-up, smoothing, decimation "
                                        "or offset_ids): call ctr_mt3d_components again");
  if (n_keep != ctx->comp_count || (!keep && n_keep > 0))
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "keep must hold one byte per component of the last ctr_mt3d_components call");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  return keep_components_run(ctx, keep, n_verts, n_tris);
}

extern "C" int ctr_mt3d_clean(ctr_ctx* ctx, const ctr_clean_params* cp, ctr_clean_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!cp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (int rc = check_pass(ctx, PASS_CLEAN)) return rc;
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  for (int a = 0; a < 3; ++a) {
    if (p->origin[a] != 0.0 || p->delta[a] != 1.0)
      return ctr_fail(ctx, CTR_ERR_STATE, "mesh clean-up works in grid coordinates: run with origin 0, delta 1 and pass the transform here");
    if (cp->corner[a] < 1) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "corner must be >= 1 on every axis");
    if (cp->delta[a] == 0.0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "delta must be non-zero");
  }
  if (cp->divisions < 1 || cp->divisions >= (1 << 21)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "divisions must be in [1, 2^21)");
  if (!(cp->epsilon == cp->epsilon)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "epsilon is NaN");
  return with_geom_type(ctx, [&](auto g) { return clean_typed<decltype(g)>(ctx, cp, out); });
}

extern "C" int ctr_mt3d_decimate(ctr_ctx* ctx, const ctr_decimate_params* dp, ctr_decimate_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!dp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  for (int a = 0; a < 3; ++a) {
    if (!(dp->cell[a] > 0.0 && isfinite(dp->cell[a]))) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "cell must be > 0 and finite on every axis");
    if (!isfinite(dp->origin[a])) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "origin must be finite");
  }
  if (int rc = check_pass(ctx, PASS_DECIMATE)) return rc;
  return with_geom_type(ctx, [&](auto g) { return decimate_typed<decltype(g)>(ctx, dp, out); });
}

extern "C" int ctr_mt3d_cap(ctr_ctx* ctx, const ctr_cap_params* cp, ctr_cap_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!cp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (cp->side != CTR_CAP_HIGH && cp->side != CTR_CAP_LOW) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "side must be CTR_CAP_HIGH or CTR_CAP_LOW");
  if (cp->reserved != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "reserved must be 0");
  if (int rc = check_pass(ctx, PASS_CAP)) return rc;
  return with_sample_type(ctx, ((const ctr_mt3d_params*)ctx->last3_params)->dtype, [&](auto t) {
    return with_geom_type(ctx, [&](auto g) { return cap_typed<decltype(t), decltype(g)>(ctx, cp, out); });
  });
}

extern "C" int ctr_mt3d_clip(ctr_ctx* ctx, const ctr_clip_params* cp, ctr_clip_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!cp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (cp->source != CTR_CLIP_PLANE && cp->source != CTR_CLIP_VALUE)
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "source must be CTR_CLIP_PLANE or CTR_CLIP_VALUE");
  if (cp->side != CTR_CLIP_HIGH && cp->side != CTR_CLIP_LOW) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "side must be CTR_CLIP_HIGH or CTR_CLIP_LOW");
  const double* n = cp->normal;
  if (cp->source == CTR_CLIP_PLANE) {
    if (!(isfinite(n[0]) && isfinite(n[1]) && isfinite(n[2])) || (n[0] == 0.0 && n[1] == 0.0 && n[2] == 0.0))
      return ctr_fail(ctx, CTR_ERR_BAD_ARG, "normal must be finite and not zero");
    if (cp->component != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "component must be 0 for a plane clip");
  } else {
    if (n[0] != 0.0 || n[1] != 0.0 || n[2] != 0.0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "normal must be 0 for a value clip");
    if (cp->component < 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "component must be in [0, ncomp) of the last interpolation");
  }
  if (!isfinite(cp->offset)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "offset must be finite");
  if (cp->reserved != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "reserved must be 0");
  if (int rc = check_pass(ctx, PASS_CLIP)) return rc;
  return with_geom_type(ctx, [&](auto g) { return clip_typed<decltype(g)>(ctx, cp, out); });
}

extern "C" int ctr_mt3d_closest(ctr_ctx* ctx, const ctr_closest_params* cp, ctr_closest_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  ctx->closest_n = -1;                                 // a failed call leaves no results
  if (!cp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (cp->dtype != CTR_F32 && cp->dtype != CTR_F64) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32 or CTR_F64");
  if (cp->flags & ~(uint32_t)CTR_FIELD_ON_DEVICE) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "flags must be 0 or CTR_FIELD_ON_DEVICE");
  if (cp->n_points < 0 || cp->n_points > 0x7fffffffll) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "n_points must be in [0, 2^31-1]");
  if (cp->n_points > 0 && !cp->points) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (!(cp->max_distance >= 0.0)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "max_distance must be >= 0 (and not NaN)");
  const size_t nc = (size_t)cp->n_points * 3;
  if (!(cp->flags & CTR_FIELD_ON_DEVICE))              // device points are checked on the device, at the first host wait
    for (size_t i = 0; i < nc; ++i)
      if (!isfinite(cp->dtype == CTR_F64 ? ((const double*)cp->points)[i] : (double)((const float*)cp->points)[i]))
        return ctr_fail(ctx, CTR_ERR_BAD_ARG, "query points must be finite");
  if (int rc = check_pass(ctx, PASS_CLOSEST)) return rc;
  if ((cp->flags & CTR_FIELD_ON_DEVICE) && nc) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, cp->points) != cudaSuccess || at.device != ctx->device ||
        (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
      cudaGetLastError();
      return ctr_fail(ctx, CTR_ERR_BAD_ARG, "device points must be device memory on the context's device");
    }
  }
  return with_geom_type(ctx, [&](auto g) { return closest_typed<decltype(g)>(ctx, cp, out); });
}

extern "C" int ctr_mt3d_closest_fetch(ctr_ctx* ctx, double* distance, int32_t* triangle, double* point) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->closest_n < 0) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_closest since the last 3D run");
  const size_t n = (size_t)ctx->closest_n;
  if (!n) return 0;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  double *dist, *pt;
  int* tri;
  ctr_carve c{(char*)ctx->aux[AUX_CLOSEST_RESULT].p, 0};
  c(dist, n * 8);
  c(tri, n * 4);
  c(pt, n * 24);
  if (distance) CTR_CUDA(ctx, cudaMemcpyAsync(distance, dist, n * 8, cudaMemcpyDefault, st));
  if (triangle) CTR_CUDA(ctx, cudaMemcpyAsync(triangle, tri, n * 4, cudaMemcpyDefault, st));
  if (point) CTR_CUDA(ctx, cudaMemcpyAsync(point, pt, n * 24, cudaMemcpyDefault, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}

extern "C" int ctr_mt3d_raycast(ctr_ctx* ctx, const ctr_ray_params* rp, ctr_ray_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  ctx->ray_n = -1;                                     // a failed call leaves no results
  if (!rp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (rp->dtype != CTR_F32 && rp->dtype != CTR_F64) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32 or CTR_F64");
  if (rp->flags & ~(uint32_t)CTR_FIELD_ON_DEVICE) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "flags must be 0 or CTR_FIELD_ON_DEVICE");
  if (rp->n_rays < 0 || rp->n_rays > 0x7fffffffll) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "n_rays must be in [0, 2^31-1]");
  if (rp->n_rays > 0 && (!rp->origins || !rp->directions)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (!(rp->t_min <= rp->t_max)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "t_min and t_max must not be NaN, and t_min <= t_max");
  const size_t nR = (size_t)rp->n_rays;
  if (!(rp->flags & CTR_FIELD_ON_DEVICE))              // device rays are checked on the device, at the first host wait
    for (size_t i = 0; i < nR; ++i) {
      bool ok = true, moves = false;
      for (int k = 0; k < 3; ++k) {
        const size_t j = i * 3 + k;
        const bool f64 = rp->dtype == CTR_F64;
        const double o = f64 ? ((const double*)rp->origins)[j] : (double)((const float*)rp->origins)[j];
        const double d = f64 ? ((const double*)rp->directions)[j] : (double)((const float*)rp->directions)[j];
        ok = ok && isfinite(o) && isfinite(d);
        moves = moves || d != 0.0;
      }
      if (!(ok && moves)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "rays must be finite with a non-zero direction");
    }
  if (int rc = check_pass(ctx, PASS_RAYCAST)) return rc;
  if ((rp->flags & CTR_FIELD_ON_DEVICE) && nR)
    for (const void* p : {rp->origins, rp->directions}) {
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.device != ctx->device ||
          (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return ctr_fail(ctx, CTR_ERR_BAD_ARG, "device rays must be device memory on the context's device");
      }
    }
  return with_geom_type(ctx, [&](auto g) { return raycast_typed<decltype(g)>(ctx, rp, out); });
}

extern "C" int ctr_mt3d_raycast_fetch(ctr_ctx* ctx, double* t, int32_t* triangle, double* weights, double* point,
                                      int8_t* side) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->ray_n < 0) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_raycast since the last 3D run");
  const size_t n = (size_t)ctx->ray_n;
  if (!n) return 0;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  double *t_d, *wt, *pt;
  int* tri;
  signed char* sd;
  ctr_carve c{(char*)ctx->aux[AUX_RAY_RESULT].p, 0};
  c(t_d, n * 8);
  c(wt, n * 24);
  c(pt, n * 24);
  c(tri, n * 4);
  c(sd, n);
  if (t) CTR_CUDA(ctx, cudaMemcpyAsync(t, t_d, n * 8, cudaMemcpyDefault, st));
  if (triangle) CTR_CUDA(ctx, cudaMemcpyAsync(triangle, tri, n * 4, cudaMemcpyDefault, st));
  if (weights) CTR_CUDA(ctx, cudaMemcpyAsync(weights, wt, n * 24, cudaMemcpyDefault, st));
  if (point) CTR_CUDA(ctx, cudaMemcpyAsync(point, pt, n * 24, cudaMemcpyDefault, st));
  if (side) CTR_CUDA(ctx, cudaMemcpyAsync(side, sd, n, cudaMemcpyDefault, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}

extern "C" int ctr_mt3d_interpolate(ctr_ctx* ctx, const ctr_attr_params* a, int64_t* n_verts) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!a || !a->field) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (a->ncomp < 1 || a->ncomp > 4) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "ncomp must be 1..4");
  if (a->dtype != CTR_F32 && a->dtype != CTR_F64 && a->dtype != CTR_U8 && a->dtype != CTR_I16 && a->dtype != CTR_U16)
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32, CTR_F64, CTR_U8, CTR_I16 or CTR_U16");
  if (int rc = check_pass(ctx, PASS_INTERPOLATE)) return rc;
  ctx->attr_ncomp = 0;                                 // the buffer is rewritten: earlier values are gone
  return with_sample_type(ctx, ((const ctr_mt3d_params*)ctx->last3_params)->dtype, [&](auto t) {
    return with_geom_type(ctx, [&](auto g) { return interp_typed<decltype(t), decltype(g)>(ctx, a, n_verts); });
  });
}

static int interp_check(ctr_ctx* ctx) {
  if (ctx->last_kind != 3 || !ctx->attr_ncomp) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_interpolate since the last 3D run");
  return 0;
}

extern "C" int ctr_mt3d_interpolate_fetch(ctr_ctx* ctx, void* values) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!values) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  int rc = interp_check(ctx);
  if (rc) return rc;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t bytes = ctx->attr_rows * (size_t)ctx->attr_ncomp * ((ctx->last_flags & CTR_GEOM_F64) ? 8 : 4);
  if (bytes) CTR_CUDA(ctx, cudaMemcpyAsync(values, ctx->aux[AUX_VALUES].p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CTR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int ctr_mt3d_interpolate_device_ptr(ctr_ctx* ctx, void** values) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!values) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  int rc = interp_check(ctx);
  if (rc) return rc;
  *values = ctx->aux[AUX_VALUES].p;
  return 0;
}
