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
#include <math.h>
#include <string.h>

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
  size_t nslots = 1;
  while (nslots < (size_t)nt * 4) nslots <<= 1;       // 1.5 nt distinct edges on closed sheets (3 nt at worst): load <= 3/8 (3/4)
  int rc;
  DevBuf& b_tab = ctx->aux[27];
  DevBuf& b_par = ctx->aux[29];
  DevBuf& b_comp = ctx->aux[30];
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

#include "components3d.cuh"
#include "smooth3d.cuh"

}  // namespace

extern "C" int ctr_mt3d_orient_reference(ctr_ctx* ctx, int64_t* n_components, int64_t* n_flipped) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to orient");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->last_flags & CTR_GEOM_F64) return orient_typed<double>(ctx, n_components, n_flipped);
  return orient_typed<float>(ctx, n_components, n_flipped);
}

extern "C" int ctr_mt3d_components(ctr_ctx* ctx, int64_t* n_components) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (n_components) *n_components = 0;
  ctx->comp_count = -1;                               // the buffers are rewritten: earlier results are gone
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to measure");
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  if (p->i_lo != 0 || p->i_hi != p->n0 || p->vert_id_base != 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "components need a full-volume run with vert_id_base 0 (components cross slab faces)");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->last_flags & CTR_GEOM_F64) return components_typed<double>(ctx, n_components);
  return components_typed<float>(ctx, n_components);
}

extern "C" int ctr_mt3d_smooth(ctr_ctx* ctx, const ctr_smooth_params* sp, ctr_smooth_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!sp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (sp->iterations < 0 || sp->iterations > 1000) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "iterations must be in [0, 1000]");
  if (sp->reserved != 0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "reserved must be 0");
  if (!(sp->lambda > 0.0 && sp->lambda <= 1.0)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "lambda must be in (0, 1]");
  if (!(sp->mu >= -1.0 && sp->mu <= 0.0)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "mu must be in [-1, 0]");
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to smooth");
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  if (p->i_lo != 0 || p->i_hi != p->n0 || p->vert_id_base != 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "smoothing needs a full-volume run with vert_id_base 0 (a slab's halo ids belong to another shard)");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->last_flags & CTR_GEOM_F64) return smooth_typed<double>(ctx, sp, out);
  return smooth_typed<float>(ctx, sp, out);
}

extern "C" int ctr_mt3d_components_fetch(ctr_ctx* ctx, int32_t* tri_component, ctr_mt3d_component* components) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->comp_count < 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_components since the last 3D run");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (tri_component && ctx->comp_tris)
    CTR_CUDA(ctx, cudaMemcpyAsync(tri_component, ctx->aux[44].p, (size_t)ctx->comp_tris * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (components && ctx->comp_count)
    CTR_CUDA(ctx, cudaMemcpyAsync(components, ctx->aux[45].p, (size_t)ctx->comp_count * sizeof(ctr_mt3d_component),
                                  cudaMemcpyDeviceToHost, ctx->stream));
  CTR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}
