// Polylines of the 2D contours on the device (SURVEY.md 8 a23 / f4): the reference chains its contour pairs a vertex at
// a time (triangulated.py:221-305 find_adjacencies / get_contour_sequences); here the segment soup of the last
// ctr_mt2d_run is ranked by pointer jumping over darts.
//
//   vertex  = (level, edge key); a key of one level lies on at most two segments unless a sample sits exactly on the level;
//   darts.cuh : the darts, their successors, the first dart and position of every dart, the kept contours, the scans;
//   k_p_points : points written in position order, one contour after the other;
//   k_p_dedupe* : consecutive np.allclose points dropped (triangulated.py:269), a contour that returns to its start is closed.
// The numpy statement of the same rules is contourist_b200/triangulated.py rank_darts / chain_segments (host, kept for
// levels where a key has more than two segments: there the reference's result is a matter of visiting order, and the
// facade's fixed-order walk decides).
#include <math.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "uf_hash.cuh"

namespace {

#include "darts.cuh"

// the vertex of a dart's tail is (level, key): keys are < 2^35 ((lin << 3 | d << 1 | lowmin), lin < 2^32), levels < 64
struct Vert2 {
  const uint8_t* __restrict__ level;
  __device__ __forceinline__ unsigned long long id(const unsigned long long* __restrict__ keys, unsigned d) const {
    return ((unsigned long long)level[d >> 1] << 40) | keys[d];
  }
  __device__ __forceinline__ unsigned long long prio(const unsigned long long* __restrict__ keys, unsigned d) const { return id(keys, d); }
  __device__ __forceinline__ void junction(unsigned d, PolyCounters* ctr) const { atomicOr(&ctr->junction_levels, 1ull << level[d >> 1]); }
};

// contour descriptors + points: the first dart writes (level, closed, start key, first point), every kept dart the
// point it arrives at
template <typename G>
__global__ void k_p_points(unsigned nd, const uint8_t* __restrict__ level, const unsigned long long* __restrict__ keys,
                           const G* __restrict__ pos, const unsigned* __restrict__ start, const unsigned* __restrict__ dist,
                           const unsigned* __restrict__ npts, const unsigned* __restrict__ off, const unsigned* __restrict__ pidx,
                           G* __restrict__ pts, unsigned* __restrict__ poly_of_point, int* __restrict__ p_level,
                           uint8_t* __restrict__ p_closed, unsigned long long* __restrict__ p_key, unsigned* __restrict__ p_off) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const unsigned sd = start[d];
  const unsigned n = npts[sd];
  if (!n) return;
  const unsigned len = dist[sd] + 1u;
  const unsigned p = len - 1u - dist[d];                      // position of this dart behind the first one
  const bool open = start[sd ^ 1u] == sd;
  const unsigned o = off[sd], pl = pidx[sd];
  if (d == sd) {
    p_level[pl] = (int)level[d >> 1];
    p_closed[pl] = open ? 0 : 1;
    p_key[pl] = keys[d];
    p_off[pl] = o;
    pts[(size_t)o * 2] = pos[(size_t)d * 2];                   // end q of segment s is row 2s+q of the position array
    pts[(size_t)o * 2 + 1] = pos[(size_t)d * 2 + 1];
    poly_of_point[o] = pl;
  }
  if (p + 1u < n) {                                            // open: p < m; closed: p < m - 1
    const unsigned h = d ^ 1u;
    pts[(size_t)(o + p + 1u) * 2] = pos[(size_t)h * 2];
    pts[(size_t)(o + p + 1u) * 2 + 1] = pos[(size_t)h * 2 + 1];
    poly_of_point[o + p + 1u] = pl;
  }
}

template <typename G>
__device__ __forceinline__ bool close2(const G* a, const G* b) {        // np.allclose(a, b)
  return fabs((double)a[0] - (double)b[0]) <= 1e-8 + 1e-5 * fabs((double)b[0]) &&
         fabs((double)a[1] - (double)b[1]) <= 1e-8 + 1e-5 * fabs((double)b[1]);
}

// keep[q] = 0 for a point np.allclose to the one before it in the same contour (triangulated.py:269)
template <typename G>
__global__ void k_p_dedupe_flag(unsigned np_, const G* __restrict__ pts, const unsigned* __restrict__ poly_of_point,
                                const unsigned* __restrict__ p_off, unsigned* __restrict__ keep) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= np_) return;
  const bool first = p_off[poly_of_point[q]] == q;
  keep[q] = (first || !close2(pts + (size_t)q * 2, pts + (size_t)(q - 1) * 2)) ? 1u : 0u;
}

template <typename G>
__global__ void k_p_dedupe_move(unsigned np_, const G* __restrict__ pts, const unsigned* __restrict__ keep, const unsigned* __restrict__ idx,
                                G* __restrict__ out) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= np_ || !keep[q]) return;
  out[(size_t)idx[q] * 2] = pts[(size_t)q * 2];
  out[(size_t)idx[q] * 2 + 1] = pts[(size_t)q * 2 + 1];
}

// new offsets of the contours; a contour whose (filtered) ends are np.allclose is closed
template <typename G>
__global__ void k_p_dedupe_polys(unsigned npoly, unsigned np_, unsigned np_final, const unsigned* __restrict__ idx,
                                 const unsigned* __restrict__ old_off, const unsigned* __restrict__ sorted_old_off_next,
                                 const G* __restrict__ out, unsigned* __restrict__ new_off, unsigned* __restrict__ new_len,
                                 uint8_t* __restrict__ p_closed) {
  const unsigned pl = blockIdx.x * blockDim.x + threadIdx.x;
  if (pl >= npoly) return;
  const unsigned o = old_off[pl], e = sorted_old_off_next[pl];                  // old range [o, e)
  const unsigned no = idx[o], ne = e < np_ ? idx[e] : np_final;
  new_off[pl] = no;
  new_len[pl] = ne - no;
  if (ne - no > 1u && close2(out + (size_t)no * 2, out + (size_t)(ne - 1u) * 2)) p_closed[pl] |= 2;   // bit 0 stays structural
}

__global__ void k_p_old_ends(unsigned npoly, const unsigned* __restrict__ p_off, const unsigned* __restrict__ npts_of_poly,
                             unsigned* __restrict__ end_of) {
  const unsigned pl = blockIdx.x * blockDim.x + threadIdx.x;
  if (pl >= npoly) return;
  end_of[pl] = p_off[pl] + npts_of_poly[pl];
}

__global__ void k_p_len(unsigned nd, const unsigned* __restrict__ npts, const unsigned* __restrict__ pidx, unsigned* __restrict__ len_of_poly) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd || !npts[d]) return;
  len_of_poly[pidx[d]] = npts[d];
}

template <typename G>
int polylines_typed(ctr_ctx* ctx, ctr_poly_counts* out) {
  cudaStream_t st = ctx->stream;
  const size_t S = (size_t)ctx->last_counts[0];
  memset(out, 0, sizeof *out);
  ctx->poly_counts[0] = ctx->poly_counts[1] = 0;
  if (S == 0) return 0;
  if (S >= (1ull << 30)) return ctr_fail(ctx, CTR_ERR_OVERFLOW, "more than 2^30 segments: chain row bands separately");
  const unsigned nd = (unsigned)(2 * S);
  const uint8_t* level = (const uint8_t*)ctx->aux[8].p;
  const unsigned long long* keys = (const unsigned long long*)ctx->aux[9].p;
  const G* pos = (const G*)ctx->aux[10].p;
  size_t nslots = 1024;
  while (nslots < (size_t)nd * 2) nslots <<= 1;
  const unsigned nb_scan = (nd + PS_TILE - 1) / PS_TILE;
  size_t off = 0;
  auto carve = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t o_tab = carve(nslots * sizeof(VSlot)), o_succ = carve((size_t)nd * 4), o_bp = carve((size_t)nd * 8),
               o_bp2 = carve((size_t)nd * 8), o_bd = carve((size_t)nd * 4), o_bd2 = carve((size_t)nd * 4), o_j = carve((size_t)nd * 4),
               o_j2 = carve((size_t)nd * 4), o_d = carve((size_t)nd * 4), o_d2 = carve((size_t)nd * 4), o_np = carve((size_t)nd * 4),
               o_off = carve((size_t)nd * 4), o_pi = carve((size_t)nd * 4), o_bs = carve((size_t)nb_scan * 8 + 64), o_ctr = carve(256),
               o_tot = carve(64);
  DevBuf& b_s = ctx->aux[36];
  int rc;
  if ((rc = ctr_ensure(ctx, b_s, off))) return rc;
  char* base = (char*)b_s.p;
  VSlot* tab = (VSlot*)(base + o_tab);
  unsigned* succ = (unsigned*)(base + o_succ);
  unsigned long long *bp = (unsigned long long*)(base + o_bp), *bp2 = (unsigned long long*)(base + o_bp2);
  unsigned *bd = (unsigned*)(base + o_bd), *bd2 = (unsigned*)(base + o_bd2), *jmp = (unsigned*)(base + o_j), *jmp2 = (unsigned*)(base + o_j2);
  unsigned *dist = (unsigned*)(base + o_d), *dist2 = (unsigned*)(base + o_d2);
  unsigned *npts = (unsigned*)(base + o_np), *poff = (unsigned*)(base + o_off), *pidx = (unsigned*)(base + o_pi);
  unsigned* bsum = (unsigned*)(base + o_bs);
  PolyCounters* dctr = (PolyCounters*)(base + o_ctr);
  unsigned* dtot = (unsigned*)(base + o_tot);
  const unsigned blocks = (nd + 255) / 256;
  PolyCounters h;
  k_p_init<<<ctx->sm_count * 8, 256, 0, st>>>(tab, nslots, dctr);
  const Vert2 vert{level};
  k_p_insert<<<blocks, 256, 0, st>>>(vert, keys, nd, tab, nslots - 1, dctr);
  k_p_succ<<<blocks, 256, 0, st>>>(vert, keys, nd, tab, nslots - 1, succ, bp, bd, jmp);
  ctx->launches += 3;
  // first dart of every cycle
  for (int round = 0; round < 40; round += 2) {
    CTR_CUDA(ctx, cudaMemsetAsync(&dctr->changed, 0, 4, st));
    k_p_min<<<blocks, 256, 0, st>>>(nd, bp, bd, jmp, bp2, bd2, jmp2, dctr);
    k_p_min<<<blocks, 256, 0, st>>>(nd, bp2, bd2, jmp2, bp, bd, jmp, dctr);
    ctx->launches += 2;
    CTR_CUDA(ctx, cudaMemcpyAsync(&h, dctr, sizeof h, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (h.junction_levels) {
      out->junction_levels = h.junction_levels;                 // the host's fixed-order walk decides such levels
      return 0;
    }
    if (!h.changed) break;
  }
  unsigned* start = bd;                                         // first dart of each dart's cycle
  // positions: cut in front of the first dart, rank
  unsigned *nxt = jmp, *nxt2 = jmp2;
  k_p_cut<<<blocks, 256, 0, st>>>(nd, succ, start, nxt, dist);
  ctx->launches++;
  for (int round = 0; round < 40; round += 2) {
    CTR_CUDA(ctx, cudaMemsetAsync(&dctr->live, 0, 4, st));
    k_p_rank<<<blocks, 256, 0, st>>>(nd, nxt, dist, nxt2, dist2, dctr);
    k_p_rank<<<blocks, 256, 0, st>>>(nd, nxt2, dist2, nxt, dist, dctr);
    ctx->launches += 2;
    CTR_CUDA(ctx, cudaMemcpyAsync(&h, dctr, sizeof h, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (!h.live) break;
  }
  // kept contours, their sizes and places
  k_p_mark<<<blocks, 256, 0, st>>>(nd, keys, start, dist, npts);
  ctx->launches++;
  scan_u32(ctx, npts, nd, poff, pidx, bsum, dtot);
  unsigned tot[2];
  CTR_CUDA(ctx, cudaMemcpyAsync(tot, dtot, 8, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned np_ = tot[0], npoly = tot[1];
  if (!npoly) return 0;
  DevBuf &b_pts = ctx->aux[37], &b_pts2 = ctx->aux[38], &b_desc = ctx->aux[39], &b_tmp = ctx->aux[40];
  if ((rc = ctr_ensure(ctx, b_pts, (size_t)np_ * 2 * sizeof(G) + 16))) return rc;
  if ((rc = ctr_ensure(ctx, b_pts2, (size_t)np_ * 2 * sizeof(G) + 16))) return rc;
  // descriptors: level i32, start key u64, offset u32, length u32, closed u8
  const size_t d_key = 0, d_lvl = (size_t)npoly * 8, d_off = d_lvl + (size_t)npoly * 4, d_len = d_off + (size_t)npoly * 4,
               d_cl = d_len + (size_t)npoly * 4;
  if ((rc = ctr_ensure(ctx, b_desc, d_cl + npoly + 64))) return rc;
  // scratch per point / per contour
  const unsigned nb2 = (np_ + PS_TILE - 1) / PS_TILE;
  size_t t_off = 0;
  auto carve2 = [&](size_t bytes) {
    const size_t o = t_off;
    t_off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t t_pop = carve2((size_t)np_ * 4), t_keep = carve2((size_t)np_ * 4), t_idx = carve2((size_t)np_ * 4),
               t_bs = carve2((size_t)nb2 * 8 + 64), t_ooff = carve2((size_t)npoly * 4), t_oend = carve2((size_t)npoly * 4),
               t_olen = carve2((size_t)npoly * 4);
  if ((rc = ctr_ensure(ctx, b_tmp, t_off))) return rc;
  char* tb = (char*)b_tmp.p;
  unsigned *pop = (unsigned*)(tb + t_pop), *keep = (unsigned*)(tb + t_keep), *idx = (unsigned*)(tb + t_idx), *bs2 = (unsigned*)(tb + t_bs),
           *ooff = (unsigned*)(tb + t_ooff), *oend = (unsigned*)(tb + t_oend), *olen = (unsigned*)(tb + t_olen);
  char* db = (char*)b_desc.p;
  unsigned long long* p_key = (unsigned long long*)(db + d_key);
  int* p_level = (int*)(db + d_lvl);
  unsigned* p_off = (unsigned*)(db + d_off);
  unsigned* p_len = (unsigned*)(db + d_len);
  uint8_t* p_closed = (uint8_t*)(db + d_cl);
  k_p_points<G><<<blocks, 256, 0, st>>>(nd, level, keys, pos, start, dist, npts, poff, pidx, (G*)b_pts.p, pop, p_level, p_closed, p_key, ooff);
  k_p_len<<<blocks, 256, 0, st>>>(nd, npts, pidx, olen);
  const unsigned pb = (npoly + 255) / 256, qb = (np_ + 255) / 256;
  k_p_old_ends<<<pb, 256, 0, st>>>(npoly, ooff, olen, oend);
  k_p_dedupe_flag<G><<<qb, 256, 0, st>>>(np_, (const G*)b_pts.p, pop, ooff, keep);
  ctx->launches += 4;
  scan_u32(ctx, keep, np_, idx, nullptr, bs2, dtot);
  CTR_CUDA(ctx, cudaMemcpyAsync(tot, dtot, 8, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned np_final = tot[0];
  k_p_dedupe_move<G><<<qb, 256, 0, st>>>(np_, (const G*)b_pts.p, keep, idx, (G*)b_pts2.p);
  k_p_dedupe_polys<G><<<pb, 256, 0, st>>>(npoly, np_, np_final, idx, ooff, oend, (const G*)b_pts2.p, p_off, p_len, p_closed);
  ctx->launches += 2;
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->poly_counts[0] = npoly;
  ctx->poly_counts[1] = np_final;
  out->n_polylines = npoly;
  out->n_points = np_final;
  return 0;
}

}  // namespace

extern "C" int ctr_mt2d_polylines(ctr_ctx* ctx, ctr_poly_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (ctx->last_kind != 2 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt2d_run with geometry to chain");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  return with_geom_type(ctx, [&](auto g) { return polylines_typed<decltype(g)>(ctx, out); });
}

extern "C" int ctr_mt2d_polylines_fetch(ctr_ctx* ctx, int32_t* level, uint8_t* closed, uint64_t* start_key, uint32_t* offset,
                                        uint32_t* length, void* points) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 2) return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt2d_run");
  const size_t npoly = (size_t)ctx->poly_counts[0], np_ = (size_t)ctx->poly_counts[1];
  if (!npoly) return 0;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t gsz = (ctx->last_flags & CTR_GEOM_F64) ? 8 : 4;
  const char* db = (const char*)ctx->aux[39].p;
  const size_t d_lvl = npoly * 8, d_off = d_lvl + npoly * 4, d_len = d_off + npoly * 4, d_cl = d_len + npoly * 4;
  if (start_key) CTR_CUDA(ctx, cudaMemcpyAsync(start_key, db, npoly * 8, cudaMemcpyDeviceToHost, st));
  if (level) CTR_CUDA(ctx, cudaMemcpyAsync(level, db + d_lvl, npoly * 4, cudaMemcpyDeviceToHost, st));
  if (offset) CTR_CUDA(ctx, cudaMemcpyAsync(offset, db + d_off, npoly * 4, cudaMemcpyDeviceToHost, st));
  if (length) CTR_CUDA(ctx, cudaMemcpyAsync(length, db + d_len, npoly * 4, cudaMemcpyDeviceToHost, st));
  if (closed) CTR_CUDA(ctx, cudaMemcpyAsync(closed, db + d_cl, npoly, cudaMemcpyDeviceToHost, st));
  if (points && np_) CTR_CUDA(ctx, cudaMemcpyAsync(points, ctx->aux[38].p, np_ * 2 * gsz, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}
