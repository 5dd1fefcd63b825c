// Clipping of the 3D device mesh by a plane or by a vertex value (ctr_mt3d_clip), like VTK's vtkClipPolyData.
//
// Included into mesh3d.cu after section3d.cuh (sec_side, sec_point) and cap3d.cuh (edge_changes, the corner walk), inside
// its anonymous namespace.  The definition is oracle/mt3d_clip.py:clip; every output is a selection, a copy or one
// fixed-order fp64 formula (__dadd_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn: nothing contracts), so the device result
// equals it bit for bit.  A vertex is kept when its side value s (plane: (n0 x + n1 y) + n2 z; value: one component of
// the current vertex values) is >= offset for CTR_CLIP_HIGH, < offset for CTR_CLIP_LOW.
//   k_clip_side  : thread per vertex: the kept flag; a NaN s raises a flag;
//   k_clip_count : thread per triangle: ids checked; the corner walk's token count gives 0, 1 or 2 pieces (one flag byte
//                  per piece slot, 2 per triangle), a flag for a cut triangle (corners on both sides); dropped triangles
//                  counted per warp, then per block: one global atomic per block;
//   k_flag_scan x 3 : output index of every piece, every kept vertex, every cut triangle.  Host wait 1: the totals and
//                  the flags.  Every vertex kept: nothing is written.  The crossing-edge table is sized from the cut
//                  count (8 slots per cut triangle, load <= 1/4) rather than from the whole mesh;
//   k_clip_edges : thread per cut triangle: its two crossed edges into the ufh::Slot table, atomicMin of the triangle
//                  index: the edge's owner is the first triangle that uses it;
//   k_clip_own   : thread per cut triangle: one flag per crossed edge in walk order (2 per cut triangle), set where the
//                  triangle owns the edge (and for the first of two equal edges of a triangle with a repeated id);
//   k_flag_scan  : the new vertices numbered in first-use order.  Host wait 2: their count, so the overflow check comes
//                  before anything is written;
//   k_clip_verts : thread per cut triangle: the new rows of the edges it owns (position, normal, key, lowmin, values) into
//                  a scratch piece, read from the old rows; the ordinal goes into the slot's spare word;
//   k_sel_rows   : the kept rows of every vertex array through the staging rows, then the new rows behind them;
//   k_clip_tris  : thread per triangle with pieces: the walk again, kept corners renumbered, crossings n_kept + ordinal;
//                  written to the staging rows and copied over the triangles (a piece's index may lie below or above
//                  its source's, so the triangles cannot be rewritten in place).
// Scratch: AUX_SCRATCH0 (per-vertex and per-triangle flags and indices), AUX_SCRATCH1 (edge table, new rows, staging).
// The output buffers and AUX_VALUES grow with ctr_grow_keep, so device pointers handed out before may change.

struct ClipCounters {                                  // head of the scan piece
  unsigned bad_ids, nan, n_dropped, pad;
  unsigned ticket[4];                                  // tile tickets: pieces, kept vertices, cut triangles, new vertices
  unsigned long long total[4];
};
static_assert(sizeof(ClipCounters) <= 64, "ClipCounters fits the 64-byte head of the scan piece");

// s of a vertex: the plane's sec_side on the widened position, or one component of the vertex values
template <typename G>
struct ClipSrc {
  const G* __restrict__ p;                             // positions (3 per row) or vertex values (ncomp per row)
  int stride, comp;
  bool plane;
  SecPlanes P;                                         // (n0, n1, n2 only)
  __device__ __forceinline__ double operator()(unsigned v) const {
    const G* r = p + (size_t)v * stride;
    return plane ? sec_side(P, (double)r[0], (double)r[1], (double)r[2]) : (double)r[comp];
  }
};

struct ClipRows {                                      // the new vertex rows, by ordinal
  void* verts;
  void* normals;
  unsigned long long* keys;
  uint8_t* lowmin;
  void* values;
};

template <typename G>
__global__ void __launch_bounds__(256) k_clip_side(ClipSrc<G> src, unsigned nv, double offset, int side,
                                                   uint8_t* __restrict__ keep_v, ClipCounters* ctr) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const double s = src(v);
  if (s != s) ctr->nan = 1u;
  keep_v[v] = (s >= offset) == (side == CTR_CLIP_HIGH) ? 1 : 0;
}

// bit i: corner i of triangle t is kept
__device__ __forceinline__ unsigned clip_corners(const uint8_t* __restrict__ keep_v, const int v[3]) {
  return (unsigned)keep_v[v[0]] | ((unsigned)keep_v[v[1]] << 1) | ((unsigned)keep_v[v[2]] << 2);
}

__device__ __forceinline__ void clip_tri(const int* __restrict__ tris, unsigned t, int v[3]) {
  v[0] = tris[(size_t)t * 3];
  v[1] = tris[(size_t)t * 3 + 1];
  v[2] = tris[(size_t)t * 3 + 2];
}

__global__ void __launch_bounds__(256) k_clip_count(const int* __restrict__ tris, unsigned nt, unsigned nv,
                                                    const uint8_t* __restrict__ keep_v, uint8_t* __restrict__ piece_flags,
                                                    uint8_t* __restrict__ cut, ClipCounters* ctr) {
  __shared__ unsigned s_drop;
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (threadIdx.x == 0) s_drop = 0u;
  __syncthreads();
  bool drop = false;
  if (t < nt) {
    int v[3];
    clip_tri(tris, t, v);
    if ((unsigned)v[0] >= nv || (unsigned)v[1] >= nv || (unsigned)v[2] >= nv) {
      ctr->bad_ids = 1u;
      piece_flags[2 * (size_t)t] = piece_flags[2 * (size_t)t + 1] = 0;
      cut[t] = 0;
    } else {
      const unsigned k = clip_corners(keep_v, v);
      const bool x = k != 0u && k != 7u;               // two crossed edges, else none
      const int n = __popc(k) + (x ? 2 : 0);           // tokens of the walk: 0, 3 or 4
      piece_flags[2 * (size_t)t] = n >= 3 ? 1 : 0;
      piece_flags[2 * (size_t)t + 1] = n == 4 ? 1 : 0;
      cut[t] = x ? 1 : 0;
      drop = k == 0u;
    }
  }
  // dropped triangles: summed per warp, then per block, then one global atomic per block
  const unsigned b = __ballot_sync(0xffffffffu, drop);
  if (b && lane_id() == 0u) atomicAdd(&s_drop, (unsigned)__popc(b));
  __syncthreads();
  if (threadIdx.x == 0 && s_drop) atomicAdd(&ctr->n_dropped, s_drop);
}

// the undirected key of the crossed edge (v_i, v_i+1)
template <int i>
__device__ __forceinline__ unsigned long long clip_edge(const int v[3]) {
  return edge_key(v[i], v[(i + 1) % 3]);
}

__global__ void __launch_bounds__(256) k_clip_edges(const int* __restrict__ tris, unsigned nt, const uint8_t* __restrict__ cut,
                                                    const uint8_t* __restrict__ keep_v, EdgeSlot* tab, size_t mask) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !cut[t]) return;
  int v[3];
  clip_tri(tris, t, v);
  const unsigned k = clip_corners(keep_v, v);
  if (edge_changes(k, 0)) atomicMin(&edge_slot(tab, mask, clip_edge<0>(v), true)->tri, (int)t);
  if (edge_changes(k, 1)) atomicMin(&edge_slot(tab, mask, clip_edge<1>(v), true)->tri, (int)t);
  if (edge_changes(k, 2)) atomicMin(&edge_slot(tab, mask, clip_edge<2>(v), true)->tri, (int)t);
}

// the two crossed edges of a cut triangle in walk order: their positions i0 < i1
__device__ __forceinline__ void clip_crossed(unsigned k, int& i0, int& i1) {
  i0 = edge_changes(k, 0) ? 0 : 1;
  i1 = edge_changes(k, 2) ? 2 : 1;
}

__device__ __forceinline__ unsigned long long clip_edge_at(const int v[3], int i) {
  return i == 0 ? clip_edge<0>(v) : i == 1 ? clip_edge<1>(v) : clip_edge<2>(v);
}

__global__ void __launch_bounds__(256) k_clip_own(const int* __restrict__ tris, unsigned nt, const uint8_t* __restrict__ cut,
                                                  const uint32_t* __restrict__ cut_idx, const uint8_t* __restrict__ keep_v,
                                                  EdgeSlot* tab, size_t mask, uint8_t* __restrict__ eflags) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !cut[t]) return;
  int v[3], i0, i1;
  clip_tri(tris, t, v);
  clip_crossed(clip_corners(keep_v, v), i0, i1);
  const unsigned long long k0 = clip_edge_at(v, i0), k1 = clip_edge_at(v, i1);
  const size_t c = (size_t)cut_idx[t] * 2;
  eflags[c] = edge_slot(tab, mask, k0, false)->tri == (int)t ? 1 : 0;
  eflags[c + 1] = k1 != k0 && edge_slot(tab, mask, k1, false)->tri == (int)t ? 1 : 0;
}

// the new vertex of crossed edge {a, b} (one end kept) at ordinal o
template <typename G>
__device__ __forceinline__ void clip_new_vertex(const ClipSrc<G>& src, const G* __restrict__ verts, const G* __restrict__ normals,
                                                const unsigned long long* __restrict__ keys, const uint8_t* __restrict__ lowmin,
                                                const G* __restrict__ values, int ncomp, const uint8_t* __restrict__ keep_v,
                                                double offset, int a, int b, size_t o, const ClipRows& out) {
  const double sa = src((unsigned)a), sb = src((unsigned)b);
  const bool a_low = !(sa >= offset);
  const int lo = a_low ? a : b, hi = a_low ? b : a, ke = keep_v[a] ? a : b;
  const double sl = a_low ? sa : sb, sh = a_low ? sb : sa;
  sec_point(verts, lo, hi, sl, sh, offset, (G*)out.verts + o * 3);
  const double t = __ddiv_rn(__dsub_rn(offset, sl), __dsub_rn(sh, sl));
  if (normals) {
    double m[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double na = (double)normals[(size_t)lo * 3 + c], nb = (double)normals[(size_t)hi * 3 + c];
      m[c] = __dadd_rn(na, __dmul_rn(t, __dsub_rn(nb, na)));
    }
    const double len2 = __dadd_rn(__dadd_rn(__dmul_rn(m[0], m[0]), __dmul_rn(m[1], m[1])), __dmul_rn(m[2], m[2]));
    G* n = (G*)out.normals + o * 3;
    if (len2 == 0.0) {
#pragma unroll
      for (int c = 0; c < 3; ++c) n[c] = normals[(size_t)ke * 3 + c];
    } else {
      const double len = __dsqrt_rn(len2);
#pragma unroll
      for (int c = 0; c < 3; ++c) n[c] = (G)__ddiv_rn(m[c], len);
    }
  }
  if (keys) {
    out.keys[o] = keys[ke];
    out.lowmin[o] = lowmin[ke];
  }
  if (values) {
    G* w = (G*)out.values + o * ncomp;
    for (int c = 0; c < ncomp; ++c) {
      const double va = (double)values[(size_t)lo * ncomp + c], vb = (double)values[(size_t)hi * ncomp + c];
      w[c] = (G)__dadd_rn(va, __dmul_rn(t, __dsub_rn(vb, va)));
    }
  }
}

template <typename G>
__global__ void __launch_bounds__(256) k_clip_verts(ClipSrc<G> src, const int* __restrict__ tris, unsigned nt,
                                                    const uint8_t* __restrict__ cut, const uint32_t* __restrict__ cut_idx,
                                                    const uint8_t* __restrict__ keep_v, EdgeSlot* tab, size_t mask,
                                                    const uint8_t* __restrict__ eflags, const uint32_t* __restrict__ eidx,
                                                    double offset, const G* __restrict__ verts, const G* __restrict__ normals,
                                                    const unsigned long long* __restrict__ keys, const uint8_t* __restrict__ lowmin,
                                                    const G* __restrict__ values, int ncomp, ClipRows out) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !cut[t]) return;
  const size_t c = (size_t)cut_idx[t] * 2;
  if (!eflags[c] && !eflags[c + 1]) return;
  int v[3], i0, i1;
  clip_tri(tris, t, v);
  clip_crossed(clip_corners(keep_v, v), i0, i1);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    if (!eflags[c + j]) continue;
    const int i = j ? i1 : i0;
    const int a = i == 0 ? v[0] : i == 1 ? v[1] : v[2];
    const int b = i == 0 ? v[1] : i == 1 ? v[2] : v[0];
    const unsigned o = eidx[c + j];
    edge_slot(tab, mask, edge_key(a, b), false)->pad = (int)o;
    clip_new_vertex(src, verts, normals, keys, lowmin, values, ncomp, keep_v, offset, a, b, o, out);
  }
}

__global__ void __launch_bounds__(256) k_clip_tris(const int* __restrict__ tris, unsigned nt, const uint8_t* __restrict__ keep_v,
                                                   const uint32_t* __restrict__ idx_v, unsigned n_kept, EdgeSlot* tab, size_t mask,
                                                   const uint8_t* __restrict__ piece_flags, const uint32_t* __restrict__ piece_idx,
                                                   int* __restrict__ dst) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !piece_flags[2 * (size_t)t]) return;
  int v[3];
  clip_tri(tris, t, v);
  const unsigned k = clip_corners(keep_v, v);
  int p[4] = {0, 0, 0, 0}, n = 0;                      // the polygon's vertex ids, in walk order
  auto push = [&](int id) {
    p[3] = n == 3 ? id : p[3];
    p[2] = n == 2 ? id : p[2];
    p[1] = n == 1 ? id : p[1];
    p[0] = n == 0 ? id : p[0];
    ++n;
  };
  auto crossing = [&](unsigned long long key) { return (int)n_kept + edge_slot(tab, mask, key, false)->pad; };
  if (k & 1u) push((int)idx_v[v[0]]);
  if (edge_changes(k, 0)) push(crossing(clip_edge<0>(v)));
  if (k & 2u) push((int)idx_v[v[1]]);
  if (edge_changes(k, 1)) push(crossing(clip_edge<1>(v)));
  if (k & 4u) push((int)idx_v[v[2]]);
  if (edge_changes(k, 2)) push(crossing(clip_edge<2>(v)));
  // the fan from p[0]: (p0, p1, p2), and (p0, p2, p3) for a quad
  int* o = dst + (size_t)piece_idx[2 * (size_t)t] * 3;
  o[0] = p[0];
  o[1] = p[1];
  o[2] = p[2];
  if (n == 4) {
    o = dst + (size_t)piece_idx[2 * (size_t)t + 1] * 3;
    o[0] = p[0];
    o[1] = p[2];
    o[2] = p[3];
  }
}

template <typename G>
int clip_typed(ctr_ctx* ctx, const ctr_clip_params* cp, ctr_clip_counts* out) {
  cudaStream_t st = ctx->stream;
  const uint32_t fl = ctx->last_flags;
  const size_t nV = (size_t)ctx->last_counts[0], nT = (size_t)ctx->last_counts[1], gsz = sizeof(G);
  const bool values = ctx->attr_ncomp > 0 && ctx->attr_gen == ctx->mesh_gen;   // carried: made on this very mesh
  const int ncomp = values ? ctx->attr_ncomp : 0;
  const bool plane = cp->source == CTR_CLIP_PLANE;
  if (!plane && !values)
    return ctr_fail(ctx, CTR_ERR_STATE, "a value clip needs a ctr_mt3d_interpolate on the mesh as it stands: interpolate first");
  if (!plane && cp->component >= ncomp) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "component must be in [0, ncomp) of the last interpolation");
  ClipSrc<G> src;
  src.p = plane ? (const G*)ctx->verts.p : (const G*)ctx->aux[AUX_VALUES].p;
  src.stride = plane ? 3 : ncomp;
  src.comp = plane ? 0 : cp->component;
  src.plane = plane;
  src.P = SecPlanes{cp->normal[0], cp->normal[1], cp->normal[2], nullptr, 0, 0};
  const double off = cp->offset;
  // ---- phase 1: sides, pieces, kept vertices, cut triangles
  const int tiles_p = (int)((2 * nT + SC_TILE - 1) / SC_TILE), tiles_v = (int)((nV + SC_TILE - 1) / SC_TILE),
            tiles_c = (int)((nT + SC_TILE - 1) / SC_TILE);
  const size_t scan_bytes = 64 + ((size_t)tiles_p + tiles_v + tiles_c + 3) * 8;
  char* scan;
  uint8_t *keep_v, *piece_flags, *cut;
  uint32_t *idx_v, *piece_idx, *cut_idx;
  int rc;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH0], [&](ctr_carve& c) {
         c(scan, scan_bytes);
         c(keep_v, nV + 8);
         c(idx_v, nV * 4 + 4);
         c(piece_flags, 2 * nT + 8);
         c(piece_idx, 2 * nT * 4 + 4);
         c(cut, nT + 8);
         c(cut_idx, nT * 4 + 4);
       })))
    return rc;
  ClipCounters* ctr = (ClipCounters*)scan;
  unsigned long long* st_p = (unsigned long long*)(scan + 64);
  unsigned long long* st_v = st_p + tiles_p + 1;
  unsigned long long* st_c = st_v + tiles_v + 1;
  CTR_CUDA(ctx, cudaMemsetAsync(scan, 0, scan_bytes, st));
  const int* tris = (const int*)ctx->tris.p;
  const unsigned vb = (unsigned)((nV + 255) / 256), tb = (unsigned)((nT + 255) / 256);
  if (nV) {
    k_clip_side<G><<<vb, 256, 0, st>>>(src, (unsigned)nV, off, cp->side, keep_v, ctr);
    k_flag_scan<<<tiles_v, SC_THREADS, 0, st>>>(keep_v, (unsigned)nV, idx_v, st_v, &ctr->ticket[1], &ctr->total[1], tiles_v);
    ctx->launches += 2;
  }
  if (nT) {
    k_clip_count<<<tb, 256, 0, st>>>(tris, (unsigned)nT, (unsigned)nV, keep_v, piece_flags, cut, ctr);
    k_flag_scan<<<tiles_p, SC_THREADS, 0, st>>>(piece_flags, (unsigned)(2 * nT), piece_idx, st_p, &ctr->ticket[0], &ctr->total[0],
                                                tiles_p);
    k_flag_scan<<<tiles_c, SC_THREADS, 0, st>>>(cut, (unsigned)nT, cut_idx, st_c, &ctr->ticket[2], &ctr->total[2], tiles_c);
    ctx->launches += 3;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  ClipCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.bad_ids) return fail_shifted_ids(ctx);
  if (h.nan) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "a vertex's side value is NaN");
  const size_t n_kept = (size_t)h.total[1], newT = (size_t)h.total[0], n_cut = (size_t)h.total[2];
  out->n_verts = (int64_t)nV;
  out->n_tris = (int64_t)nT;
  if (n_kept == nV) return 0;                          // every vertex kept: no triangle is cut or dropped, nothing changes
  // ---- phase 2: the crossed edges and their new vertices
  size_t nslots = 256;
  while (nslots < 8 * n_cut) nslots <<= 1;
  const size_t ne = 2 * n_cut;                         // crossed-edge slots of the cut triangles, and the new-vertex bound
  const int tiles_e = (int)((ne + SC_TILE - 1) / SC_TILE);
  const size_t vrow = std::max<size_t>(3 * gsz, (size_t)ncomp * gsz);
  EdgeSlot* tab;
  uint8_t *eflags, *new_low;
  uint32_t* eidx;
  unsigned long long *st_e, *new_keys;
  void *new_verts, *new_nrm, *new_vals, *stage;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH1], [&](ctr_carve& c) {
         c(tab, nslots * sizeof(EdgeSlot));
         c(st_e, ((size_t)tiles_e + 1) * 8);
         c(eflags, ne + 8);
         c(eidx, ne * 4 + 4);
         c(new_verts, ne * 3 * gsz);
         c(new_nrm, ne * 3 * gsz);
         c(new_keys, ne * 8);
         c(new_low, ne);
         c(new_vals, ne * (size_t)ncomp * gsz);
         c(stage, std::max(n_kept * vrow, newT * 12) + 16);
       })))
    return rc;
  const size_t mask = nslots - 1;
  k_o_init<<<ctx->sm_count * 8, 256, 0, st>>>(tab, nslots, nullptr, 0u, nullptr, nullptr);
  ctx->launches++;
  if (n_cut) {
    CTR_CUDA(ctx, cudaMemsetAsync(st_e, 0, ((size_t)tiles_e + 1) * 8, st));
    k_clip_edges<<<tb, 256, 0, st>>>(tris, (unsigned)nT, cut, keep_v, tab, mask);
    k_clip_own<<<tb, 256, 0, st>>>(tris, (unsigned)nT, cut, cut_idx, keep_v, tab, mask, eflags);
    k_flag_scan<<<tiles_e, SC_THREADS, 0, st>>>(eflags, (unsigned)ne, eidx, st_e, &ctr->ticket[3], &ctr->total[3], tiles_e);
    ctx->launches += 3;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  unsigned long long n_new = 0;
  CTR_CUDA(ctx, cudaMemcpyAsync(&n_new, &ctr->total[3], 8, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const size_t newV = n_kept + (size_t)n_new;
  if (newV > 0x7fffffffull || newT > 0x7fffffffull)
    return ctr_fail(ctx, CTR_ERR_OVERFLOW, "the clipped mesh would have 2^31 or more vertices or triangles");
  // ---- the writes
  mesh_edited(ctx, EDIT_CLIP);
  const bool nrm = fl & CTR_WANT_NORMALS, key = fl & CTR_WANT_KEYS;
  const size_t vbytes = (size_t)ncomp * gsz;
  if ((rc = ctr_grow_keep(ctx, ctx->verts, newV * 3 * gsz, nV * 3 * gsz))) return rc;
  if (nrm && (rc = ctr_grow_keep(ctx, ctx->normals, newV * 3 * gsz, nV * 3 * gsz))) return rc;
  if (key && (rc = ctr_grow_keep(ctx, ctx->keys, newV * 8, nV * 8))) return rc;
  if (key && (rc = ctr_grow_keep(ctx, ctx->lowmin, newV, nV))) return rc;
  if (values && (rc = ctr_grow_keep(ctx, ctx->aux[AUX_VALUES], newV * vbytes, nV * vbytes))) return rc;
  if ((rc = ctr_grow_keep(ctx, ctx->tris, newT * 12, nT * 12))) return rc;
  tris = (const int*)ctx->tris.p;
  src.p = plane ? (const G*)ctx->verts.p : (const G*)ctx->aux[AUX_VALUES].p;
  if (n_new) {
    const ClipRows rows = {new_verts, new_nrm, new_keys, new_low, new_vals};
    k_clip_verts<G><<<tb, 256, 0, st>>>(src, tris, (unsigned)nT, cut, cut_idx, keep_v, tab, mask, eflags, eidx, off,
                                        (const G*)ctx->verts.p, nrm ? (const G*)ctx->normals.p : nullptr,
                                        key ? (const unsigned long long*)ctx->keys.p : nullptr,
                                        key ? (const uint8_t*)ctx->lowmin.p : nullptr,
                                        values ? (const G*)ctx->aux[AUX_VALUES].p : nullptr, ncomp, rows);
    ctx->launches++;
  }
  // kept rows compacted through the staging rows, then the new rows behind them
  auto rows = [&](void* p, const void* fresh, size_t row_bytes) -> int {
    if (nV) {
      k_sel_rows<<<vb, 256, 0, st>>>((const uint32_t*)p, (uint32_t*)stage, keep_v, idx_v, (unsigned)nV, (int)(row_bytes / 4));
      ctx->launches++;
    }
    if (n_kept) CTR_CUDA(ctx, cudaMemcpyAsync(p, stage, n_kept * row_bytes, cudaMemcpyDeviceToDevice, st));
    if (n_new) CTR_CUDA(ctx, cudaMemcpyAsync((char*)p + n_kept * row_bytes, fresh, n_new * row_bytes, cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  if ((rc = rows(ctx->verts.p, new_verts, 3 * gsz))) return rc;
  if (nrm && (rc = rows(ctx->normals.p, new_nrm, 3 * gsz))) return rc;
  if (key && (rc = rows(ctx->keys.p, new_keys, 8))) return rc;
  if (key && (rc = rows(ctx->lowmin.p, new_low, 1))) return rc;
  if (values && (rc = rows(ctx->aux[AUX_VALUES].p, new_vals, vbytes))) return rc;
  if (newT) {
    k_clip_tris<<<tb, 256, 0, st>>>(tris, (unsigned)nT, keep_v, idx_v, (unsigned)n_kept, tab, mask, piece_flags, piece_idx,
                                    (int*)stage);
    ctx->launches++;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->tris.p, stage, newT * 12, cudaMemcpyDeviceToDevice, st));
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  if (values) {
    ctx->attr_rows = newV;
    ctx->attr_gen = ctx->mesh_gen;
  }
  out->n_verts = (int64_t)newV;
  out->n_tris = (int64_t)newT;
  out->n_new_verts = (int64_t)n_new;
  out->n_cut_tris = (int64_t)n_cut;
  out->n_dropped_tris = (int64_t)h.n_dropped;
  return 0;
}
