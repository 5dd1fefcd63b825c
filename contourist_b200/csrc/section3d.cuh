// Plane sections of the 3D device mesh (ctr_mt3d_section), like VTK's vtkCutter on polydata.
//
// Included into mesh3d.cu after components3d.cuh and smooth3d.cuh, inside its anonymous namespace.  The definition is
// oracle/mt3d_section.py:section.  Plane l is {x : n . x == offsets[l]}; a vertex is high for it when
// s = (n0 x + n1 y) + n2 z >= offsets[l] (fp64, every operation rounded on its own).
//   k_m_init / k_m_edges : the components pass's edge table: every undirected edge once, triangle ids checked;
//   k_sec_count : per triangle the planes it crosses, [first, first + count), by binary search of its side range over
//                 the offsets (every 2^shift-th offset staged in shared memory, the last steps in global memory);
//   k_s_scan    : (smoothing's) counts -> the first segment of every triangle, with the exact 64-bit total;
//   k_sec_emit  : per triangle and plane one segment: plane, crossing edges (start edge first: the one the corner walk
//                 takes from high to low), points; per dart its edge key (the order) and (plane, edge slot) (the vertex);
//   darts.cuh   : k_p_insert (junction planes flagged) ... k_p_mark, scan_u32: the polylines;
//   k_sec_kill  : the segments of junction planes made dead before the successors are taken (they are not chained);
//   k_sec_points: descriptors and points in their final order, reversed where the first segment runs from its point 1
//                 to its point 0; darts that run against the first one clear the polyline's consistent flag;
//   k_sec_measure : length and area per polyline, one thread per point, sums combined over the warp's lanes first.
// Scratch: AUX_SCRATCH0 edge table, AUX_SCRATCH1 per-triangle counts / per-point polyline, AUX_SCRATCH2 chaining,
// AUX_SCRATCH3 counters, look-back words and offsets, AUX_SCRATCH4 per-dart keys.  Results: AUX_SECTION_SEGS,
// AUX_SECTION_POLYS; the component results and vertex values are not touched.

#include "darts.cuh"

constexpr int SEC_THREADS = 256;
constexpr int SEC_STAGE = 4096;                       // offsets staged per block (32 KiB)

struct SecPlanes {
  double n0, n1, n2;
  const double* __restrict__ off;
  int np;
  int shift;                                          // off[k << shift] staged, k < ceil(np / 2^shift) <= SEC_STAGE
};

__device__ __forceinline__ double sec_side(const SecPlanes& P, double x, double y, double z) {
  return __dadd_rn(__dadd_rn(__dmul_rn(P.n0, x), __dmul_rn(P.n1, y)), __dmul_rn(P.n2, z));
}

// number of offsets <= x
__device__ __forceinline__ unsigned sec_upper(const double* s_off, int ns, const SecPlanes& P, double x) {
  int lo = 0, hi = ns;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (s_off[m] <= x) lo = m + 1;
    else hi = m;
  }
  if (lo == 0) return 0u;
  unsigned u = ((unsigned)(lo - 1) << P.shift) + 1u;
  const unsigned e = min((unsigned)lo << P.shift, (unsigned)P.np);
  while (u < e && P.off[u] <= x) ++u;
  return u;
}

template <typename G>
__device__ __forceinline__ void sec_sides(const G* __restrict__ verts, const int v[3], const SecPlanes& P, double s[3]) {
#pragma unroll
  for (int q = 0; q < 3; ++q)
    s[q] = sec_side(P, (double)verts[(size_t)v[q] * 3], (double)verts[(size_t)v[q] * 3 + 1], (double)verts[(size_t)v[q] * 3 + 2]);
}

// grid-stride, so that the staging is paid once per resident block
template <typename G>
__global__ void __launch_bounds__(SEC_THREADS) k_sec_count(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                           unsigned nv, SecPlanes P, unsigned* __restrict__ cnt,
                                                           unsigned* __restrict__ first) {
  __shared__ double s_off[SEC_STAGE];
  const int ns = (P.np + (1 << P.shift) - 1) >> P.shift;
  for (int k = threadIdx.x; k < ns; k += blockDim.x) s_off[k] = P.off[(size_t)k << P.shift];
  __syncthreads();
  for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
    if ((unsigned)v[0] >= nv || (unsigned)v[1] >= nv || (unsigned)v[2] >= nv) {   // k_m_edges flags it; the host stops
      cnt[t] = 0u;
      first[t] = 0u;
      continue;
    }
    double s[3];
    sec_sides(verts, v, P, s);
    // crossed: some corner high (s >= d) and some low (s < d), i.e. smin < d <= smax
    const unsigned lo = sec_upper(s_off, ns, P, fmin(s[0], fmin(s[1], s[2])));
    const unsigned hi = sec_upper(s_off, ns, P, fmax(s[0], fmax(s[1], s[2])));
    cnt[t] = hi - lo;
    first[t] = lo;
  }
}

// crossing of edge {a, b}, a the low end: t = (d - s_a) / (s_b - s_a), p = p_a + t (p_b - p_a), rounded once to G
template <typename G>
__device__ __forceinline__ void sec_point(const G* __restrict__ verts, int a, int b, double sa, double sb, double d, G* out) {
  const double t = __ddiv_rn(__dsub_rn(d, sa), __dsub_rn(sb, sa));
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double pa = (double)verts[(size_t)a * 3 + c], pb = (double)verts[(size_t)b * 3 + c];
    out[c] = (G)__dadd_rn(pa, __dmul_rn(t, __dsub_rn(pb, pa)));
  }
}

template <typename G>
__global__ void __launch_bounds__(SEC_THREADS) k_sec_emit(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                          SecPlanes P, const unsigned* __restrict__ seg_off,
                                                          const unsigned* __restrict__ first, EdgeSlot* etab, size_t mask,
                                                          int* __restrict__ plane, int* __restrict__ edges, G* __restrict__ pts,
                                                          unsigned long long* __restrict__ keys, unsigned long long* __restrict__ vid) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const unsigned o = seg_off[t], c = seg_off[t + 1] - o;
  if (!c) return;
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
  double s[3];
  sec_sides(verts, v, P, s);
  const unsigned l0 = first[t];
  for (unsigned i = 0; i < c; ++i) {
    const unsigned l = l0 + i, g = o + i;
    const double d = P.off[l];
    const bool h[3] = {s[0] >= d, s[1] >= d, s[2] >= d};
    // the walk v0 -> v1 -> v2 -> v0 takes one edge from high to low (start) and one from low to high (end)
    int ks = 0, ke = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (h[k] && !h[(k + 1) % 3]) ks = k;
      if (!h[k] && h[(k + 1) % 3]) ke = k;
    }
    // (selects, not indexing with ks / ke: that would put v[] and s[] on the stack)
    auto pick = [](const auto* a, int k) { return k == 0 ? a[0] : k == 1 ? a[1] : a[2]; };
    const int ks1 = ks == 2 ? 0 : ks + 1, ke1 = ke == 2 ? 0 : ke + 1;
    const int sl = pick(v, ks1), sh = pick(v, ks);            // start edge: low end, high end
    const int el = pick(v, ke), eh = pick(v, ke1);            // end edge
    const double ssl = pick(s, ks1), ssh = pick(s, ks), sel = pick(s, ke), seh = pick(s, ke1);
    plane[g] = (int)l;
    const int e[4] = {min(sl, sh), max(sl, sh), min(el, eh), max(el, eh)};
    reinterpret_cast<int4*>(edges)[g] = make_int4(e[0], e[1], e[2], e[3]);
    sec_point(verts, sl, sh, ssl, ssh, d, pts + (size_t)g * 6);
    sec_point(verts, el, eh, sel, seh, d, pts + (size_t)g * 6 + 3);
    keys[2 * (size_t)g] = ((unsigned long long)(unsigned)e[0] << 32) | (unsigned)e[1];
    keys[2 * (size_t)g + 1] = ((unsigned long long)(unsigned)e[2] << 32) | (unsigned)e[3];
    // the vertex: (plane, edge slot); slots < 2^34, planes < 2^16
    vid[2 * (size_t)g] = ((unsigned long long)l << 40) | (size_t)(edge_slot(etab, mask, edge_key(sl, sh), false) - etab);
    vid[2 * (size_t)g + 1] = ((unsigned long long)l << 40) | (size_t)(edge_slot(etab, mask, edge_key(el, eh), false) - etab);
  }
}

// the vertex of a dart's tail is (plane, edge slot); contours are ordered by edge key (min << 32 | max)
struct Vert3 {
  const unsigned long long* __restrict__ vid;
  const int* __restrict__ plane;
  unsigned* jplane;                                   // per plane: 1 = junction
  __device__ __forceinline__ unsigned long long id(const unsigned long long* __restrict__, unsigned d) const { return vid[d]; }
  __device__ __forceinline__ unsigned long long prio(const unsigned long long* __restrict__ keys, unsigned d) const { return keys[d]; }
  __device__ __forceinline__ void junction(unsigned d, PolyCounters* ctr) const {
    if (atomicExch(&jplane[plane[d >> 1]], 1u) == 0u) atomicAdd(&ctr->junction_levels, 1ull);
  }
};

__global__ void k_sec_kill(unsigned ns, const int* __restrict__ plane, const unsigned* __restrict__ jplane,
                           unsigned long long* __restrict__ keys) {
  const unsigned s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ns || !jplane[plane[s]]) return;
  keys[2 * (size_t)s + 1] = keys[2 * (size_t)s];
}

// per dart of a kept polyline: the first dart writes the descriptor and point 0, every kept dart the point it arrives
// at, at its final index.  Row 2s+q of the segment points is end q of segment s, the end dart 2s+q leaves.
template <typename G>
__global__ void k_sec_points(unsigned nd, const unsigned long long* __restrict__ keys, const int* __restrict__ plane,
                             const G* __restrict__ seg_pts, const unsigned* __restrict__ start, const unsigned* __restrict__ dist,
                             const unsigned* __restrict__ npts, const unsigned* __restrict__ off, const unsigned* __restrict__ pidx,
                             G* __restrict__ pts, unsigned* __restrict__ poly_of_point, int* __restrict__ p_plane,
                             uint8_t* __restrict__ p_flags, unsigned long long* __restrict__ p_key, unsigned* __restrict__ p_off,
                             unsigned* __restrict__ p_len, uint8_t* __restrict__ bad) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const unsigned sd = start[d];
  const unsigned n = npts[sd];
  if (!n) return;
  const unsigned len = dist[sd] + 1u;
  const unsigned p = len - 1u - dist[d];                      // position of this dart behind the first one
  const bool open = start[sd ^ 1u] == sd;
  const unsigned m = open ? n - 1u : n;                       // segments
  if (p >= m) return;                                         // the way back of an open tour
  const bool rev = sd & 1u;                                   // the first segment runs from its point 1 to point 0
  const unsigned o = off[sd], pl = pidx[sd];
  auto at = [&](unsigned i) { return o + (!rev ? i : open ? n - 1u - i : (i ? n - i : 0u)); };
  if (d == sd) {
    p_plane[pl] = plane[d >> 1];
    p_flags[pl] = open ? 0 : 1;
    p_off[pl] = o;
    p_len[pl] = n;
    if (!(rev && open)) p_key[pl] = keys[d];
    const unsigned q = at(0);
#pragma unroll
    for (int c = 0; c < 3; ++c) pts[(size_t)q * 3 + c] = seg_pts[(size_t)d * 3 + c];
    poly_of_point[q] = pl;
  }
  if ((d ^ sd) & 1u) bad[pl] = 1;                            // runs against the first segment
  if (p + 1u < n) {                                          // open: every kept dart; closed: all but the last
    const unsigned q = at(p + 1u), h = d ^ 1u;
#pragma unroll
    for (int c = 0; c < 3; ++c) pts[(size_t)q * 3 + c] = seg_pts[(size_t)h * 3 + c];
    poly_of_point[q] = pl;
    if (rev && open && p + 1u == m) p_key[pl] = keys[h];      // reversed open polyline: starts at the other end
  }
}

// length = sum |p_{i+1} - p_i| (closing segment included), area = 1/2 sum ((p_i - p_0) x (p_{i+1} - p_0)) . u
template <typename G>
__global__ void __launch_bounds__(SEC_THREADS) k_sec_measure(unsigned np_, const G* __restrict__ pts, const unsigned* __restrict__ poly_of_point,
                                                             const unsigned* __restrict__ p_off, const unsigned* __restrict__ p_len,
                                                             uint8_t* p_flags, const uint8_t* __restrict__ bad, double u0,
                                                             double u1, double u2, double* __restrict__ meas) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = i < np_;
  const unsigned act = __ballot_sync(0xffffffffu, in);
  if (!in) return;
  const unsigned pl = poly_of_point[i], o = p_off[pl], n = p_len[pl], j = i - o;
  const bool closed = p_flags[pl] & 1u;                      // (bit 0 is not written below)
  double len = 0.0, area = 0.0;
  if (j + 1u < n || closed) {
    const unsigned k = j + 1u < n ? i + 1u : o;
    double a[3], b[3], p0[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      p0[c] = (double)pts[(size_t)o * 3 + c];
      a[c] = (double)pts[(size_t)i * 3 + c] - p0[c];
      b[c] = (double)pts[(size_t)k * 3 + c] - p0[c];
    }
    const double dx = b[0] - a[0], dy = b[1] - a[1], dz = b[2] - a[2];
    len = sqrt(dx * dx + dy * dy + dz * dz);
    const double cx = a[1] * b[2] - a[2] * b[1], cy = a[2] * b[0] - a[0] * b[2], cz = a[0] * b[1] - a[1] * b[0];
    area = 0.5 * (cx * u0 + cy * u1 + cz * u2);
  }
  const unsigned peers = __match_any_sync(act, pl);
  len = peer_reduce(peers, len, MAdd());
  area = peer_reduce(peers, area, MAdd());
  if ((__ffs(peers) - 1) == (int)lane_id()) {
    atomicAdd(&meas[2 * (size_t)pl], len);
    atomicAdd(&meas[2 * (size_t)pl + 1], area);
  }
  if (j == 0 && !bad[pl]) p_flags[pl] = closed ? 3 : 2;
}

// the pieces of the two result buffers; the fetches carve them again from the stored counts
struct SecSegs {
  int* plane;
  int* edges;
  char* pts;
  unsigned* jplane;
  template <typename C>
  void carve(C& c, size_t S, size_t gsz, size_t nplanes) {
    c(plane, S * 4);
    c(edges, S * 16);
    c(pts, S * 6 * gsz);
    c(jplane, nplanes * 4);
  }
};
struct SecPolys {
  unsigned long long* key;
  int* plane;
  unsigned *off, *len;
  uint8_t* flags;
  double* meas;
  char* pts;
  template <typename C>
  void carve(C& c, size_t P, size_t N, size_t gsz) {
    c(key, P * 8);
    c(plane, P * 4);
    c(off, P * 4);
    c(len, P * 4);
    c(flags, P);
    c(meas, P * 16);
    c(pts, N * 3 * gsz);
  }
};

template <typename G>
int section_typed(ctr_ctx* ctx, const ctr_section_params* sp, ctr_section_counts* out) {
  const unsigned nt = (unsigned)ctx->last_counts[1], nv = (unsigned)ctx->last_counts[0];
  const size_t nplanes = (size_t)sp->nplanes, gsz = sizeof(G);
  cudaStream_t st = ctx->stream;
  int rc;
  SecSegs sg;
  auto finish = [&](int64_t S, int64_t P, int64_t N, int64_t J) {
    ctx->sect_count[0] = S;
    ctx->sect_count[1] = P;
    ctx->sect_count[2] = N;
    ctx->sect_count[3] = J;
    ctx->sect_nplanes = sp->nplanes;
    out->n_segments = S;
    out->n_polylines = P;
    out->n_points = N;
    out->n_junction_planes = J;
    return 0;
  };
  if (nt == 0) {
    if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SECTION_SEGS], [&](ctr_carve& c) { sg.carve(c, 0, gsz, nplanes); }))) return rc;
    CTR_CUDA(ctx, cudaMemsetAsync(sg.jplane, 0, nplanes * 4, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    return finish(0, 0, 0, 0);
  }
  // ---- edge table, crossings per triangle, their scan; one host wait for the total
  const size_t nslots = edge_slots(nt);
  const unsigned blocks = (nt + SEC_THREADS - 1) / SEC_THREADS;   // also the look-back tiles of k_s_scan
  DevBuf& b_etab = ctx->aux[AUX_SCRATCH0];
  DevBuf& b_tri = ctx->aux[AUX_SCRATCH1];
  DevBuf& b_ctr = ctx->aux[AUX_SCRATCH3];
  const size_t o_off = (64 + (size_t)blocks * 8 + 255) & ~(size_t)255;
  if ((rc = ctr_ensure(ctx, b_etab, nslots * sizeof(EdgeSlot)))) return rc;
  if ((rc = ctr_ensure(ctx, b_tri, ((size_t)nt + 1) * 12))) return rc;
  if ((rc = ctr_ensure(ctx, b_ctr, o_off + nplanes * 8))) return rc;
  EdgeSlot* etab = (EdgeSlot*)b_etab.p;
  unsigned* cnt = (unsigned*)b_tri.p;                 // counts, then the scan's cursors
  unsigned* seg_off = cnt + nt + 1;                   // first segment of every triangle, [nt] = total
  unsigned* first = seg_off + nt + 1;                 // first plane crossed
  SCounters* ctr = (SCounters*)b_ctr.p;               // k_m_edges' bad-id flag; k_s_scan's ticket and total
  unsigned long long* status = (unsigned long long*)((char*)b_ctr.p + 64);
  double* d_off = (double*)((char*)b_ctr.p + o_off);
  CTR_CUDA(ctx, cudaMemsetAsync(b_ctr.p, 0, 64 + (size_t)blocks * 8, st));
  CTR_CUDA(ctx, cudaMemcpyAsync(d_off, sp->offsets, nplanes * 8, cudaMemcpyHostToDevice, st));
  SecPlanes P{sp->normal[0], sp->normal[1], sp->normal[2], d_off, sp->nplanes, 0};
  while (((P.np + (1 << P.shift) - 1) >> P.shift) > SEC_STAGE) ++P.shift;
  const G* verts = (const G*)ctx->verts.p;
  const int* tris = (const int*)ctx->tris.p;
  // the (component, vertex) table of k_m_init aliases the edge table: this pass does not read slot.tri
  k_m_init<<<ctx->sm_count * 8, 256, 0, st>>>(etab, etab, nslots, nullptr, 0u);
  k_m_edges<<<blocks, M_THREADS, 0, st>>>(tris, nt, nv, etab, nslots - 1, &ctr->m);
  k_sec_count<G><<<std::min(blocks, (unsigned)ctx->sm_count * 4), SEC_THREADS, 0, st>>>(verts, tris, nt, nv, P, cnt, first);
  k_s_scan<<<blocks, S_THREADS, 0, st>>>(cnt, nt, seg_off, status, ctr, (int)blocks);
  ctx->launches += 4;
  CTR_CUDA(ctx, cudaGetLastError());
  SCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.m.bad) return fail_shifted_ids(ctx);
  if (h.m.total >= (1ull << 31)) return ctr_fail(ctx, CTR_ERR_OVERFLOW, "2^31 or more section segments: use fewer planes");
  const size_t S = (size_t)h.m.total, nd = 2 * S;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SECTION_SEGS], [&](ctr_carve& c) { sg.carve(c, S, gsz, nplanes); }))) return rc;
  CTR_CUDA(ctx, cudaMemsetAsync(sg.jplane, 0, nplanes * 4, st));
  if (S == 0) {
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    return finish(0, 0, 0, 0);
  }
  // ---- segments
  unsigned long long *keys, *vid;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH4], [&](ctr_carve& c) {
         c(keys, nd * 8);
         c(vid, nd * 8);
       })))
    return rc;
  k_sec_emit<G><<<blocks, SEC_THREADS, 0, st>>>(verts, tris, nt, P, seg_off, first, etab, nslots - 1, sg.plane, sg.edges,
                                                (G*)sg.pts, keys, vid);
  ctx->launches++;
  // ---- chaining (darts.cuh), as in ctr_mt2d_polylines
  size_t vslots = 1024;
  while (vslots < nd * 2) vslots <<= 1;
  VSlot* tab;
  unsigned *succ, *bd, *bd2, *jmp, *jmp2, *dist, *dist2, *npts, *poff, *pidx, *bsum, *dtot;
  unsigned long long *bp, *bp2;
  PolyCounters* dctr;
  const size_t nb_scan = (nd + PS_TILE - 1) / PS_TILE;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH2], [&](ctr_carve& c) {
         c(tab, vslots * sizeof(VSlot));
         c(succ, nd * 4);
         c(bp, nd * 8);
         c(bp2, nd * 8);
         c(bd, nd * 4);
         c(bd2, nd * 4);
         c(jmp, nd * 4);
         c(jmp2, nd * 4);
         c(dist, nd * 4);
         c(dist2, nd * 4);
         c(npts, nd * 4);
         c(poff, nd * 4);
         c(pidx, nd * 4);
         c(bsum, nb_scan * 8 + 64);
         c(dctr, sizeof(PolyCounters));
         c(dtot, 64);
       })))
    return rc;
  const unsigned dblocks = (unsigned)((nd + 255) / 256), sblocks = (unsigned)((S + 255) / 256);
  const Vert3 vert{vid, sg.plane, sg.jplane};
  k_p_init<<<ctx->sm_count * 8, 256, 0, st>>>(tab, vslots, dctr);
  k_p_insert<<<dblocks, 256, 0, st>>>(vert, keys, (unsigned)nd, tab, vslots - 1, dctr);
  k_sec_kill<<<sblocks, 256, 0, st>>>((unsigned)S, sg.plane, sg.jplane, keys);
  k_p_succ<<<dblocks, 256, 0, st>>>(vert, keys, (unsigned)nd, tab, vslots - 1, succ, bp, bd, jmp);
  ctx->launches += 4;
  PolyCounters hp;
  for (int round = 0; round < 40; round += 2) {       // first dart of every cycle
    CTR_CUDA(ctx, cudaMemsetAsync(&dctr->changed, 0, 4, st));
    k_p_min<<<dblocks, 256, 0, st>>>((unsigned)nd, bp, bd, jmp, bp2, bd2, jmp2, dctr);
    k_p_min<<<dblocks, 256, 0, st>>>((unsigned)nd, bp2, bd2, jmp2, bp, bd, jmp, dctr);
    ctx->launches += 2;
    CTR_CUDA(ctx, cudaMemcpyAsync(&hp, dctr, sizeof hp, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (!hp.changed) break;
  }
  const int64_t J = (int64_t)hp.junction_levels;
  unsigned* start = bd;
  unsigned *nxt = jmp, *nxt2 = jmp2;
  k_p_cut<<<dblocks, 256, 0, st>>>((unsigned)nd, succ, start, nxt, dist);
  ctx->launches++;
  for (int round = 0; round < 40; round += 2) {       // positions
    CTR_CUDA(ctx, cudaMemsetAsync(&dctr->live, 0, 4, st));
    k_p_rank<<<dblocks, 256, 0, st>>>((unsigned)nd, nxt, dist, nxt2, dist2, dctr);
    k_p_rank<<<dblocks, 256, 0, st>>>((unsigned)nd, nxt2, dist2, nxt, dist, dctr);
    ctx->launches += 2;
    CTR_CUDA(ctx, cudaMemcpyAsync(&hp, dctr, sizeof hp, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (!hp.live) break;
  }
  k_p_mark<<<dblocks, 256, 0, st>>>((unsigned)nd, keys, start, dist, npts);
  ctx->launches++;
  scan_u32(ctx, npts, (unsigned)nd, poff, pidx, bsum, dtot);
  unsigned tot[2];
  CTR_CUDA(ctx, cudaMemcpyAsync(tot, dtot, 8, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const size_t N = tot[0], NP = tot[1];
  if (N >= (1ull << 31)) return ctr_fail(ctx, CTR_ERR_OVERFLOW, "2^31 or more section points: use fewer planes");
  if (NP == 0) return finish((int64_t)S, 0, 0, J);
  // ---- polylines: points in their final order, measures
  SecPolys pg;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SECTION_POLYS], [&](ctr_carve& c) { pg.carve(c, NP, N, gsz); }))) return rc;
  unsigned* pop;
  uint8_t* bad;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH1], [&](ctr_carve& c) {
         c(pop, N * 4);
         c(bad, NP);
       })))
    return rc;
  CTR_CUDA(ctx, cudaMemsetAsync(bad, 0, NP, st));
  CTR_CUDA(ctx, cudaMemsetAsync(pg.meas, 0, NP * 16, st));
  k_sec_points<G><<<dblocks, 256, 0, st>>>((unsigned)nd, keys, sg.plane, (const G*)sg.pts, start, dist, npts, poff, pidx,
                                           (G*)pg.pts, pop, pg.plane, pg.flags, pg.key, pg.off, pg.len, bad);
  const double nn = sqrt(sp->normal[0] * sp->normal[0] + sp->normal[1] * sp->normal[1] + sp->normal[2] * sp->normal[2]);
  k_sec_measure<G><<<(unsigned)((N + SEC_THREADS - 1) / SEC_THREADS), SEC_THREADS, 0, st>>>(
      (unsigned)N, (const G*)pg.pts, pop, pg.off, pg.len, pg.flags, bad, sp->normal[0] / nn, sp->normal[1] / nn,
      sp->normal[2] / nn, pg.meas);
  ctx->launches += 2;
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return finish((int64_t)S, (int64_t)NP, (int64_t)N, J);
}
