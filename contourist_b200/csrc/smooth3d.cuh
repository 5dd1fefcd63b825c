// Taubin lambda|mu smoothing of the 3D device mesh (ctr_mt3d_smooth).
//
// Included into mesh3d.cu after components3d.cuh, inside its anonymous namespace: the pass builds its edge table with
// the components pass's k_m_init / k_m_edges (distinct undirected edges with their use counts in slot.pad, bad ids
// flagged) and scans with lb_lookback.  The definition is oracle/mt3d_smooth.py:smooth (positions bit for bit) and
// :normals (within rounding: the face normals are summed with atomics).
//   k_s_fixed  : per edge slot (self-edges skipped): edges counted, both ends of an edge with uses != 2 marked fixed;
//   k_s_degree : per edge slot: one more neighbour for each end that is not fixed;
//   k_s_scan   : degrees -> CSR offsets by a decoupled look-back over ticketed tiles; vertices of degree 0 (fixed, or on
//                no edge) counted;
//   k_s_fill   : per edge slot: each free end appends the other end through an atomic cursor;
//   k_s_sort   : per vertex, its list sorted in place (ascending ids: the order the definition sums in);
//   k_s_widen  : geometry type -> both fp64 working copies (fixed vertices are never written again);
//   k_s_step   : one Jacobi step, one thread per free vertex, reading one copy and writing the other;
//   k_s_store  : the result rounded into ctx->verts in place;
//   k_s_nsum / k_s_nfin (normals3d.cuh): (CTR_WANT_NORMALS) per-triangle cross products summed into the corners (fp64
//                atomicAdd), then normalised with the sign of the old gradient normal.
// Scratch: AUX_SCRATCH0 edge table, AUX_SCRATCH1 per-vertex offsets / cursors / fixed flags, AUX_SCRATCH2 neighbour
// lists, AUX_SCRATCH3 counters and look-back words, AUX_SMOOTH_X0 / AUX_SMOOTH_X1 the two fp64 copies.

constexpr int S_THREADS = 256;

struct SCounters {                                    // head of AUX_SCRATCH3, then one look-back word per vertex tile
  MCounters m;                                        // k_m_edges' bad-id flag; the scan's ticket and total degree
  unsigned long long n_edges, n_fixed;
};
static_assert(sizeof(SCounters) <= 64, "SCounters fits the 64-byte head of the scratch block");

// an edge slot that names a real edge: not empty, not a self-edge {a, a} of a degenerate triangle
__device__ __forceinline__ bool s_edge(const EdgeSlot& s, unsigned& lo, unsigned& hi) {
  lo = (unsigned)s.key;
  hi = (unsigned)(s.key >> 32);
  return s.key != EMPTY && lo != hi;
}

__global__ void k_s_fixed(const EdgeSlot* __restrict__ tab, size_t nslots, uint8_t* __restrict__ fixed, SCounters* ctr) {
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  unsigned long long edges = 0;
  for (size_t q = t0; q < nslots; q += n) {
    const EdgeSlot s = tab[q];
    unsigned lo, hi;
    if (!s_edge(s, lo, hi)) continue;
    ++edges;
    if (s.pad != 2) {                                 // boundary or non-manifold
      fixed[lo] = 1;
      fixed[hi] = 1;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) edges += __shfl_xor_sync(0xffffffffu, edges, o);
  if (lane_id() == 0 && edges) atomicAdd(&ctr->n_edges, edges);
}

__global__ void k_s_degree(const EdgeSlot* __restrict__ tab, size_t nslots, const uint8_t* __restrict__ fixed,
                           unsigned* __restrict__ deg) {
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t0; q < nslots; q += n) {
    const EdgeSlot s = tab[q];
    unsigned lo, hi;
    if (!s_edge(s, lo, hi)) continue;
    if (!fixed[lo]) atomicAdd(&deg[lo], 1u);
    if (!fixed[hi]) atomicAdd(&deg[hi], 1u);
  }
}

// cur[v]: degree in, start of v's list out (the cursor of k_s_fill); off[v] the same start, off[nv] the total
__global__ void __launch_bounds__(S_THREADS) k_s_scan(unsigned* __restrict__ cur, unsigned nv, unsigned* __restrict__ off,
                                                      unsigned long long* status, SCounters* ctr, int ntiles) {
  __shared__ unsigned s_tile;
  __shared__ unsigned s_warp[S_THREADS / 32];
  __shared__ unsigned long long s_excl;
  if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->m.ticket, 1u);
  __syncthreads();
  const int tile = (int)s_tile;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned v = (unsigned)tile * S_THREADS + threadIdx.x;
  const unsigned d = v < nv ? cur[v] : 0u;
  const unsigned incl = warp_incl_scan_u32(d);
  const unsigned zero = __ballot_sync(0xffffffffu, v < nv && d == 0);
  if (lane == 31) s_warp[warp] = incl;
  if (lane == 0 && zero) atomicAdd(&ctr->n_fixed, (unsigned long long)__popc(zero));
  __syncthreads();
  unsigned woff = 0, blk = 0;
#pragma unroll
  for (int w = 0; w < S_THREADS / 32; ++w) {
    if (w < (int)warp) woff += s_warp[w];
    blk += s_warp[w];
  }
  if (warp == 0) {
    const unsigned long long e = lb_lookback(status, tile, (unsigned long long)blk);
    if (lane == 0) s_excl = e;
  }
  __syncthreads();
  if (v < nv) {
    const unsigned o = (unsigned)s_excl + woff + incl - d;
    off[v] = o;
    cur[v] = o;
  }
  if (tile == ntiles - 1 && threadIdx.x == 0) {
    off[nv] = (unsigned)(s_excl + blk);
    ctr->m.total = s_excl + blk;
  }
}

__global__ void k_s_fill(const EdgeSlot* __restrict__ tab, size_t nslots, const uint8_t* __restrict__ fixed,
                         unsigned* __restrict__ cur, int* __restrict__ nbr) {
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t0; q < nslots; q += n) {
    const EdgeSlot s = tab[q];
    unsigned lo, hi;
    if (!s_edge(s, lo, hi)) continue;
    if (!fixed[lo]) nbr[atomicAdd(&cur[lo], 1u)] = (int)hi;
    if (!fixed[hi]) nbr[atomicAdd(&cur[hi], 1u)] = (int)lo;
  }
}

__global__ void k_s_sort(const unsigned* __restrict__ off, unsigned nv, int* __restrict__ nbr) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const unsigned b = off[v], e = off[v + 1];
  for (unsigned i = b + 1; i < e; ++i) {             // insertion sort: the lists are short (about 6 ids)
    const int x = nbr[i];
    unsigned j = i;
    for (; j > b && nbr[j - 1] > x; --j) nbr[j] = nbr[j - 1];
    nbr[j] = x;
  }
}

template <typename G>
__global__ void k_s_widen(const G* __restrict__ verts, size_t n, double* __restrict__ a, double* __restrict__ b) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = (double)verts[i];
  a[i] = x;
  b[i] = x;
}

// x' = x + w * (avg - x), avg = (x[n0] + x[n1] + ...) / deg in ascending neighbour order; every operation rounded on its
// own (the _rn intrinsics are never contracted into a fused multiply-add)
__global__ void __launch_bounds__(S_THREADS) k_s_step(const double* __restrict__ x, double* __restrict__ y,
                                                      const unsigned* __restrict__ off, const int* __restrict__ nbr,
                                                      unsigned nv, double w) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const unsigned b = off[v], e = off[v + 1];
  if (b == e) return;                                 // fixed: both copies hold it since k_s_widen
  const double* p = x + (size_t)nbr[b] * 3;
  double sx = p[0], sy = p[1], sz = p[2];
  for (unsigned i = b + 1; i < e; ++i) {
    p = x + (size_t)nbr[i] * 3;
    sx = __dadd_rn(sx, p[0]);
    sy = __dadd_rn(sy, p[1]);
    sz = __dadd_rn(sz, p[2]);
  }
  const double d = (double)(e - b);
  const double* c = x + (size_t)v * 3;
  double* o = y + (size_t)v * 3;
  o[0] = __dadd_rn(c[0], __dmul_rn(w, __dsub_rn(__ddiv_rn(sx, d), c[0])));
  o[1] = __dadd_rn(c[1], __dmul_rn(w, __dsub_rn(__ddiv_rn(sy, d), c[1])));
  o[2] = __dadd_rn(c[2], __dmul_rn(w, __dsub_rn(__ddiv_rn(sz, d), c[2])));
}

template <typename G>
__global__ void k_s_store(const double* __restrict__ x, size_t n, G* __restrict__ verts) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  verts[i] = (G)x[i];
}

template <typename G>
int smooth_typed(ctr_ctx* ctx, const ctr_smooth_params* sp, ctr_smooth_counts* out) {
  const unsigned nt = (unsigned)ctx->last_counts[1], nv = (unsigned)ctx->last_counts[0];
  cudaStream_t st = ctx->stream;
  if (nt == 0) {                                      // no edges: every vertex is fixed, nothing moves
    out->n_fixed_verts = nv;
    return 0;
  }
  size_t nslots = 1;
  while (nslots < (size_t)nt * 4) nslots <<= 1;       // the components pass's table size: load <= 3/4
  const unsigned blocks_t = (nt + S_THREADS - 1) / S_THREADS, tiles_v = (nv + S_THREADS - 1) / S_THREADS;
  const unsigned slot_blocks = (unsigned)ctx->sm_count * 8;
  int rc;
  DevBuf& b_etab = ctx->aux[AUX_SCRATCH0];
  DevBuf& b_vert = ctx->aux[AUX_SCRATCH1];
  DevBuf& b_nbr = ctx->aux[AUX_SCRATCH2];
  DevBuf& b_scan = ctx->aux[AUX_SCRATCH3];
  DevBuf& b_x0 = ctx->aux[AUX_SMOOTH_X0];
  DevBuf& b_x1 = ctx->aux[AUX_SMOOTH_X1];
  const size_t vbytes = (size_t)(nv + 1) * 4 + (size_t)nv * 4 + nv;   // off, cur, fixed
  if ((rc = ctr_ensure(ctx, b_etab, nslots * sizeof(EdgeSlot)))) return rc;
  if ((rc = ctr_ensure(ctx, b_vert, vbytes))) return rc;
  if ((rc = ctr_ensure(ctx, b_scan, 64 + (size_t)tiles_v * 8))) return rc;
  EdgeSlot* etab = (EdgeSlot*)b_etab.p;
  unsigned* off = (unsigned*)b_vert.p;
  unsigned* cur = off + nv + 1;
  uint8_t* fixed = (uint8_t*)(cur + nv);
  SCounters* ctr = (SCounters*)b_scan.p;
  unsigned long long* status = (unsigned long long*)((char*)b_scan.p + 64);
  const int* tris = (const int*)ctx->tris.p;
  CTR_CUDA(ctx, cudaMemsetAsync(b_scan.p, 0, 64 + (size_t)tiles_v * 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(cur, 0, (size_t)nv * 5, st));          // cur and fixed
  // the (component, vertex) table of k_m_init aliases the edge table: this pass reads only slot.key and slot.pad
  k_m_init<<<slot_blocks, 256, 0, st>>>(etab, etab, nslots, nullptr, 0u);
  k_m_edges<<<blocks_t, M_THREADS, 0, st>>>(tris, nt, nv, etab, nslots - 1, &ctr->m);
  ctx->launches += 2;
  CTR_CUDA(ctx, cudaGetLastError());
  SCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.m.bad) return ctr_fail(ctx, CTR_ERR_STATE, "triangle ids outside [0, n_verts): the ids were shifted (ctr_mt3d_offset_ids)");
  k_s_fixed<<<slot_blocks, 256, 0, st>>>(etab, nslots, fixed, ctr);
  k_s_degree<<<slot_blocks, 256, 0, st>>>(etab, nslots, fixed, cur);
  k_s_scan<<<tiles_v, S_THREADS, 0, st>>>(cur, nv, off, status, ctr, (int)tiles_v);   // (nv > 0: the ids were checked)
  ctx->launches += 3;
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  out->n_edges = (int64_t)h.n_edges;
  out->n_fixed_verts = (int64_t)h.n_fixed;
  if (sp->iterations == 0) return 0;
  const size_t n3 = (size_t)nv * 3;
  if ((rc = ctr_ensure(ctx, b_nbr, (size_t)h.m.total * 4))) return rc;
  if ((rc = ctr_ensure(ctx, b_x0, n3 * 8))) return rc;
  if ((rc = ctr_ensure(ctx, b_x1, n3 * 8))) return rc;
  ctx->mesh_gen++;                                    // from here on the mesh is edited
  ctx->last3_edited |= EDIT_SMOOTH;
  int* nbr = (int*)b_nbr.p;
  double* x = (double*)b_x0.p;
  double* y = (double*)b_x1.p;
  G* verts = (G*)ctx->verts.p;
  const unsigned vblocks = (nv + S_THREADS - 1) / S_THREADS, cblocks = (unsigned)((n3 + 255) / 256);
  k_s_fill<<<slot_blocks, 256, 0, st>>>(etab, nslots, fixed, cur, nbr);
  k_s_sort<<<vblocks, S_THREADS, 0, st>>>(off, nv, nbr);
  k_s_widen<G><<<cblocks, 256, 0, st>>>(verts, n3, x, y);
  ctx->launches += 3;
  for (int it = 0; it < sp->iterations; ++it) {
    k_s_step<<<vblocks, S_THREADS, 0, st>>>(x, y, off, nbr, nv, sp->lambda);
    std::swap(x, y);
    ctx->launches++;
    if (sp->mu != 0.0) {
      k_s_step<<<vblocks, S_THREADS, 0, st>>>(x, y, off, nbr, nv, sp->mu);
      std::swap(x, y);
      ctx->launches++;
    }
  }
  k_s_store<G><<<cblocks, 256, 0, st>>>(x, n3, verts);
  ctx->launches++;
  if (ctx->last_flags & CTR_WANT_NORMALS) {           // y is free now: the per-vertex sums
    CTR_CUDA(ctx, cudaMemsetAsync(y, 0, n3 * 8, st));
    k_s_nsum<G><<<blocks_t, S_THREADS, 0, st>>>(verts, tris, nt, y);
    k_s_nfin<G><<<vblocks, S_THREADS, 0, st>>>(y, nv, (G*)ctx->normals.p);
    ctx->launches += 2;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}
