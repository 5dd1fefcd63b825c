// Seeded extraction (SURVEY.md 8(f3)) -- included by mt3d.cu inside its anonymous namespace.
//
// The reference tracks the surface from seed segments: find_initial_voxels (tetrahedral.py:396-441, restated on the
// host side of the binding: it reads a handful of samples) and a flood fill over the 26-neighbourhood of "border"
// voxels (expand_voxels / in_range, tetrahedral.py:443-469).  Its result is therefore the full scan restricted to the
// 26-connected components of border voxels that contain a seed voxel.  That is what these kernels compute on the mesh
// of the last full-volume ctr_mt3d_run:
//   nodes      = the emitting voxels of the run's work list  +  "connectors": border voxels that emit nothing (a corner
//                with f == value exactly on an otherwise high voxel, or every crossing tet skipped by np.allclose);
//                the flood fill walks through those, so they have to be in the graph;
//   k_sel_insert / k_sel_union : voxel id -> node in an open-addressing table; every node looks up its 13 "forward"
//                neighbours and unites with the ones that exist (lock-free union-find, uf_hash.cuh);
//   k_sel_seeds : the components of the seed voxels get flagged;
//   k_sel_mark  : every emitting voxel copies its component's flag to its triangles (contiguous in the output);
//   k_sel_used  : the vertices of the kept triangles; then compact_mesh (compact3d.cuh) compacts both in place, in order.

struct SelCounters {
  unsigned n_extra;                  // connector voxels found
};

template <typename T>
__device__ __forceinline__ unsigned long long vox_key(const Grid<T>& g, int i, int j, int k) {
  return ((unsigned long long)i * (unsigned long long)g.n1 + (unsigned long long)j) * (unsigned long long)g.n2 + (unsigned long long)k;
}

template <typename T>
__global__ void k_sel_cells(Grid<T> g, const unsigned long long* __restrict__ cell_id, unsigned n_cell,
                            unsigned long long* __restrict__ node_vox) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cell) return;
  const unsigned long long id = cell_id[c];
  int i, j, w;
  g.word_coords((unsigned)(id >> 28), i, j, w);
  node_vox[c] = vox_key(g, i, j, w * 32 + (int)((id >> 14) & 31u));
}

// node_vox == nullptr: count only
template <typename T>
__global__ void k_sel_connectors(Grid<T> g, unsigned nwords, unsigned long long* __restrict__ node_vox, unsigned base,
                                 unsigned cap, unsigned* n_extra) {
  const unsigned gw = blockIdx.x * blockDim.x + threadIdx.x;
  if (gw >= nwords) return;
  int i, j, w;
  g.word_coords(gw, i, j, w);
  if (i >= g.n0 - 1 || j >= g.n1 - 1) return;
  if (!g.rowflag[(size_t)i * g.n1 + j]) return;      // no sample of the voxel row anywhere near the isovalue
  Planes npl;
  load_planes(g, g.nbits, i, j, w, npl);
  uint32_t cand = (npl.P[0] | npl.P[1] | npl.P[2] | npl.P[3] | npl.S[0] | npl.S[1] | npl.S[2] | npl.S[3]) & npl.kp1;
  while (cand) {
    const int b = __ffs(cand) - 1;
    cand &= cand - 1;
    const int k = w * 32 + b;
    if (cell_emit_exact(g, i, j, k, nullptr)) continue;          // an emitting voxel: already a node
    double mn = INFINITY, mx = -INFINITY;
    bool all_a = true;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const double f = sample(g, i + ((c >> 2) & 1), j + ((c >> 1) & 1), k + (c & 1));
      mn = fmin(mn, f);
      mx = fmax(mx, f);
      all_a = all_a && near_a(f, g.v);
    }
    if (mn <= g.v && g.v <= mx && !all_a) {                       // border_voxel, tetrahedral.py:383-394
      const unsigned slot = atomicAdd(n_extra, 1u);
      if (node_vox && base + slot < cap) node_vox[base + slot] = vox_key(g, i, j, k);
    }
  }
}

__global__ void k_sel_init(ufh::Slot* tab, size_t nslots, int* parent, uint8_t* flag, unsigned n_nodes) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t; q < nslots; q += n) reinterpret_cast<int4*>(tab)[q] = make_int4(-1, -1, -1, 0);
  for (size_t q = t; q < n_nodes; q += n) {
    parent[q] = (int)q;
    flag[q] = 0;
  }
}

__global__ void k_sel_insert(const unsigned long long* __restrict__ node_vox, unsigned n_nodes, ufh::Slot* tab, size_t mask) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_nodes) return;
  ufh::hash_slot(tab, mask, node_vox[c], true)->tri = (int)c;    // voxel ids are unique: one writer per slot
}

__global__ void k_sel_union(const unsigned long long* __restrict__ node_vox, unsigned n_nodes, ufh::Slot* tab, size_t mask,
                            int* parent, long long n1, long long n2) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_nodes) return;
  const long long key = (long long)node_vox[c];
  // the 13 offsets that follow (0,0,0) lexicographically: each adjacent pair is visited once.  A step that leaves the
  // voxel range lands on sample index n1-1 or n2-1 of some row, which is never a voxel, so it is simply not found.
  for (int o = 14; o < 27; ++o) {
    const int di = o / 9 - 1, dj = (o / 3) % 3 - 1, dk = o % 3 - 1;
    const long long nk = key + ((long long)di * n1 + dj) * n2 + dk;
    if (nk < 0) continue;
    const ufh::Slot* s = ufh::hash_slot(tab, mask, (unsigned long long)nk, false);
    if (s->key == (unsigned long long)nk) ufh::uf_union(parent, (int)c, s->tri);
  }
}

__global__ void k_sel_seeds(const int* __restrict__ seeds, unsigned n_seeds, int n0, int n1, int n2, ufh::Slot* tab,
                            size_t mask, int* parent, uint8_t* flag) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_seeds) return;
  const int i = seeds[q * 3], j = seeds[q * 3 + 1], k = seeds[q * 3 + 2];
  if (i < 0 || j < 0 || k < 0 || i >= n0 - 1 || j >= n1 - 1 || k >= n2 - 1) return;   // a "leak" voxel of the reference
  const unsigned long long key = ((unsigned long long)i * (unsigned long long)n1 + (unsigned long long)j) * (unsigned long long)n2 + (unsigned long long)k;
  const ufh::Slot* s = ufh::hash_slot(tab, mask, key, false);
  if (s->key == key) flag[ufh::uf_find(parent, s->tri)] = 1;
}

__global__ void k_sel_mark(const unsigned long long* __restrict__ cell_id, unsigned n_cell, const uint4* __restrict__ wrec, int* parent, const uint8_t* __restrict__ flag,
                           uint8_t* __restrict__ keep_t, unsigned n_tris, unsigned* n_sel_cells) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cell) return;
  int r = (int)c;
  for (int q = parent[r]; q != r; q = parent[r]) r = q;          // unions are over: read-only walk
  if (!flag[r]) return;
  atomicAdd(n_sel_cells, 1u);
  const unsigned long long id = cell_id[c];
  const unsigned c8 = (unsigned)(id & 255u), emit = (unsigned)((id >> 8) & 63u);
  unsigned nt = 0;
#pragma unroll
  for (int t = 0; t < 6; ++t)
    if ((emit >> t) & 1u) nt += (__popc(tet_mask_of(c8, t)) == 2) ? 2u : 1u;
  const unsigned t0 = wrec[(unsigned)(id >> 28)].y + ((unsigned)(id >> 19) & 511u);
  for (unsigned q = 0; q < nt; ++q)
    if (t0 + q < n_tris) keep_t[t0 + q] = 1;
}

template <typename T>
int select_typed(ctr_ctx* ctx, const ctr_mt3d_params* p, const int32_t* seeds, int64_t n_seeds, int64_t* out_verts,
                 int64_t* out_tris, int64_t* out_voxels) {
  const int n0 = (int)p->n0, n1 = (int)p->n1, n2 = (int)p->n2;
  const int W = (n2 + 31) / 32;
  const long long nwords = (long long)n0 * n1 * W;
  cudaStream_t st = ctx->stream;
  Grid<T> g;
  g.f = (p->flags & CTR_FIELD_ON_DEVICE) ? (const T*)p->field : (const T*)ctx->field.p;
  g.n0 = n0; g.n1 = n1; g.n2 = n2; g.W = W;
  g.i_lo = 0; g.i_hi = n0; g.i_hiv = n0;
  g.plane_offset = p->plane_offset;
  g.id_base = (unsigned)p->vert_id_base;
  g.v = p->isovalue;
  g.tolv = 1e-8 + 1e-5 * fabs(p->isovalue);
  g.any_near = 0;
  g.divW.init((unsigned)W);
  g.divN1.init((unsigned)n1);
  g.bits = (const uint32_t*)ctx->bits.p;
  g.nbits = (const uint32_t*)ctx->nbits.p;
  g.rowflag = (const uint8_t*)ctx->aux[AUX_ROW_FLAGS].p;
  g.wordflag = (const uint32_t*)ctx->aux[AUX_WORD_FLAGS].p;
  g.exactflag = (uint32_t*)ctx->aux[AUX_EXACT_FLAGS].p;
  g.wshift = 0;
  while ((W >> g.wshift) > 32) ++g.wshift;
  const unsigned nV = (unsigned)ctx->last_counts[0], nT = (unsigned)ctx->last_counts[1];
  const unsigned n_cell = (unsigned)ctx->last_cell;
  const size_t gsz = (p->flags & CTR_GEOM_F64) ? 8 : 4;
  const unsigned long long* cell_id = (const unsigned long long*)ctx->aux[AUX_CELL_LIST].p;
  int rc;
  DevBuf& b_ctr = ctx->aux[AUX_SCRATCH4];
  if ((rc = ctr_ensure(ctx, b_ctr, sizeof(SelCounters) + 64))) return rc;
  SelCounters* dctr = (SelCounters*)b_ctr.p;
  SelCounters h;
  CTR_CUDA(ctx, cudaMemsetAsync(dctr, 0, sizeof(SelCounters), st));
  // connectors, counted first (rare: they need a sample exactly on the isovalue)
  const unsigned wb = (unsigned)((nwords + 255) / 256);
  k_sel_connectors<T><<<wb, 256, 0, st>>>(g, (unsigned)nwords, nullptr, 0u, 0u, &dctr->n_extra);
  ctx->launches++;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, dctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned n_extra = h.n_extra;
  const size_t n_nodes = (size_t)n_cell + n_extra;
  if (n_nodes >= 0x7fffffffull) return ctr_fail(ctx, CTR_ERR_OVERFLOW, "too many border voxels for one selection");
  size_t nslots = 1024;
  while (nslots < n_nodes * 2) nslots <<= 1;
  unsigned long long* node_vox;
  ufh::Slot* tab;
  int* parent;
  uint8_t* flag;
  CompactBufs cb;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH3], [&](ctr_carve& c) {
         c(node_vox, n_nodes * 8 + 8);
         c(tab, nslots * sizeof(ufh::Slot));
         c(parent, n_nodes * 4 + 4);
         c(flag, n_nodes + 1);
         compact_carve(c, nV, nT, sizeof(unsigned), cb);
         c(cb.stage, std::max<size_t>((size_t)nV * 3 * gsz, (size_t)nT * 12) + 16);
       })))
    return rc;
  DevBuf& b_seeds = ctx->aux[AUX_SCRATCH2];
  if ((rc = ctr_ensure(ctx, b_seeds, (size_t)std::max<int64_t>(n_seeds, 1) * 12))) return rc;
  if (n_seeds) CTR_CUDA(ctx, cudaMemcpyAsync(b_seeds.p, seeds, (size_t)n_seeds * 12, cudaMemcpyHostToDevice, st));
  unsigned* n_voxels = (unsigned*)cb.scan;           // emitting voxels selected: the pass's counter of the scan piece
  CTR_CUDA(ctx, cudaMemsetAsync(dctr, 0, sizeof(SelCounters), st));
  CTR_CUDA(ctx, cudaMemsetAsync(n_voxels, 0, sizeof(unsigned), st));
  CTR_CUDA(ctx, cudaMemsetAsync(cb.keep_t, 0, (size_t)nT + 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(cb.used_v, 0, (size_t)nV + 8, st));
  const unsigned nb = (unsigned)((n_nodes + 255) / 256), cblk = (n_cell + 255) / 256;
  if (n_cell) k_sel_cells<T><<<cblk, 256, 0, st>>>(g, cell_id, n_cell, node_vox);
  if (n_extra) k_sel_connectors<T><<<wb, 256, 0, st>>>(g, (unsigned)nwords, node_vox, n_cell, (unsigned)n_nodes, &dctr->n_extra);
  k_sel_init<<<ctx->sm_count * 8, 256, 0, st>>>(tab, nslots, parent, flag, (unsigned)n_nodes);
  if (n_nodes) {
    k_sel_insert<<<nb, 256, 0, st>>>(node_vox, (unsigned)n_nodes, tab, nslots - 1);
    k_sel_union<<<nb, 256, 0, st>>>(node_vox, (unsigned)n_nodes, tab, nslots - 1, parent, n1, n2);
  }
  if (n_seeds)
    k_sel_seeds<<<(unsigned)((n_seeds + 255) / 256), 256, 0, st>>>((const int*)b_seeds.p, (unsigned)n_seeds, n0, n1, n2, tab,
                                                                    nslots - 1, parent, flag);
  if (n_cell)
    k_sel_mark<<<cblk, 256, 0, st>>>(cell_id, n_cell, (const uint4*)ctx->wdir.p, parent, flag, cb.keep_t, nT, n_voxels);
  if (nT) k_sel_used<<<(nT + 255) / 256, 256, 0, st>>>((const int*)ctx->tris.p, nT, cb.keep_t, g.id_base, cb.used_v, nV);
  ctx->launches += 1 + (n_cell ? 2 : 0) + (n_extra ? 1 : 0) + (n_nodes ? 2 : 0) + (n_seeds ? 1 : 0) + (nT ? 1 : 0);
  CTR_CUDA(ctx, cudaGetLastError());
  unsigned h_voxels = 0;
  size_t newV, newT;
  if ((rc = compact_mesh(ctx, cb, nV, nT, (const int*)ctx->tris.p, g.id_base, false, &h_voxels, newV, newT))) return rc;
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  ctx->last3_edited |= EDIT_SELECT;
  if (out_verts) *out_verts = (int64_t)newV;
  if (out_tris) *out_tris = (int64_t)newT;
  if (out_voxels) *out_voxels = (int64_t)h_voxels;
  return 0;
}
