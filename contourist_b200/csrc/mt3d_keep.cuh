// Component filter (ctr_mt3d_keep_components) -- included by mt3d.cu after compact3d.cuh, inside its anonymous
// namespace.
//
// The labels (AUX_LABELS) and the table (AUX_COMPONENTS) of the last ctr_mt3d_components call say which component every
// triangle is in; the host says which components stay (one byte each).  Then
//   k_keep_tris : keep_t[t] = keep[label[t]];
//   k_sel_used, k_flag_scan : the vertices of the kept triangles; the new numbers of the kept components;
//   compact_mesh : positions, normals, keys, lowmin, vertex values and triangles compacted in order, ids rewritten;
//   k_keep_labels / k_keep_table : the labels and the table rows of the kept components, renumbered 0..K-1 in order.
// A component is kept or dropped whole and no edge joins two components, so every field of a kept row stays true;
// only first_tri moves.  Everything goes through one scratch piece and back with cudaMemcpyAsync: the device pointers
// handed out before (ctr_mt3d_device_ptrs, ctr_mt3d_interpolate_device_ptr) stay valid.
struct KeepCounters {
  unsigned ticket;                   // tile ticket of the component scan
  unsigned long long total;          // kept components
};

__global__ void k_keep_tris(const int* __restrict__ label, unsigned n_tris, const uint8_t* __restrict__ keep_c,
                            uint8_t* __restrict__ keep_t) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris) return;
  keep_t[t] = keep_c[label[t]] ? 1 : 0;
}

__global__ void k_keep_labels(const int* __restrict__ label, unsigned n_tris, const uint8_t* __restrict__ keep_t,
                              const uint32_t* __restrict__ idx_t, const uint32_t* __restrict__ idx_c, int* __restrict__ dst) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris || !keep_t[t]) return;
  dst[idx_t[t]] = (int)idx_c[label[t]];
}

__global__ void k_keep_table(const ctr_mt3d_component* __restrict__ src, unsigned n_comp, const uint8_t* __restrict__ keep_c,
                             const uint32_t* __restrict__ idx_t, const uint32_t* __restrict__ idx_c,
                             ctr_mt3d_component* __restrict__ dst) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_comp || !keep_c[c]) return;
  ctr_mt3d_component row = src[c];
  row.first_tri = idx_t[row.first_tri];       // still the component's smallest triangle: the numbering rule holds
  dst[idx_c[c]] = row;
}

int keep_components_run(ctr_ctx* ctx, const uint8_t* keep, int64_t* out_verts, int64_t* out_tris) {
  const unsigned nV = (unsigned)ctx->last_counts[0], nT = (unsigned)ctx->last_counts[1], nC = (unsigned)ctx->comp_count;
  const size_t gsz = (ctx->last_flags & CTR_GEOM_F64) ? 8 : 4;
  // values interpolated on this very mesh are compacted with it; older ones are left as they are
  const bool values = ctx->attr_ncomp > 0 && ctx->attr_gen == ctx->mesh_gen;
  const size_t vrow = std::max<size_t>(3 * gsz, values ? (size_t)ctx->attr_ncomp * gsz : 0);   // widest vertex row
  ctx->mesh_gen++;                                    // from here on the mesh is edited
  cudaStream_t st = ctx->stream;
  int rc;
  const int tiles_c = (int)(((size_t)nC + SC_TILE - 1) / SC_TILE);
  uint8_t* keep_c;
  uint32_t* idx_c;
  unsigned long long* st_c;                           // look-back words of the component scan
  CompactBufs cb;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH3], [&](ctr_carve& c) {
         c(keep_c, (size_t)nC + 8);
         c(idx_c, (size_t)nC * 4 + 4);
         c(st_c, (size_t)tiles_c * 8 + 8);
         compact_carve(c, nV, nT, sizeof(KeepCounters), cb);
         c(cb.stage, std::max({(size_t)nV * vrow, (size_t)nT * 12, (size_t)nC * sizeof(ctr_mt3d_component)}) + 16);
       })))
    return rc;
  KeepCounters* dctr = (KeepCounters*)cb.scan;        // the pass's counters of the scan piece
  const int* label = (const int*)ctx->aux[AUX_LABELS].p;
  ctr_mt3d_component* table = (ctr_mt3d_component*)ctx->aux[AUX_COMPONENTS].p;
  CTR_CUDA(ctx, cudaMemsetAsync(dctr, 0, sizeof(KeepCounters), st));
  CTR_CUDA(ctx, cudaMemsetAsync(st_c, 0, (size_t)tiles_c * 8 + 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(cb.used_v, 0, (size_t)nV + 8, st));
  if (nC) CTR_CUDA(ctx, cudaMemcpyAsync(keep_c, keep, nC, cudaMemcpyHostToDevice, st));
  const unsigned tb = (nT + 255) / 256, cblk = (nC + 255) / 256;
  if (nT) {
    k_keep_tris<<<tb, 256, 0, st>>>(label, nT, keep_c, cb.keep_t);
    // components need vert_id_base 0 and no offset_ids since: the ids are local
    k_sel_used<<<tb, 256, 0, st>>>((const int*)ctx->tris.p, nT, cb.keep_t, 0u, cb.used_v, nV);
    ctx->launches += 2;
  }
  if (nC) {
    k_flag_scan<<<tiles_c, SC_THREADS, 0, st>>>(keep_c, nC, idx_c, st_c, &dctr->ticket, &dctr->total, tiles_c);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  KeepCounters h;
  size_t newV, newT;
  if ((rc = compact_mesh(ctx, cb, nV, nT, (const int*)ctx->tris.p, 0u, values, &h, newV, newT))) return rc;
  const size_t newC = (size_t)h.total;
  if (nT) {
    k_keep_labels<<<tb, 256, 0, st>>>(label, nT, cb.keep_t, cb.idx_t, idx_c, (int*)cb.stage);
    ctx->launches++;
    if (newT) CTR_CUDA(ctx, cudaMemcpyAsync(ctx->aux[AUX_LABELS].p, cb.stage, newT * 4, cudaMemcpyDeviceToDevice, st));
  }
  if (nC) {
    k_keep_table<<<cblk, 256, 0, st>>>(table, nC, keep_c, cb.idx_t, idx_c, (ctr_mt3d_component*)cb.stage);
    ctx->launches++;
    if (newC) CTR_CUDA(ctx, cudaMemcpyAsync(table, cb.stage, newC * sizeof(ctr_mt3d_component), cudaMemcpyDeviceToDevice, st));
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  ctx->last3_edited |= EDIT_KEEP;
  ctx->comp_tris = (int64_t)newT;
  ctx->comp_count = (int64_t)newC;
  ctx->comp_gen = ctx->mesh_gen;
  if (values) {
    ctx->attr_rows = newV;
    ctx->attr_gen = ctx->mesh_gen;
  }
  if (out_verts) *out_verts = (int64_t)newV;
  if (out_tris) *out_tris = (int64_t)newT;
  return 0;
}
