// Component filter (ctr_mt3d_keep_components) -- included by mt3d.cu after mt3d_select.cuh, inside its anonymous
// namespace, so that it calls the selection's compaction kernels as they are.
//
// The labels (aux[44]) and the table (aux[45]) of the last ctr_mt3d_components call say which component every
// triangle is in; the host says which components stay (one byte each).  Then
//   k_keep_tris : keep_t[t] = keep[label[t]];
//   k_sel_used, k_flag_scan x 3 (triangles, vertices, components) : as in the seeded selection, plus the new numbers of
//                 the kept components;
//   k_sel_rows / k_sel_tris : positions, normals, keys, lowmin, vertex values and triangles compacted in order, ids
//                 rewritten;
//   k_keep_labels / k_keep_table : the labels and the table rows of the kept components, renumbered 0..K-1 in order.
// A component is kept or dropped whole and no edge joins two components, so every field of a kept row stays true;
// only first_tri moves.  Everything goes through one scratch piece and back with cudaMemcpyAsync: the device pointers
// handed out before (ctr_mt3d_device_ptrs, ctr_mt3d_interpolate_device_ptr) stay valid.
struct KeepCounters {
  unsigned ticket[3];                // tile tickets of the three scans
  unsigned pad;
  unsigned long long total[3];       // kept triangles, used vertices, kept components
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
  const uint32_t fl = ctx->last_flags;
  const size_t gsz = (fl & CTR_GEOM_F64) ? 8 : 4;
  const bool want_n = (fl & CTR_WANT_NORMALS) != 0, want_k = (fl & CTR_WANT_KEYS) != 0;
  // values interpolated on this very mesh are compacted with it; older ones are left as they are
  const bool values = ctx->attr_ncomp > 0 && ctx->attr_gen == ctx->mesh_gen;
  const size_t vrow = std::max<size_t>(3 * gsz, values ? (size_t)ctx->attr_ncomp * gsz : 0);   // widest vertex row
  ctx->mesh_gen++;                                    // from here on the mesh is edited
  cudaStream_t st = ctx->stream;
  int rc;
  DevBuf& b_ctr = ctx->aux[31];
  if ((rc = ctr_ensure(ctx, b_ctr, sizeof(KeepCounters) + 64))) return rc;
  KeepCounters* dctr = (KeepCounters*)b_ctr.p;
  const int tiles_t = (int)(((size_t)nT + SC_TILE - 1) / SC_TILE), tiles_v = (int)(((size_t)nV + SC_TILE - 1) / SC_TILE),
            tiles_c = (int)(((size_t)nC + SC_TILE - 1) / SC_TILE);
  // one scratch allocation, carved (256-byte aligned pieces); aux[30] aliases none of aux[43..45]
  size_t off = 0;
  auto carve = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t o_kc = carve((size_t)nC + 8), o_kt = carve((size_t)nT + 8), o_used = carve((size_t)nV + 8),
               o_it = carve((size_t)nT * 4 + 4), o_iv = carve((size_t)nV * 4 + 4), o_ic = carve((size_t)nC * 4 + 4),
               o_st = carve((size_t)tiles_t * 8 + 8), o_sv = carve((size_t)tiles_v * 8 + 8), o_sc = carve((size_t)tiles_c * 8 + 8),
               o_out = carve(std::max<size_t>(std::max<size_t>((size_t)nV * vrow, (size_t)nT * 12),
                                              (size_t)nC * sizeof(ctr_mt3d_component)) + 16);
  DevBuf& b_s = ctx->aux[30];
  if ((rc = ctr_ensure(ctx, b_s, off))) return rc;
  char* base = (char*)b_s.p;
  uint8_t* keep_c = (uint8_t*)(base + o_kc);
  uint8_t* keep_t = (uint8_t*)(base + o_kt);
  uint8_t* used_v = (uint8_t*)(base + o_used);
  uint32_t* idx_t = (uint32_t*)(base + o_it);
  uint32_t* idx_v = (uint32_t*)(base + o_iv);
  uint32_t* idx_c = (uint32_t*)(base + o_ic);
  unsigned long long* st_t = (unsigned long long*)(base + o_st);
  unsigned long long* st_v = (unsigned long long*)(base + o_sv);
  unsigned long long* st_c = (unsigned long long*)(base + o_sc);
  void* tmp = base + o_out;
  const int* label = (const int*)ctx->aux[44].p;
  ctr_mt3d_component* table = (ctr_mt3d_component*)ctx->aux[45].p;
  CTR_CUDA(ctx, cudaMemsetAsync(dctr, 0, sizeof(KeepCounters), st));
  CTR_CUDA(ctx, cudaMemsetAsync(used_v, 0, (size_t)nV + 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(st_t, 0, (size_t)tiles_t * 8 + 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(st_v, 0, (size_t)tiles_v * 8 + 8, st));
  CTR_CUDA(ctx, cudaMemsetAsync(st_c, 0, (size_t)tiles_c * 8 + 8, st));
  if (nC) CTR_CUDA(ctx, cudaMemcpyAsync(keep_c, keep, nC, cudaMemcpyHostToDevice, st));
  const unsigned tb = (nT + 255) / 256, vb = (nV + 255) / 256, cb = (nC + 255) / 256;
  if (nT) {
    k_keep_tris<<<tb, 256, 0, st>>>(label, nT, keep_c, keep_t);
    // components need vert_id_base 0 and no offset_ids since: the ids are local
    k_sel_used<<<tb, 256, 0, st>>>((const int*)ctx->tris.p, nT, keep_t, 0u, used_v, nV);
    k_flag_scan<<<tiles_t, SC_THREADS, 0, st>>>(keep_t, nT, idx_t, st_t, &dctr->ticket[0], &dctr->total[0], tiles_t);
    ctx->launches += 3;
  }
  if (nV) {
    k_flag_scan<<<tiles_v, SC_THREADS, 0, st>>>(used_v, nV, idx_v, st_v, &dctr->ticket[1], &dctr->total[1], tiles_v);
    ctx->launches++;
  }
  if (nC) {
    k_flag_scan<<<tiles_c, SC_THREADS, 0, st>>>(keep_c, nC, idx_c, st_c, &dctr->ticket[2], &dctr->total[2], tiles_c);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  KeepCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, dctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const size_t newT = (size_t)h.total[0], newV = (size_t)h.total[1], newC = (size_t)h.total[2];
  // compaction through the scratch piece, array by array
  auto rows = [&](void* p, int wpr, size_t row_bytes) -> int {
    if (!nV || !p) return 0;
    k_sel_rows<<<vb, 256, 0, st>>>((const uint32_t*)p, (uint32_t*)tmp, used_v, idx_v, nV, wpr);
    ctx->launches++;
    if (newV) CTR_CUDA(ctx, cudaMemcpyAsync(p, tmp, newV * row_bytes, cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  if ((rc = rows(ctx->verts.p, (int)(3 * gsz / 4), 3 * gsz))) return rc;
  if (want_n && (rc = rows(ctx->normals.p, (int)(3 * gsz / 4), 3 * gsz))) return rc;
  if (want_k && (rc = rows(ctx->keys.p, 2, 8))) return rc;
  if (want_k && (rc = rows(ctx->lowmin.p, 0, 1))) return rc;
  if (values && (rc = rows(ctx->aux[43].p, (int)(ctx->attr_ncomp * gsz / 4), ctx->attr_ncomp * gsz))) return rc;
  if (nT) {
    k_sel_tris<<<tb, 256, 0, st>>>((const int*)ctx->tris.p, (int*)tmp, keep_t, idx_t, idx_v, nT, 0u);
    ctx->launches++;
    if (newT) CTR_CUDA(ctx, cudaMemcpyAsync(ctx->tris.p, tmp, newT * 12, cudaMemcpyDeviceToDevice, st));
    k_keep_labels<<<tb, 256, 0, st>>>(label, nT, keep_t, idx_t, idx_c, (int*)tmp);
    ctx->launches++;
    if (newT) CTR_CUDA(ctx, cudaMemcpyAsync(ctx->aux[44].p, tmp, newT * 4, cudaMemcpyDeviceToDevice, st));
  }
  if (nC) {
    k_keep_table<<<cb, 256, 0, st>>>(table, nC, keep_c, idx_t, idx_c, (ctr_mt3d_component*)tmp);
    ctx->launches++;
    if (newC) CTR_CUDA(ctx, cudaMemcpyAsync(table, tmp, newC * sizeof(ctr_mt3d_component), cudaMemcpyDeviceToDevice, st));
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  ctx->last3_edited |= 4u;
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
