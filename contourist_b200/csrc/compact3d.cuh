// Order-preserving compaction of the 3D device mesh in place -- included by mt3d.cu inside its anonymous namespace,
// before the passes that drop triangles and the vertices no kept triangle uses: the seeded selection, the component
// filter, the clean-up and the decimation.  A pass carves the pieces below out of its scratch (compact_carve), flags the
// triangles it keeps (keep_t) and the vertices they use (used_v: k_sel_used, or the pass's own kernel), then calls
// compact_mesh:
//   k_flag_scan x 2 : new triangle and vertex indices, single-pass look-back scans;
//   k_sel_rows      : positions, normals, keys, lowmin and optionally the vertex values, array by array through the
//                     staging rows and back with cudaMemcpyAsync, so the device pointers handed out before stay valid;
//   k_sel_tris      : the kept triangles, ids renumbered.
constexpr int SC_THREADS = 256;
constexpr int SC_PER = 8;
constexpr int SC_TILE = SC_THREADS * SC_PER;

struct CompactCounters {
  unsigned ticket[2];                // tile tickets of the two scans
  unsigned long long total[2];       // kept triangles, used vertices
};
static_assert(sizeof(CompactCounters) <= 64, "CompactCounters fits the 64-byte head of the scan piece");

__global__ void k_sel_used(const int* __restrict__ tris, unsigned n_tris, const uint8_t* __restrict__ keep_t, unsigned id_base,
                           uint8_t* __restrict__ used_v, unsigned n_verts) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris || !keep_t[t]) return;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    const unsigned v = (unsigned)tris[(size_t)t * 3 + q] - id_base;
    if (v < n_verts) used_v[v] = 1;
  }
}

// idx[q] = number of set flags before q; *total = number of set flags.  Tiles take tickets, prefixes by look-back.
__global__ void __launch_bounds__(SC_THREADS) k_flag_scan(const uint8_t* __restrict__ flags, unsigned n, uint32_t* __restrict__ idx,
                                                          unsigned long long* status, unsigned* ticket,
                                                          unsigned long long* total, int ntiles) {
  __shared__ unsigned s_tile;
  __shared__ unsigned s_warp[SC_THREADS / 32];
  __shared__ unsigned long long s_excl;
  if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const int tile = (int)s_tile;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned q0 = (unsigned)tile * SC_TILE + threadIdx.x * SC_PER;
  unsigned f[SC_PER], cnt = 0;
#pragma unroll
  for (int u = 0; u < SC_PER; ++u) {
    f[u] = (q0 + u < n && flags[q0 + u]) ? 1u : 0u;
    cnt += f[u];
  }
  const unsigned inc = warp_incl_scan_u32(cnt);
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  unsigned woff = 0, blk = 0;
#pragma unroll
  for (int w = 0; w < SC_THREADS / 32; ++w) {
    if (w < (int)warp) woff += s_warp[w];
    blk += s_warp[w];
  }
  if (warp == 0) {
    const unsigned long long e = lb_lookback(status, tile, (unsigned long long)blk);
    if (lane == 0) s_excl = e;
  }
  __syncthreads();
  unsigned run = (unsigned)s_excl + woff + inc - cnt;
#pragma unroll
  for (int u = 0; u < SC_PER; ++u) {
    if (q0 + u < n) idx[q0 + u] = run;
    run += f[u];
  }
  if (tile == ntiles - 1 && threadIdx.x == 0) *total = s_excl + blk;
}

// rows of `wpr` 32-bit words (or single bytes when wpr == 0): dst[idx[r]] = src[r] for flagged rows
__global__ void k_sel_rows(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, const uint8_t* __restrict__ flags,
                           const uint32_t* __restrict__ idx, unsigned n, int wpr) {
  const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n || !flags[r]) return;
  const size_t d = idx[r];
  if (wpr == 0) {
    reinterpret_cast<uint8_t*>(dst)[d] = reinterpret_cast<const uint8_t*>(src)[r];
    return;
  }
  for (int q = 0; q < wpr; ++q) dst[d * wpr + q] = src[(size_t)r * wpr + q];
}

__global__ void k_sel_tris(const int* __restrict__ src, int* __restrict__ dst, const uint8_t* __restrict__ keep_t,
                           const uint32_t* __restrict__ idx_t, const uint32_t* __restrict__ idx_v, unsigned n_tris,
                           unsigned id_base) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tris || !keep_t[t]) return;
  const size_t d = idx_t[t];
#pragma unroll
  for (int q = 0; q < 3; ++q) dst[d * 3 + q] = (int)(idx_v[(unsigned)src[(size_t)t * 3 + q] - id_base] + id_base);
}

struct CompactBufs {
  uint8_t *keep_t, *used_v;          // filled by the pass
  uint32_t *idx_t, *idx_v;
  // the scan piece: the pass's own counters (pass_bytes, zeroed by the pass) at the start, CompactCounters at ctr_off,
  // then the look-back words of both scans; one copy brings the pass's counters back with the totals
  char* scan;
  size_t pass_bytes, ctr_off, scan_bytes;
  void* stage;                       // staging rows: carved by the pass, last, for the widest array it compacts (at least
                                     // n_verts * 3 * geometry size and n_tris * 12 bytes)
  int tiles_t, tiles_v;
};

// The compaction's pieces of a pass's scratch but the staging rows; `pass_bytes` (at most 64): the pass's own counters.
static void compact_carve(ctr_carve& c, unsigned nV, unsigned nT, size_t pass_bytes, CompactBufs& b) {
  b.tiles_t = (int)(((size_t)nT + SC_TILE - 1) / SC_TILE);
  b.tiles_v = (int)(((size_t)nV + SC_TILE - 1) / SC_TILE);
  b.pass_bytes = pass_bytes;
  b.ctr_off = (pass_bytes + 7) & ~(size_t)7;
  b.scan_bytes = b.ctr_off + 64 + ((size_t)b.tiles_t + 1 + (size_t)b.tiles_v + 1) * 8;
  c(b.keep_t, (size_t)nT + 8);
  c(b.used_v, (size_t)nV + 8);
  c(b.idx_t, (size_t)nT * 4 + 4);
  c(b.idx_v, (size_t)nV * 4 + 4);
  c(b.scan, b.scan_bytes);
}

// Compacts the mesh of the last 3D run in place: the triangles with keep_t, their ids read from `tris` (ctx->tris, or a
// pass's mapped copy) less id_base, renumbered, plus id_base; the vertices with used_v: positions, normals, keys and
// lowmin as the run has them, and the vertex values of AUX_VALUES when `values`.  Waits once, for the two totals and
// the pass's own counters (copied to `pass`); the rest is stream-ordered, and the caller synchronises before it
// returns.  newV / newT receive the new counts.
static int compact_mesh(ctr_ctx* ctx, const CompactBufs& b, unsigned nV, unsigned nT, const int* tris, unsigned id_base,
                        bool values, void* pass, size_t& newV, size_t& newT) {
  cudaStream_t st = ctx->stream;
  const uint32_t fl = ctx->last_flags;
  const size_t gsz = (fl & CTR_GEOM_F64) ? 8 : 4;
  CompactCounters* ctr = (CompactCounters*)(b.scan + b.ctr_off);
  unsigned long long* st_t = (unsigned long long*)((char*)ctr + 64);
  unsigned long long* st_v = st_t + b.tiles_t + 1;
  CTR_CUDA(ctx, cudaMemsetAsync(ctr, 0, b.scan_bytes - b.ctr_off, st));
  if (nT) {
    k_flag_scan<<<b.tiles_t, SC_THREADS, 0, st>>>(b.keep_t, nT, b.idx_t, st_t, &ctr->ticket[0], &ctr->total[0], b.tiles_t);
    ctx->launches++;
  }
  if (nV) {
    k_flag_scan<<<b.tiles_v, SC_THREADS, 0, st>>>(b.used_v, nV, b.idx_v, st_v, &ctr->ticket[1], &ctr->total[1], b.tiles_v);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  char hbuf[64 + sizeof(CompactCounters)];
  CTR_CUDA(ctx, cudaMemcpyAsync(hbuf, b.scan, b.ctr_off + sizeof(CompactCounters), cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  CompactCounters h;
  memcpy(&h, hbuf + b.ctr_off, sizeof h);
  if (b.pass_bytes) memcpy(pass, hbuf, b.pass_bytes);
  newT = (size_t)h.total[0];
  newV = (size_t)h.total[1];
  auto rows = [&](void* p, size_t row_bytes) -> int {   // rows of one byte or of whole 32-bit words
    k_sel_rows<<<(nV + 255) / 256, 256, 0, st>>>((const uint32_t*)p, (uint32_t*)b.stage, b.used_v, b.idx_v, nV,
                                                 (int)(row_bytes / 4));
    ctx->launches++;
    if (newV) CTR_CUDA(ctx, cudaMemcpyAsync(p, b.stage, newV * row_bytes, cudaMemcpyDeviceToDevice, st));
    return 0;
  };
  int rc;
  if (nV) {
    if ((rc = rows(ctx->verts.p, 3 * gsz))) return rc;
    if ((fl & CTR_WANT_NORMALS) && (rc = rows(ctx->normals.p, 3 * gsz))) return rc;
    if ((fl & CTR_WANT_KEYS) && (rc = rows(ctx->keys.p, 8))) return rc;
    if ((fl & CTR_WANT_KEYS) && (rc = rows(ctx->lowmin.p, 1))) return rc;
    if (values && (rc = rows(ctx->aux[AUX_VALUES].p, (size_t)ctx->attr_ncomp * gsz))) return rc;
  }
  if (nT) {
    k_sel_tris<<<(nT + 255) / 256, 256, 0, st>>>(tris, (int*)b.stage, b.keep_t, b.idx_t, b.idx_v, nT, id_base);
    ctx->launches++;
    if (newT) CTR_CUDA(ctx, cudaMemcpyAsync(ctx->tris.p, b.stage, newT * 12, cudaMemcpyDeviceToDevice, st));
  }
  CTR_CUDA(ctx, cudaGetLastError());
  return 0;
}
