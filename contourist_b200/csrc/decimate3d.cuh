// Quadric vertex-clustering decimation of the 3D device mesh (ctr_mt3d_decimate; Lindstrom 2000, the GPU form of
// DeCoro & Tatarchuk 2007, VTK's vtkQuadricClustering).
//
// Included into mt3d.cu after mt3d_clean.cuh, inside its anonymous namespace: clustering is the clean-up's quantize
// step with another cell key, so the pass runs that step's kernels through its helpers (cluster_bufs, cluster_tris),
// compacts with compact_mesh (compact3d.cuh) and takes the normals of normals3d.cuh.  The definition is
// oracle/mt3d_decimate.py:decimate (positions within rounding: the sums below are fp64 atomics in an unspecified order;
// everything else exactly).
//   k_d_ids               : every triangle id in [0, n_verts), checked (and synchronised) before anything else runs;
//   k_c_qinsert / k_c_qmap: with CellKey, every vertex's cluster = the smallest vertex id in its cell (out-of-range cell
//                           indices flagged there); k_c_qtris / k_c_qdedupe: triangles through that map, those with
//                           fewer than three clusters or an earlier equal triple dropped (collision retry included);
//   k_d_vsum              : per vertex, P - lo and 1 added to its cluster's row;
//   k_d_quadric           : per triangle, n n^T and d n added to the row of each corner's cluster (d = -(n . (P_a - lo)));
//                           triangles with fewer than three clusters counted;
//   k_c_final             : (identity parents) flags the clusters the kept triangles use;
//   k_d_place             : per used cluster, the regularised 3 x 3 solve by the adjugate and the clamp to the cell,
//                           written into the representative's row of ctx->verts (every read of old positions is done);
//   compact_mesh          : vertices in the order of their representative, triangles through the cluster map;
//   k_s_nsum / k_s_nfin   : (CTR_WANT_NORMALS) normals of the decimated mesh, signed by the representative's old normal.
// The warp's lanes combine the rows they add to one cluster before the fp64 atomics (warp_add_row): triangles come out of
// the engine by owner word, so the lanes of a warp mostly hit the same few clusters.
// Scratch: AUX_SCRATCH1 only (cluster_bufs; its extra block holds the 13 fp64 sums per vertex row, reused for the normal
// sums after compaction).  No other aux slot is touched: vertex values and component results stay (stale).

constexpr int D_ROW = 13;                              // A: xx xy xz yy yz zz, g: x y z, position sums: x y z, count
constexpr double D_QLIM = 1048576.0;                   // cell indices lie in [-2^20, 2^20): 21 bits per axis

struct DecCounters {                                   // head of the scratch block
  CleanCounters c;                                     // k_c_qdedupe: n_quant (collapsed + duplicate), collision
  unsigned bad_ids, out_of_range, n_collapsed, n_clusters;
};

// q = floor((p - origin) / cell) per axis, offset into 3 x 21 bits; an index outside [-2^20, 2^20) (or NaN) raises the flag
struct CellKey {
  double origin[3], cell[3];
  unsigned* out_of_range;
  template <typename G>
  __device__ __forceinline__ unsigned long long operator()(const G* __restrict__ verts, unsigned v) const {
    unsigned long long key = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double q = floor(__ddiv_rn(__dsub_rn((double)verts[(size_t)v * 3 + a], origin[a]), cell[a]));
      if (!(q >= -D_QLIM && q < D_QLIM)) *out_of_range = 1u;
      key |= ((unsigned long long)((long long)q + (1ll << 20)) & 0x1fffffull) << (21 * a);
    }
    return key;
  }
};

struct DecParams {
  double origin[3], cell[3];
};

// the corner lo of the cell of point p (the same for every member of a cluster)
__device__ __forceinline__ void cell_lo(const DecParams& d, const double p[3], double lo[3]) {
#pragma unroll
  for (int a = 0; a < 3; ++a)
    lo[a] = __dadd_rn(d.origin[a], __dmul_rn(floor(__ddiv_rn(__dsub_rn(p[a], d.origin[a]), d.cell[a])), d.cell[a]));
}

__global__ void k_d_ids(const int* __restrict__ tris, size_t n, unsigned nv, DecCounters* ctr) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && (unsigned)tris[i] >= nv) ctr->bad_ids = 1u;
}

// row[key * D_ROW + i] += v[i] (i < N) for a whole warp: the lanes with one key (a __match_any_sync group) first sum
// their values by pointer jumping along the group (each lane adds its next peer's partial sum, then jumps twice as far;
// at most five rounds), then the group's first lane adds the sum.
template <int N>
__device__ __forceinline__ void warp_add_row(double* __restrict__ acc, int key, double (&v)[N], bool valid) {
  const unsigned act = __ballot_sync(0xffffffffu, valid);
  if (!valid) return;
  const unsigned lane = lane_id();
  const unsigned peers = __match_any_sync(act, key);
  const unsigned after = peers & ~((2u << lane) - 1u);
  int nxt = after ? __ffs(after) - 1 : -1;
  while (__any_sync(act, nxt >= 0)) {
    const int src = nxt >= 0 ? nxt : (int)lane;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const double o = __shfl_sync(act, v[i], src);
      if (nxt >= 0) v[i] = __dadd_rn(v[i], o);
    }
    nxt = __shfl_sync(act, nxt, src);
  }
  if (peers & ((1u << lane) - 1u)) return;            // not the first lane of its group
  double* r = acc + (size_t)key * D_ROW;
#pragma unroll
  for (int i = 0; i < N; ++i) atomicAdd(r + i, v[i]);
}

template <typename G>
__global__ void __launch_bounds__(256) k_d_vsum(const G* __restrict__ verts, unsigned nv, const int* __restrict__ rep, DecParams d,
                                                double* __restrict__ acc, DecCounters* ctr) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = v < nv;
  int k = 0;
  double s[4] = {0.0, 0.0, 0.0, 1.0};
  if (in) {
    k = rep[v];
    double p[3], lo[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) p[a] = (double)verts[(size_t)v * 3 + a];
    cell_lo(d, p, lo);
#pragma unroll
    for (int a = 0; a < 3; ++a) s[a] = __dsub_rn(p[a], lo[a]);
  }
  const unsigned reps = __ballot_sync(0xffffffffu, in && k == (int)v);
  if (lane_id() == 0 && reps) atomicAdd(&ctr->n_clusters, (unsigned)__popc(reps));
  warp_add_row(acc + 9, k, s, in);
}

template <typename G>
__global__ void __launch_bounds__(256) k_d_quadric(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                   const int* __restrict__ rep, DecParams d, double* __restrict__ acc,
                                                   DecCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = t < nt;
  int v[3] = {0, 0, 0}, k[3] = {0, 0, 0};
  double p[3][3] = {}, n[3] = {0.0, 0.0, 0.0};
  if (in) {
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      v[q] = tris[(size_t)t * 3 + q];
      k[q] = rep[v[q]];
    }
    tri_corners(verts, v, p);
    // cross(P_b - P_a, P_c - P_a) in the expression order of k_s_nsum
    const double ux = __dsub_rn(p[1][0], p[0][0]), uy = __dsub_rn(p[1][1], p[0][1]), uz = __dsub_rn(p[1][2], p[0][2]);
    const double wx = __dsub_rn(p[2][0], p[0][0]), wy = __dsub_rn(p[2][1], p[0][1]), wz = __dsub_rn(p[2][2], p[0][2]);
    n[0] = __dsub_rn(__dmul_rn(uy, wz), __dmul_rn(uz, wy));
    n[1] = __dsub_rn(__dmul_rn(uz, wx), __dmul_rn(ux, wz));
    n[2] = __dsub_rn(__dmul_rn(ux, wy), __dmul_rn(uy, wx));
  }
  const unsigned collapsed = __ballot_sync(0xffffffffu, in && (k[0] == k[1] || k[0] == k[2] || k[1] == k[2]));
  if (lane_id() == 0 && collapsed) atomicAdd(&ctr->n_collapsed, (unsigned)__popc(collapsed));
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    double lo[3];
    cell_lo(d, p[q], lo);                               // the corner of corner q's cluster
    const double rx = __dsub_rn(p[0][0], lo[0]), ry = __dsub_rn(p[0][1], lo[1]), rz = __dsub_rn(p[0][2], lo[2]);
    const double dd = -__dadd_rn(__dadd_rn(__dmul_rn(n[0], rx), __dmul_rn(n[1], ry)), __dmul_rn(n[2], rz));
    double s[9] = {__dmul_rn(n[0], n[0]), __dmul_rn(n[0], n[1]), __dmul_rn(n[0], n[2]), __dmul_rn(n[1], n[1]),
                   __dmul_rn(n[1], n[2]), __dmul_rn(n[2], n[2]), __dmul_rn(dd, n[0]), __dmul_rn(dd, n[1]),
                   __dmul_rn(dd, n[2])};
    warp_add_row(acc, k[q], s, in);
  }
}

// x = argmin sum (n . x + d)^2 + lambda |x - m|^2, lambda = 1e-3 trace(A): (A + lambda I) x = lambda m - g, by the
// adjugate; x = m where lambda == 0; each axis clamped to [0, cell]
template <typename G>
__global__ void __launch_bounds__(256) k_d_place(G* __restrict__ verts, unsigned nv, const uint8_t* __restrict__ used,
                                                 DecParams d, const double* __restrict__ acc) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv || !used[v]) return;                    // used[] is set on representatives only
  const double* r = acc + (size_t)v * D_ROW;
  double p[3], lo[3], m[3], x[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) p[a] = (double)verts[(size_t)v * 3 + a];
  cell_lo(d, p, lo);
#pragma unroll
  for (int a = 0; a < 3; ++a) m[a] = __ddiv_rn(r[9 + a], r[12]);
  const double lam = __dmul_rn(1e-3, __dadd_rn(__dadd_rn(r[0], r[3]), r[5]));
  if (lam == 0.0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) x[a] = m[a];
  } else {
    const double a00 = __dadd_rn(r[0], lam), a01 = r[1], a02 = r[2], a11 = __dadd_rn(r[3], lam), a12 = r[4],
                 a22 = __dadd_rn(r[5], lam);
    const double b0 = __dsub_rn(__dmul_rn(lam, m[0]), r[6]), b1 = __dsub_rn(__dmul_rn(lam, m[1]), r[7]),
                 b2 = __dsub_rn(__dmul_rn(lam, m[2]), r[8]);
    const double c00 = __dsub_rn(__dmul_rn(a11, a22), __dmul_rn(a12, a12));
    const double c01 = __dsub_rn(__dmul_rn(a02, a12), __dmul_rn(a01, a22));
    const double c02 = __dsub_rn(__dmul_rn(a01, a12), __dmul_rn(a02, a11));
    const double c11 = __dsub_rn(__dmul_rn(a00, a22), __dmul_rn(a02, a02));
    const double c12 = __dsub_rn(__dmul_rn(a01, a02), __dmul_rn(a00, a12));
    const double c22 = __dsub_rn(__dmul_rn(a00, a11), __dmul_rn(a01, a01));
    const double det = __dadd_rn(__dadd_rn(__dmul_rn(a00, c00), __dmul_rn(a01, c01)), __dmul_rn(a02, c02));
    x[0] = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(c00, b0), __dmul_rn(c01, b1)), __dmul_rn(c02, b2)), det);
    x[1] = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(c01, b0), __dmul_rn(c11, b1)), __dmul_rn(c12, b2)), det);
    x[2] = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(c02, b0), __dmul_rn(c12, b1)), __dmul_rn(c22, b2)), det);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) verts[(size_t)v * 3 + a] = (G)__dadd_rn(lo[a], fmin(fmax(x[a], 0.0), d.cell[a]));
}

template <typename G>
int decimate_typed(ctr_ctx* ctx, const ctr_decimate_params* dp, ctr_decimate_counts* out) {
  cudaStream_t st = ctx->stream;
  const unsigned nV = (unsigned)ctx->last_counts[0], nT = (unsigned)ctx->last_counts[1];
  if (!nV && !nT) return 0;                           // empty mesh: a valid no-op
  DecParams d;
  CellKey key;
  for (int a = 0; a < 3; ++a) {
    d.origin[a] = key.origin[a] = dp->origin[a];
    d.cell[a] = key.cell[a] = dp->cell[a];
  }
  int rc;
  ClusterBufs b;
  if ((rc = cluster_bufs(ctx, nV, nT, sizeof(G), sizeof(DecCounters), (size_t)nV * D_ROW * 8, b))) return rc;
  DecCounters* dc = (DecCounters*)b.head;
  key.out_of_range = &dc->out_of_range;
  double* acc = (double*)b.extra;
  G* verts = (G*)ctx->verts.p;
  const int* tris = (const int*)ctx->tris.p;
  const unsigned vb = (nV + 255) / 256, tb = (nT + 255) / 256;
  DecCounters h;
  memset(&h, 0, sizeof h);
  if (nT) {                                           // qtris reads rep[] through the ids: check them first
    const size_t n3 = (size_t)nT * 3;
    CTR_CUDA(ctx, cudaMemsetAsync(dc, 0, sizeof(DecCounters), st));
    k_d_ids<<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(tris, n3, nV, dc);
    ctx->launches++;
    CTR_CUDA(ctx, cudaMemcpyAsync(&h, dc, sizeof h, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (h.bad_ids) return ctr_fail(ctx, CTR_ERR_STATE, "triangle ids outside [0, n_verts): the ids were shifted (ctr_mt3d_offset_ids)");
  }
  if ((rc = cluster_tris<G>(ctx, verts, nV, tris, nT, key, b, &h, sizeof h))) return rc;
  if (h.out_of_range) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "a cell index (p - origin) / cell lies outside [-2^20, 2^20)");
  ctx->mesh_gen++;                                    // from here on the mesh is edited
  ctx->last3_edited |= EDIT_DECIMATE;
  CTR_CUDA(ctx, cudaMemsetAsync(acc, 0, (size_t)nV * D_ROW * 8, st));
  k_d_vsum<G><<<vb, 256, 0, st>>>(verts, nV, b.rep, d, acc, dc);
  ctx->launches++;
  if (nT) {
    k_d_quadric<G><<<tb, 256, 0, st>>>(verts, tris, nT, b.rep, d, acc, dc);
    k_c_final<<<tb, 256, 0, st>>>(b.tris2, nT, b.cb.keep_t, b.parent_b, b.cb.used_v, &dc->c);   // parent_b: identity (k_c_init)
    k_d_place<G><<<vb, 256, 0, st>>>(verts, nV, b.cb.used_v, d, acc);
    ctx->launches += 3;
  }
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, dc, sizeof h, cudaMemcpyDeviceToHost, st));   // (synchronised by compact_mesh)
  size_t newV = 0, newT = 0;
  if (nT && (rc = compact_mesh(ctx, b.cb, nV, nT, b.tris2, 0u, false, nullptr, newV, newT))) return rc;
  if ((ctx->last_flags & CTR_WANT_NORMALS) && newT) {
    CTR_CUDA(ctx, cudaMemsetAsync(acc, 0, newV * 3 * 8, st));
    k_s_nsum<G><<<(unsigned)((newT + N_THREADS - 1) / N_THREADS), N_THREADS, 0, st>>>(verts, tris, (unsigned)newT, acc);
    k_s_nfin<G><<<(unsigned)((newV + N_THREADS - 1) / N_THREADS), N_THREADS, 0, st>>>(acc, (unsigned)newV, (G*)ctx->normals.p);
    ctx->launches += 2;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  out->n_verts = (int64_t)newV;
  out->n_tris = (int64_t)newT;
  out->n_clusters = h.n_clusters;
  out->n_collapsed = h.n_collapsed;
  out->n_duplicate = (int64_t)h.c.n_quant - (int64_t)h.n_collapsed;
  return 0;
}
