// The reference's mesh post-processing on the device mesh of the last ctr_mt3d_run (SURVEY.md 8 a10, a11, a13, f1) --
// included by mesh3d.cu inside its anonymous namespace, after compact3d.cuh.
//
//   tetrahedral.py:190-215    quantize_interpolations : interpolations that truncate to the same cell of the
//                             `divisions` grid become one vertex; simplices that lose a vertex, or equal another, go;
//   tetrahedral.py:353-375    remove_tiny_simplices   : a simplex whose extent is < epsilon of the grid on every axis
//                             is dropped and its vertices moved to one point;
//   surface_geometry.py:14-50 clean_triangles         : zero-area triangles are dropped, coincident vertices of those
//                             triangles merged, vertices renumbered over what the kept triangles use.
// In the reference all three depend on CPython dict / set iteration order.  Here the order is fixed: wherever the
// reference keeps "whichever came first / last", the vertex with the SMALLEST id survives (ids are the engine's
// deterministic numbering), and the sequential overwrite passes become "decide every simplex from the positions
// before the pass, then merge connected clusters" (lock-free union-find whose roots are minima).  oracle/post3d.py
// states the same rules in numpy and is pinned to final meshes of the unmodified reference.
//
//   k_c_qinsert / k_c_qmap : quantum cell (3 x 21 bits) -> open-addressing table, value = smallest vertex id in the cell;
//   k_c_qtris / k_c_qdedupe: triangles through that map; the distinct ones go into a second table keyed by a 64-bit
//                            hash of the sorted triple, value = smallest triangle index; a triangle that finds another
//                            index there compares the triples (equal: duplicate, dropped; different: a hash collision,
//                            reported to the host, which retries with another seed);
//   k_c_tiny / k_c_tinypos : extent test, union of the three vertices, positions of non-roots overwritten by their root's;
//   k_c_flat / k_c_final   : cross-product test, union of np.allclose vertex pairs of flat triangles, kept triangles
//                            mapped through the merge and checked for lost vertices; used-vertex flags;
//   compact_mesh           : order-preserving compaction of vertices, normals, keys and the mapped triangles;
//   k_c_transform          : grid -> world (grid_field.py:89-93) at the very end, after the optional orientation pass,
//                            which the reference also runs in grid coordinates (tetrahedral.py:611-617).

struct CleanCounters {
  unsigned n_quant, n_tiny, n_flat, collision;
};

__device__ __forceinline__ double c_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double c_sub(double a, double b) { return __dsub_rn(a, b); }

template <typename G>
__device__ __forceinline__ unsigned long long quantum_key(const G* __restrict__ verts, unsigned v, const double ex[3]) {
  unsigned long long key = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const long long q = (long long)c_mul((double)verts[(size_t)v * 3 + a], ex[a]);     // astype(int): towards zero
    key |= ((unsigned long long)q & 0x1fffffull) << (21 * a);
  }
  return key;
}

struct Expander {                                     // quantize's cell key (also the scale of the tiny-simplex test)
  double ex[3];
  double inv[3];
  template <typename G>
  __device__ __forceinline__ unsigned long long operator()(const G* __restrict__ verts, unsigned v) const {
    return quantum_key(verts, v, ex);
  }
};

__global__ void k_c_init(ufh::Slot* tab_v, size_t nslots_v, ufh::Slot* tab_t, size_t nslots_t, int* parent_a, int* parent_b,
                         uint8_t* used, unsigned nv) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t; q < nslots_v; q += n) reinterpret_cast<int4*>(tab_v)[q] = make_int4(-1, -1, 0x7fffffff, 0);
  for (size_t q = t; q < nslots_t; q += n) reinterpret_cast<int4*>(tab_t)[q] = make_int4(-1, -1, 0x7fffffff, 0);
  for (size_t q = t; q < nv; q += n) {
    parent_a[q] = (int)q;
    parent_b[q] = (int)q;
    used[q] = 0;
  }
}

// Key: a functor (verts, v) -> 63-bit cell key of vertex v (Expander here, CellKey in decimate3d.cuh)
template <typename G, typename Key>
__global__ void k_c_qinsert(const G* __restrict__ verts, unsigned nv, Key key, ufh::Slot* tab, size_t mask) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  atomicMin(&ufh::hash_slot(tab, mask, key(verts, v), true)->tri, (int)v);
}

template <typename G, typename Key>
__global__ void k_c_qmap(const G* __restrict__ verts, unsigned nv, Key key, ufh::Slot* tab, size_t mask, int* __restrict__ rep) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  rep[v] = ufh::hash_slot(tab, mask, key(verts, v), false)->tri;
}

__device__ __forceinline__ void sort3(int& a, int& b, int& c) {
  int t;
  if (a > b) { t = a; a = b; b = t; }
  if (b > c) { t = b; b = c; c = t; }
  if (a > b) { t = a; a = b; b = t; }
}

__device__ __forceinline__ unsigned long long triple_hash(int a, int b, int c, unsigned long long seed) {
  sort3(a, b, c);
  unsigned long long h = ufh::mix64(((unsigned long long)(unsigned)a << 32 | (unsigned)b) + seed);
  h = ufh::mix64(h ^ ((unsigned long long)(unsigned)c * 0x9e3779b97f4a7c15ull));
  return h == ufh::EMPTY ? 0ull : h;
}

// quantize: triangles through the representative map; keep[t] = 1 for triangles that still have three vertices
__global__ void k_c_qtris(const int* __restrict__ tris, unsigned nt, const int* __restrict__ rep, int* __restrict__ tris2,
                          uint8_t* __restrict__ keep, ufh::Slot* tab, size_t mask, unsigned long long seed) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int a = rep[tris[(size_t)t * 3]], b = rep[tris[(size_t)t * 3 + 1]], c = rep[tris[(size_t)t * 3 + 2]];
  tris2[(size_t)t * 3] = a;
  tris2[(size_t)t * 3 + 1] = b;
  tris2[(size_t)t * 3 + 2] = c;
  const bool distinct = a != b && a != c && b != c;                                    // tetrahedral.py:208
  keep[t] = distinct ? 1 : 0;
  if (distinct) atomicMin(&ufh::hash_slot(tab, mask, triple_hash(a, b, c, seed), true)->tri, (int)t);
}

// simplex_sets is a set of frozensets (tetrahedral.py:209): of equal triples the first in triangle order stays
__global__ void k_c_qdedupe(const int* __restrict__ tris2, unsigned nt, uint8_t* __restrict__ keep, ufh::Slot* tab, size_t mask,
                            unsigned long long seed, CleanCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  if (!keep[t]) {
    atomicAdd(&ctr->n_quant, 1u);
    return;
  }
  int a = tris2[(size_t)t * 3], b = tris2[(size_t)t * 3 + 1], c = tris2[(size_t)t * 3 + 2];
  const int m = ufh::hash_slot(tab, mask, triple_hash(a, b, c, seed), false)->tri;
  if (m == (int)t) return;
  int ma = tris2[(size_t)m * 3], mb = tris2[(size_t)m * 3 + 1], mc = tris2[(size_t)m * 3 + 2];
  sort3(a, b, c);
  sort3(ma, mb, mc);
  if (a == ma && b == mb && c == mc) {
    keep[t] = 0;
    atomicAdd(&ctr->n_quant, 1u);
  } else {
    atomicAdd(&ctr->collision, 1u);
  }
}

template <typename G>
__global__ void k_c_tiny(const G* __restrict__ verts, const int* __restrict__ tris2, unsigned nt, uint8_t* __restrict__ keep,
                         Expander e, double epsilon, int* parent, CleanCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  const int v[3] = {tris2[(size_t)t * 3], tris2[(size_t)t * 3 + 1], tris2[(size_t)t * 3 + 2]};
  double worst = -INFINITY;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) {
    const double p0 = (double)verts[(size_t)v[0] * 3 + ax], p1 = (double)verts[(size_t)v[1] * 3 + ax],
                 p2 = (double)verts[(size_t)v[2] * 3 + ax];
    const double d = c_mul(c_sub(fmax(p0, fmax(p1, p2)), fmin(p0, fmin(p1, p2))), e.inv[ax]);   // tetrahedral.py:363-365
    worst = fmax(worst, d);
  }
  if (worst < epsilon) {                                                                // :366
    keep[t] = 0;
    atomicAdd(&ctr->n_tiny, 1u);
    ufh::uf_union(parent, v[0], v[1]);
    ufh::uf_union(parent, v[0], v[2]);
  }
}

// non-roots take their root's position; roots are never written, so this runs in place
template <typename G>
__global__ void k_c_tinypos(G* __restrict__ verts, unsigned nv, int* parent) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  int r = (int)v;
  for (int q = parent[r]; q != r; q = parent[r]) r = q;
  if (r == (int)v) return;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) verts[(size_t)v * 3 + ax] = verts[(size_t)r * 3 + ax];
}

__device__ __forceinline__ bool close_to(const double p[3], const double q[3]) {       // np.allclose(p, q)
  bool ok = true;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) ok = ok && fabs(c_sub(p[ax], q[ax])) <= __dadd_rn(1e-8, c_mul(1e-5, fabs(q[ax])));
  return ok;
}

template <typename G>
__global__ void k_c_flat(const G* __restrict__ verts, const int* __restrict__ tris2, unsigned nt, uint8_t* __restrict__ keep,
                         int* parent, CleanCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  const int v[3] = {tris2[(size_t)t * 3], tris2[(size_t)t * 3 + 1], tris2[(size_t)t * 3 + 2]};
  double P[3][3];
#pragma unroll
  for (int q = 0; q < 3; ++q)
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) P[q][ax] = (double)verts[(size_t)v[q] * 3 + ax];
  double u[3], w[3];
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) {
    u[ax] = c_sub(P[0][ax], P[2][ax]);                                                  // A - C
    w[ax] = c_sub(P[1][ax], P[2][ax]);                                                  // B - C
  }
  const double cx = c_sub(c_mul(u[1], w[2]), c_mul(u[2], w[1]));
  const double cy = c_sub(c_mul(u[2], w[0]), c_mul(u[0], w[2]));
  const double cz = c_sub(c_mul(u[0], w[1]), c_mul(u[1], w[0]));
  if (fabs(cx) <= 1e-8 && fabs(cy) <= 1e-8 && fabs(cz) <= 1e-8) {                       // np.allclose(cross, 0)
    keep[t] = 0;
    atomicAdd(&ctr->n_flat, 1u);
    if (close_to(P[0], P[1])) ufh::uf_union(parent, v[0], v[1]);                        // surface_geometry.py:39-44
    if (close_to(P[0], P[2])) ufh::uf_union(parent, v[0], v[2]);
    if (close_to(P[1], P[2])) ufh::uf_union(parent, v[1], v[2]);
  }
}

__global__ void k_c_final(int* __restrict__ tris2, unsigned nt, uint8_t* __restrict__ keep, int* parent, uint8_t* __restrict__ used,
                          CleanCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  int v[3];
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    int r = tris2[(size_t)t * 3 + q];
    for (int p = parent[r]; p != r; p = parent[r]) r = p;
    v[q] = r;
  }
  if (v[0] == v[1] || v[0] == v[2] || v[1] == v[2]) {
    keep[t] = 0;
    atomicAdd(&ctr->n_flat, 1u);
    return;
  }
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    tris2[(size_t)t * 3 + q] = v[q];
    used[v[q]] = 1;
  }
}

template <typename G>
__global__ void k_c_transform(G* __restrict__ verts, G* __restrict__ normals, unsigned nv, Xform xf) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax)
    verts[(size_t)v * 3 + ax] = add_rn(mul_rn(verts[(size_t)v * 3 + ax], (G)xf.delta[ax]), (G)xf.origin[ax]);   // grid_field.py:93
  if (normals) {
    G n[3], len2 = 0;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
      n[ax] = normals[(size_t)v * 3 + ax] * (G)xf.inv_delta[ax];
      len2 += n[ax] * n[ax];
    }
    const G inv = len2 > (G)0 ? inv_sqrt(len2) : (G)0;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) normals[(size_t)v * 3 + ax] = n[ax] * inv;
  }
}

// Scratch of the passes that cluster vertices by cell (clean-up, decimation), carved from AUX_SCRATCH1: the cell and
// triangle tables, the representative map, union-find parents, the compaction's pieces, mapped triangles, a `head`
// block for the pass's own counters, an `extra` block, and the staging rows.
struct ClusterBufs {
  ufh::Slot *tab_v, *tab_t;
  size_t nslots_v, nslots_t;
  int *rep, *parent_a, *parent_b, *tris2;
  void *head, *extra;
  CompactBufs cb;
};

static int cluster_bufs(ctr_ctx* ctx, unsigned nV, unsigned nT, size_t gsz, size_t head_bytes, size_t extra_bytes, ClusterBufs& b) {
  b.nslots_v = 1024;
  b.nslots_t = 1024;
  while (b.nslots_v < (size_t)nV * 2) b.nslots_v <<= 1;
  while (b.nslots_t < (size_t)nT * 2) b.nslots_t <<= 1;
  return ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH1], [&](ctr_carve& c) {
    c(b.tab_v, b.nslots_v * sizeof(ufh::Slot));
    c(b.tab_t, b.nslots_t * sizeof(ufh::Slot));
    c(b.rep, (size_t)nV * 4 + 4);
    c(b.parent_a, (size_t)nV * 4 + 4);
    c(b.parent_b, (size_t)nV * 4 + 4);
    compact_carve(c, nV, nT, 0, b.cb);
    c(b.tris2, (size_t)nT * 12 + 16);
    c(b.head, head_bytes + 64);
    c(b.extra, extra_bytes);
    c(b.cb.stage, std::max<size_t>((size_t)nV * 3 * gsz, (size_t)nT * 12) + 16);
  });
}

// k_c_init, every vertex's representative (the smallest vertex id in its cell of `key`), the triangles through that map
// and their de-duplication; retried with another seed while the triangle table reports a hash collision.  `head` (hbytes)
// starts with the CleanCounters that k_c_qdedupe counts into: it is zeroed before each attempt and copied to `h` at
// the sync that checks for collisions.
template <typename G, typename Key>
int cluster_tris(ctr_ctx* ctx, const G* verts, unsigned nV, const int* tris, unsigned nT, const Key& key, const ClusterBufs& b,
                 void* h, size_t hbytes) {
  cudaStream_t st = ctx->stream;
  const unsigned vb = (nV + 255) / 256, tb = (nT + 255) / 256;
  CleanCounters* dcc = (CleanCounters*)b.head;
  for (int attempt = 0;; ++attempt) {
    const unsigned long long seed = 0x51ed270b1a2c3d4full * (unsigned long long)(attempt + 1);
    CTR_CUDA(ctx, cudaMemsetAsync(b.head, 0, hbytes, st));
    k_c_init<<<ctx->sm_count * 8, 256, 0, st>>>(b.tab_v, b.nslots_v, b.tab_t, b.nslots_t, b.parent_a, b.parent_b, b.cb.used_v, nV);
    k_c_qinsert<G><<<vb, 256, 0, st>>>(verts, nV, key, b.tab_v, b.nslots_v - 1);
    k_c_qmap<G><<<vb, 256, 0, st>>>(verts, nV, key, b.tab_v, b.nslots_v - 1, b.rep);
    ctx->launches += 3;
    if (nT) {
      k_c_qtris<<<tb, 256, 0, st>>>(tris, nT, b.rep, b.tris2, b.cb.keep_t, b.tab_t, b.nslots_t - 1, seed);
      k_c_qdedupe<<<tb, 256, 0, st>>>(b.tris2, nT, b.cb.keep_t, b.tab_t, b.nslots_t - 1, seed, dcc);
      ctx->launches += 2;
    }
    CTR_CUDA(ctx, cudaMemcpyAsync(h, b.head, hbytes, cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    if (!((const CleanCounters*)h)->collision) return 0;
    if (attempt == 3) return ctr_fail(ctx, CTR_ERR_STATE, "triangle de-duplication: hash collisions under four seeds");
  }
}

template <typename G>
int clean_typed(ctr_ctx* ctx, const ctr_clean_params* cp, ctr_clean_counts* out) {
  cudaStream_t st = ctx->stream;
  const unsigned nV = (unsigned)ctx->last_counts[0], nT = (unsigned)ctx->last_counts[1];
  const bool want_n = (ctx->last_flags & CTR_WANT_NORMALS) != 0;
  Expander e;
  for (int a = 0; a < 3; ++a) {
    e.ex[a] = (double)(long long)(((double)cp->divisions * 1.0) / (double)cp->corner[a]);   // tetrahedral.py:192
    e.inv[a] = 1.0 / (double)cp->corner[a];                                                  // :360
  }
  Xform xf;
  bool identity = true;
  for (int a = 0; a < 3; ++a) {
    xf.origin[a] = cp->origin[a];
    xf.delta[a] = cp->delta[a];
    xf.inv_delta[a] = 1.0 / cp->delta[a];
    identity = identity && cp->origin[a] == 0.0 && cp->delta[a] == 1.0;
  }
  int rc;
  ClusterBufs b;
  if ((rc = cluster_bufs(ctx, nV, nT, sizeof(G), sizeof(CleanCounters), 0, b))) return rc;
  CleanCounters* dcc = (CleanCounters*)b.head;
  G* verts = (G*)ctx->verts.p;
  const int* tris = (const int*)ctx->tris.p;
  const unsigned vb = (nV + 255) / 256, tb = (nT + 255) / 256;
  CleanCounters hc;
  memset(&hc, 0, sizeof hc);
  size_t newV = 0, newT = 0;
  if (nV && nT && (rc = cluster_tris<G>(ctx, verts, nV, tris, nT, e, b, &hc, sizeof hc))) return rc;
  mesh_edited(ctx, EDIT_CLEAN);
  if (nV && nT) {
    k_c_tiny<G><<<tb, 256, 0, st>>>(verts, b.tris2, nT, b.cb.keep_t, e, cp->epsilon, b.parent_a, dcc);
    k_c_tinypos<G><<<vb, 256, 0, st>>>(verts, nV, b.parent_a);
    if (!(cp->flags & CTR_CLEAN_NO_TRIANGLES)) k_c_flat<G><<<tb, 256, 0, st>>>(verts, b.tris2, nT, b.cb.keep_t, b.parent_b, dcc);
    k_c_final<<<tb, 256, 0, st>>>(b.tris2, nT, b.cb.keep_t, b.parent_b, b.cb.used_v, dcc);
    ctx->launches += 4;
    CTR_CUDA(ctx, cudaMemcpyAsync(&hc, dcc, sizeof hc, cudaMemcpyDeviceToHost, st));   // (synchronised by compact_mesh)
    if ((rc = compact_mesh(ctx, b.cb, nV, nT, b.tris2, 0u, false, nullptr, newV, newT))) return rc;
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  out->n_verts = (int64_t)newV;
  out->n_tris = (int64_t)newT;
  out->n_quantized = hc.n_quant;
  out->n_tiny = hc.n_tiny;
  out->n_flat = hc.n_flat;
  out->n_components = 0;
  out->n_flipped = 0;
  if ((cp->flags & CTR_CLEAN_ORIENT) && newT) {
    // surface_geometry.py:52-140, in grid coordinates like the reference (tetrahedral.py:611-617)
    if ((rc = ctr_mt3d_orient_reference(ctx, &out->n_components, &out->n_flipped))) return rc;
  }
  if (!identity && newV) {
    k_c_transform<G><<<(unsigned)((newV + 255) / 256), 256, 0, st>>>(verts, want_n ? (G*)ctx->normals.p : nullptr, (unsigned)newV, xf);
    ctx->launches++;
    CTR_CUDA(ctx, cudaGetLastError());
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  return 0;
}
