// Connected components of the 3D device mesh with per-component size and topology (ctr_mt3d_components).
//
// Included into mesh3d.cu, inside its anonymous namespace: the pass shares the orientation pass's edge table
// (edge_key / edge_slot), its union-find step (k_o_union) and its order-preserving key (okey).  The definition is
// oracle/mt3d_components.py:components.
//   k_m_init      : empty edge table (slot.tri = INT_MAX, slot.pad = 0 uses), empty (component, vertex) table, parent[t] = t;
//   k_m_edges     : every undirected edge of every triangle into the edge table: atomicMin of the smallest triangle on
//                   it, one use more in slot.pad; flags triangle ids outside [0, n_verts) (the host then stops);
//   k_o_union     : (the orientation pass's) each triangle joins the smallest triangle of each of its edges;
//   k_m_roots     : parent[] flattened to the roots (roots are minima), the roots numbered in ascending order by a
//                   decoupled look-back over ticketed tiles: rank[root] = component, *total = C;
//   k_m_table_init: C empty rows of the table (box as okeys: lo = max key, hi = 0);
//   k_m_tris      : per triangle its component, area, count and box; per edge it owns (slot.tri == t) one edge, boundary
//                   or non-manifold by its use count; per corner one vertex when its (component, vertex) insert is new;
//   k_m_box       : box keys back to doubles;
//   k_m_volume    : signed volume against the component's final lo.
// Sums into a component's row are combined over the lanes of a warp that share the component first (one atomic per
// group and field, instead of one per triangle on the address of a large component).

static_assert(sizeof(ctr_mt3d_component) == 112, "ctr_mt3d_component is 112 bytes");

constexpr int M_THREADS = 256;

struct MAdd {
  template <typename T> __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};
struct MMin {
  template <typename T> __device__ __forceinline__ T operator()(T a, T b) const { return b < a ? b : a; }
};
struct MMax {
  template <typename T> __device__ __forceinline__ T operator()(T a, T b) const { return b > a ? b : a; }
};

// op over the values of the lanes in `peers`; every lane of `peers` calls it and gets the result
template <typename T, typename Op>
__device__ __forceinline__ T peer_reduce(unsigned peers, T v, Op op) {
  if (peers == 0xffffffffu) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
  }
  unsigned m = peers;
  T acc = __shfl_sync(peers, v, __ffs(m) - 1);
  for (m &= m - 1; m; m &= m - 1) acc = op(acc, __shfl_sync(peers, v, __ffs(m) - 1));
  return acc;
}

__device__ __forceinline__ double okey_value(unsigned long long k) {   // inverse of okey
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// inserts `key`; true when this call inserted it (ufh::hash_slot does not tell an insert from a hit)
__device__ __forceinline__ bool hash_insert_new(EdgeSlot* tab, size_t mask, unsigned long long key) {
  size_t s = (size_t)ufh::mix64(key) & mask;
  while (true) {
    unsigned long long k = tab[s].key;
    if (k == key) return false;
    if (k == EMPTY) {
      k = atomicCAS(&tab[s].key, EMPTY, key);
      if (k == EMPTY) return true;
      if (k == key) return false;
    }
    s = (s + 1) & mask;
  }
}

struct MCounters {                                    // head of the scratch block, then one look-back word per tile
  unsigned bad, ticket;
  unsigned long long total;
};

__global__ void k_m_init(EdgeSlot* etab, EdgeSlot* vtab, size_t nslots, int* parent, unsigned nt) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t; q < nslots; q += n) {
    reinterpret_cast<int4*>(etab)[q] = make_int4(-1, -1, 0x7fffffff, 0);
    reinterpret_cast<int4*>(vtab)[q] = make_int4(-1, -1, 0, 0);
  }
  for (size_t q = t; q < nt; q += n) parent[q] = (int)q;
}

__global__ void k_m_edges(const int* __restrict__ tris, unsigned nt, unsigned nv, EdgeSlot* tab, size_t mask, MCounters* ctr) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
  if ((unsigned)v[0] >= nv || (unsigned)v[1] >= nv || (unsigned)v[2] >= nv) {   // (a key of two ids -1 would be EMPTY)
    ctr->bad = 1u;
    return;
  }
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    EdgeSlot* s = edge_slot(tab, mask, edge_key(v[e], v[(e + 1) % 3]), true);
    atomicMin(&s->tri, (int)t);
    atomicAdd(&s->pad, 1);
  }
}

__global__ void __launch_bounds__(M_THREADS) k_m_roots(int* parent, unsigned nt, int* __restrict__ rank, unsigned long long* status,
                                                       MCounters* ctr, int ntiles) {
  __shared__ unsigned s_tile;
  __shared__ unsigned s_warp[M_THREADS / 32];
  __shared__ unsigned long long s_excl;
  if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket, 1u);
  __syncthreads();
  const int tile = (int)s_tile;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned t = (unsigned)tile * M_THREADS + threadIdx.x;
  bool root = false;
  if (t < nt) {
    int r = (int)t;                                   // no unions any more: walk read-only, then one compressing write
    for (int q = parent[r]; q != r; q = parent[r]) r = q;
    if (r != (int)t) parent[t] = r;
    else root = true;
  }
  const unsigned b = __ballot_sync(0xffffffffu, root);
  if (lane == 0) s_warp[warp] = __popc(b);
  __syncthreads();
  unsigned woff = 0, blk = 0;
#pragma unroll
  for (int w = 0; w < M_THREADS / 32; ++w) {
    if (w < (int)warp) woff += s_warp[w];
    blk += s_warp[w];
  }
  if (warp == 0) {
    const unsigned long long e = lb_lookback(status, tile, (unsigned long long)blk);
    if (lane == 0) s_excl = e;
  }
  __syncthreads();
  if (root) rank[t] = (int)(s_excl + woff + __popc(b & ((1u << lane) - 1u)));
  if (tile == ntiles - 1 && threadIdx.x == 0) ctr->total = s_excl + blk;
}

__global__ void k_m_table_init(ctr_mt3d_component* comp, unsigned nc) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nc) return;
  ctr_mt3d_component c;
  memset(&c, 0, sizeof c);
  unsigned long long* lo = reinterpret_cast<unsigned long long*>(c.lo);
  lo[0] = lo[1] = lo[2] = ~0ull;
  comp[q] = c;
}

template <typename G>
__global__ void __launch_bounds__(M_THREADS) k_m_tris(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                      const int* __restrict__ parent, const int* __restrict__ rank, EdgeSlot* etab,
                                                      EdgeSlot* vtab, size_t mask, int* __restrict__ label, ctr_mt3d_component* comp) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = t < nt;
  const unsigned act = __ballot_sync(0xffffffffu, in);
  if (!in) return;
  const int r = parent[t];
  const int l = rank[r];
  label[t] = l;
  if (r == (int)t) comp[l].first_tri = (int64_t)t;
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
  // counts of this triangle, one byte each: owned edges | boundary << 8 | non-manifold << 16 | new vertices << 24 (a
  // warp's sums stay below 256)
  unsigned cnt = 0;
  unsigned long long k[3];
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    k[e] = edge_key(v[e], v[(e + 1) % 3]);
    if ((e > 0 && k[e] == k[0]) || (e > 1 && k[e] == k[1])) continue;     // an edge twice in a degenerate triangle
    const EdgeSlot* s = edge_slot(etab, mask, k[e], false);
    if (s->tri != (int)t) continue;                                        // owned by the smallest triangle on it
    const int uses = s->pad;
    cnt += 1u + (uses == 1 ? 1u << 8 : 0u) + (uses >= 3 ? 1u << 16 : 0u);
  }
#pragma unroll
  for (int q = 0; q < 3; ++q)
    if (hash_insert_new(vtab, mask, ((unsigned long long)l << 32) | (unsigned)v[q])) cnt += 1u << 24;
  double p[3][3];
  tri_corners(verts, v, p);
  const double ux = p[1][0] - p[0][0], uy = p[1][1] - p[0][1], uz = p[1][2] - p[0][2];
  const double wx = p[2][0] - p[0][0], wy = p[2][1] - p[0][1], wz = p[2][2] - p[0][2];
  const double cx = uy * wz - uz * wy, cy = uz * wx - ux * wz, cz = ux * wy - uy * wx;
  const unsigned peers = __match_any_sync(act, l);
  const bool leader = (__ffs(peers) - 1) == (int)lane_id();
  const double area = peer_reduce(peers, 0.5 * sqrt(cx * cx + cy * cy + cz * cz), MAdd());
  cnt = peer_reduce(peers, cnt, MAdd());
  ctr_mt3d_component* c = comp + l;
  unsigned long long* lo = reinterpret_cast<unsigned long long*>(c->lo);
  unsigned long long* hi = reinterpret_cast<unsigned long long*>(c->hi);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const unsigned long long kl = peer_reduce(peers, okey(fmin(p[0][a], fmin(p[1][a], p[2][a]))), MMin());
    const unsigned long long kh = peer_reduce(peers, okey(fmax(p[0][a], fmax(p[1][a], p[2][a]))), MMax());
    // the targets only move one way, so a stale read can only let a useless atomic through
    if (leader && *(volatile unsigned long long*)&lo[a] > kl) atomicMin(&lo[a], kl);
    if (leader && *(volatile unsigned long long*)&hi[a] < kh) atomicMax(&hi[a], kh);
  }
  if (!leader) return;
  atomicAdd(&c->area, area);
  atomicAdd((unsigned long long*)&c->n_tris, (unsigned long long)__popc(peers));
  if (cnt & 0xffu) atomicAdd((unsigned long long*)&c->n_edges, (unsigned long long)(cnt & 0xffu));
  if ((cnt >> 8) & 0xffu) atomicAdd((unsigned long long*)&c->n_boundary_edges, (unsigned long long)((cnt >> 8) & 0xffu));
  if ((cnt >> 16) & 0xffu) atomicAdd((unsigned long long*)&c->n_nonmanifold_edges, (unsigned long long)((cnt >> 16) & 0xffu));
  if (cnt >> 24) atomicAdd((unsigned long long*)&c->n_verts, (unsigned long long)(cnt >> 24));
}

__global__ void k_m_box(ctr_mt3d_component* comp, unsigned nc) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nc) return;
  ctr_mt3d_component* c = comp + q;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    c->lo[a] = okey_value(reinterpret_cast<const unsigned long long*>(c->lo)[a]);
    c->hi[a] = okey_value(reinterpret_cast<const unsigned long long*>(c->hi)[a]);
  }
}

template <typename G>
__global__ void __launch_bounds__(M_THREADS) k_m_volume(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                        const int* __restrict__ label, ctr_mt3d_component* comp) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = t < nt;
  const unsigned act = __ballot_sync(0xffffffffu, in);
  if (!in) return;
  const int l = label[t];
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
  double p[3][3];
  tri_corners(verts, v, p);
  const double* lo = comp[l].lo;
#pragma unroll
  for (int q = 0; q < 3; ++q)
#pragma unroll
    for (int a = 0; a < 3; ++a) p[q][a] -= lo[a];
  const double cx = p[1][1] * p[2][2] - p[1][2] * p[2][1];
  const double cy = p[1][2] * p[2][0] - p[1][0] * p[2][2];
  const double cz = p[1][0] * p[2][1] - p[1][1] * p[2][0];
  const unsigned peers = __match_any_sync(act, l);
  const double vol = peer_reduce(peers, (p[0][0] * cx + p[0][1] * cy + p[0][2] * cz) / 6.0, MAdd());
  if ((__ffs(peers) - 1) == (int)lane_id()) atomicAdd(&comp[l].volume, vol);
}

template <typename G>
int components_typed(ctr_ctx* ctx, int64_t* n_components) {
  const unsigned nt = (unsigned)ctx->last_counts[1], nv = (unsigned)ctx->last_counts[0];
  cudaStream_t st = ctx->stream;
  if (nt == 0) {
    ctx->comp_tris = 0;
    ctx->comp_count = 0;
    ctx->comp_gen = ctx->mesh_gen;
    return 0;
  }
  const size_t nslots = edge_slots(nt);               // also the (component, vertex) table: about nt / 2 pairs (3 nt at worst)
  const unsigned blocks = (nt + M_THREADS - 1) / M_THREADS;   // also the look-back tiles of k_m_roots
  int rc;
  DevBuf& b_etab = ctx->aux[AUX_SCRATCH0];
  DevBuf& b_vtab = ctx->aux[AUX_SCRATCH1];
  DevBuf& b_par = ctx->aux[AUX_SCRATCH2];
  DevBuf& b_scan = ctx->aux[AUX_SCRATCH3];
  DevBuf& b_label = ctx->aux[AUX_LABELS];
  DevBuf& b_comp = ctx->aux[AUX_COMPONENTS];
  if ((rc = ctr_ensure(ctx, b_etab, nslots * sizeof(EdgeSlot)))) return rc;
  if ((rc = ctr_ensure(ctx, b_vtab, nslots * sizeof(EdgeSlot)))) return rc;
  if ((rc = ctr_ensure(ctx, b_par, (size_t)nt * 8))) return rc;
  if ((rc = ctr_ensure(ctx, b_scan, 64 + (size_t)blocks * 8))) return rc;
  if ((rc = ctr_ensure(ctx, b_label, (size_t)nt * 4))) return rc;
  EdgeSlot* etab = (EdgeSlot*)b_etab.p;
  EdgeSlot* vtab = (EdgeSlot*)b_vtab.p;
  int* parent = (int*)b_par.p;
  int* rank = parent + nt;
  MCounters* ctr = (MCounters*)b_scan.p;
  unsigned long long* status = (unsigned long long*)((char*)b_scan.p + 64);
  const G* verts = (const G*)ctx->verts.p;
  const int* tris = (const int*)ctx->tris.p;
  int* label = (int*)b_label.p;
  CTR_CUDA(ctx, cudaMemsetAsync(b_scan.p, 0, 64 + (size_t)blocks * 8, st));
  k_m_init<<<ctx->sm_count * 8, 256, 0, st>>>(etab, vtab, nslots, parent, nt);
  k_m_edges<<<blocks, M_THREADS, 0, st>>>(tris, nt, nv, etab, nslots - 1, ctr);
  ctx->launches += 2;
  CTR_CUDA(ctx, cudaGetLastError());
  MCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.bad) return fail_shifted_ids(ctx);
  k_o_union<<<blocks, M_THREADS, 0, st>>>(tris, nt, etab, nslots - 1, parent);
  k_m_roots<<<blocks, M_THREADS, 0, st>>>(parent, nt, rank, status, ctr, (int)blocks);
  ctx->launches += 2;
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  const unsigned nc = (unsigned)h.total;
  if ((rc = ctr_ensure(ctx, b_comp, (size_t)nc * sizeof(ctr_mt3d_component)))) return rc;
  ctr_mt3d_component* comp = (ctr_mt3d_component*)b_comp.p;
  const unsigned cblocks = (nc + 255) / 256;
  k_m_table_init<<<cblocks, 256, 0, st>>>(comp, nc);
  k_m_tris<G><<<blocks, M_THREADS, 0, st>>>(verts, tris, nt, parent, rank, etab, vtab, nslots - 1, label, comp);
  k_m_box<<<cblocks, 256, 0, st>>>(comp, nc);
  k_m_volume<G><<<blocks, M_THREADS, 0, st>>>(verts, tris, nt, label, comp);
  ctx->launches += 4;
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->comp_tris = nt;
  ctx->comp_count = nc;
  ctx->comp_gen = ctx->mesh_gen;
  if (n_components) *n_components = nc;
  return 0;
}
