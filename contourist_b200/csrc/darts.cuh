// Chaining of a segment soup into polylines by pointer jumping over darts, shared by the 2D contours (poly2d.cu,
// ctr_mt2d_polylines) and the plane sections of the 3D mesh (section3d.cuh, ctr_mt3d_section).  Included inside the
// anonymous namespace of each translation unit, after common.cuh and uf_hash.cuh.
//
//   vertex  = what a segment end lies on: (level, edge key) in 2D, (plane, mesh edge) in 3D.  A vertex lies on at most
//             two segments, except at a junction (a sample exactly on a 2D level, a non-manifold 3D edge);
//   dart    = a segment with a direction: dart 2s+q leaves end q of segment s.  The successor of a dart arriving at a
//             vertex is the dart that leaves it along the vertex's OTHER segment, or -- at the end of an open contour --
//             the dart back along the same segment.  An open contour of m segments is then ONE cycle of 2m darts (there
//             and back), a closed contour of m segments TWO cycles of m darts (one per direction);
//   k_p_insert / k_p_succ : vertex -> open-addressing table of 16-byte slots holding the (up to two) darts that leave
//             the vertex; successor and priority of every dart;
//   k_p_min  : pointer jumping, log2(longest contour) rounds: every dart learns the FIRST dart of its cycle = the dart
//             that leaves the open contour's smaller end / the closed contour's smallest vertex;
//   k_p_cut / k_p_rank : every cycle cut in front of its first dart, list ranking by pointer jumping: position of every dart;
//   k_p_mark : of a closed contour's two directions the one that starts towards the smaller neighbour is kept, of an
//             open contour's there-and-back tour the first half;
//   k_ps_* / scan_u32 : exclusive scan of 32-bit counts with the running count of non-zero entries.
// The caller describes its vertices with a functor V:
//   id(keys, d)   : 64-bit identity of the vertex dart d leaves (the table key; never ~0);
//   prio(keys, d) : its order among the vertices of one contour (keys[d] names the same order: k_p_mark compares keys);
//   junction(d) : called once for every dart that finds its vertex already holding two others.
// keys[d] == keys[d ^ 1] marks a dead segment (from a vertex to itself): no darts, never kept.

constexpr unsigned NIL = 0xffffffffu;

struct PolyCounters {
  unsigned long long junction_levels;   // 2D: bit l, some key of level l has more than two segments; 3D: junction planes
  unsigned changed;
  unsigned live;
  unsigned n_poly;
  unsigned n_points;
  unsigned n_points_final;
  unsigned pad;
};

struct __align__(16) VSlot {
  unsigned long long key;
  int a, b;                             // the darts that leave this vertex (-1: none)
};

__device__ __forceinline__ VSlot* vslot(VSlot* tab, size_t mask, unsigned long long key, bool insert) {
  size_t s = (size_t)ufh::mix64(key) & mask;
  while (true) {
    unsigned long long k = tab[s].key;
    if (k == key) return tab + s;
    if (k == ufh::EMPTY) {
      if (!insert) return nullptr;
      k = atomicCAS(&tab[s].key, ufh::EMPTY, key);
      if (k == ufh::EMPTY || k == key) return tab + s;
    }
    s = (s + 1) & mask;
  }
}

__global__ void k_p_init(VSlot* tab, size_t nslots, PolyCounters* ctr) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  for (size_t q = t; q < nslots; q += n) reinterpret_cast<int4*>(tab)[q] = make_int4(-1, -1, -1, -1);
  if (t == 0) memset(ctr, 0, sizeof *ctr);
}

// dart d = 2s+q leaves end q of segment s: registered at the vertex of that end
template <typename V>
__global__ void k_p_insert(V vert, const unsigned long long* __restrict__ keys, unsigned nd, VSlot* tab, size_t mask,
                           PolyCounters* ctr) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  if (keys[d] == keys[d ^ 1u]) return;                           // a segment from a key to itself: no dart
  VSlot* s = vslot(tab, mask, vert.id(keys, d), true);
  if (atomicCAS(&s->a, -1, (int)d) == -1) return;
  if (atomicCAS(&s->b, -1, (int)d) == -1) return;
  vert.junction(d, ctr);                                         // a third segment at this vertex
}

// successor, priority: (0 for darts that leave an end of an open contour, else 1) << 63 | prio of the tail.
// Within one cycle the smallest priority is unique: ends are visited once, and a closed contour's cycle leaves every
// vertex once.
template <typename V>
__global__ void k_p_succ(V vert, const unsigned long long* __restrict__ keys, unsigned nd, const VSlot* __restrict__ tab,
                         size_t mask, unsigned* __restrict__ succ, unsigned long long* __restrict__ best_p,
                         unsigned* __restrict__ best_d, unsigned* __restrict__ jump) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  if (keys[d] == keys[d ^ 1u]) {                                 // dead dart: a cycle of its own, never kept
    succ[d] = d;
    jump[d] = d;
    best_p[d] = ~0ull;
    best_d[d] = d;
    return;
  }
  const VSlot* hs = vslot(const_cast<VSlot*>(tab), mask, vert.id(keys, d ^ 1u), false);               // vertex the dart arrives at
  const int rev = (int)(d ^ 1u);
  int other = hs->a == rev ? hs->b : hs->a;
  const unsigned sc = other >= 0 ? (unsigned)other : (unsigned)rev;                              // an end: turn round
  const VSlot* ts = vslot(const_cast<VSlot*>(tab), mask, vert.id(keys, d), false);
  const bool leaves_end = ts->b < 0;
  succ[d] = sc;
  jump[d] = sc;
  best_p[d] = (leaves_end ? 0ull : (1ull << 63)) | vert.prio(keys, d);
  best_d[d] = d;
}

// one round of pointer jumping: minimum over twice as many darts ahead
__global__ void k_p_min(unsigned nd, const unsigned long long* __restrict__ bp, const unsigned* __restrict__ bd,
                        const unsigned* __restrict__ jmp, unsigned long long* __restrict__ bp2, unsigned* __restrict__ bd2,
                        unsigned* __restrict__ jmp2, PolyCounters* ctr) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const unsigned j = jmp[d];
  unsigned long long p = bp[d];
  unsigned b = bd[d];
  const unsigned long long pj = bp[j];
  if (pj < p) {
    p = pj;
    b = bd[j];
    ctr->changed = 1u;
  }
  bp2[d] = p;
  bd2[d] = b;
  jmp2[d] = jmp[j];
}

__global__ void k_p_cut(unsigned nd, const unsigned* __restrict__ succ, const unsigned* __restrict__ start, unsigned* __restrict__ nxt,
                        unsigned* __restrict__ dist) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const bool last = succ[d] == start[d];
  nxt[d] = last ? NIL : succ[d];
  dist[d] = last ? 0u : 1u;
}

__global__ void k_p_rank(unsigned nd, const unsigned* __restrict__ nxt, const unsigned* __restrict__ dist, unsigned* __restrict__ nxt2,
                         unsigned* __restrict__ dist2, PolyCounters* ctr) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const unsigned n = nxt[d];
  if (n == NIL) {
    nxt2[d] = NIL;
    dist2[d] = dist[d];
    return;
  }
  dist2[d] = dist[d] + dist[n];
  const unsigned nn = nxt[n];
  nxt2[d] = nn;
  if (nn != NIL) ctr->live = 1u;
}

// per dart: is it the first dart of a kept contour, and how many points does that contour have.  A closed contour of
// two segments between the same two vertices (3D only) has one neighbour both ways: the direction whose first dart
// comes first is kept.
__global__ void k_p_mark(unsigned nd, const unsigned long long* __restrict__ keys, const unsigned* __restrict__ start,
                         const unsigned* __restrict__ dist, unsigned* __restrict__ npts) {
  const unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  unsigned n = 0;
  if (start[d] == d && keys[d] != keys[d ^ 1u]) {
    const unsigned len = dist[d] + 1u;
    const unsigned twin = start[d ^ 1u];
    const unsigned long long ka = keys[d ^ 1u], kb = keys[twin ^ 1u];
    if (twin == d) n = len / 2u + 1u;                                                 // open: m segments, m + 1 points
    else if (ka < kb || (ka == kb && d < twin)) n = len;                               // closed, this direction kept: m points
  }
  npts[d] = n;
}

// exclusive scan of 32-bit counts, three kernels (block sums, one block over them, add back)
constexpr int PS_THREADS = 256, PS_PER = 8, PS_TILE = PS_THREADS * PS_PER;
__global__ void __launch_bounds__(PS_THREADS) k_ps_local(const unsigned* __restrict__ in, unsigned n, unsigned* __restrict__ out,
                                                         unsigned* __restrict__ block_sum, unsigned* __restrict__ nonzero_out) {
  __shared__ unsigned s_warp[PS_THREADS / 32], s_nz[PS_THREADS / 32];
  const unsigned q0 = blockIdx.x * PS_TILE + threadIdx.x * PS_PER;
  unsigned v[PS_PER], sum = 0, nz = 0;
#pragma unroll
  for (int u = 0; u < PS_PER; ++u) {
    v[u] = q0 + u < n ? in[q0 + u] : 0u;
    sum += v[u];
    nz += v[u] ? 1u : 0u;
  }
  const unsigned inc = warp_incl_scan_u32(sum), incz = warp_incl_scan_u32(nz);
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  if (lane == 31) {
    s_warp[warp] = inc;
    s_nz[warp] = incz;
  }
  __syncthreads();
  unsigned woff = 0, wz = 0, tot = 0, totz = 0;
#pragma unroll
  for (int w = 0; w < PS_THREADS / 32; ++w) {
    if (w < (int)warp) {
      woff += s_warp[w];
      wz += s_nz[w];
    }
    tot += s_warp[w];
    totz += s_nz[w];
  }
  unsigned run = woff + inc - sum, runz = wz + incz - nz;
#pragma unroll
  for (int u = 0; u < PS_PER; ++u) {
    if (q0 + u < n) {
      out[q0 + u] = run;
      if (nonzero_out) nonzero_out[q0 + u] = runz;
    }
    run += v[u];
    runz += v[u] ? 1u : 0u;
  }
  if (threadIdx.x == 0) {
    block_sum[2 * blockIdx.x] = tot;
    block_sum[2 * blockIdx.x + 1] = totz;
  }
}
__global__ void __launch_bounds__(1024) k_ps_blocks(unsigned* __restrict__ block_sum, unsigned nblocks, unsigned* __restrict__ total) {
  __shared__ unsigned long long s_warp[32];
  __shared__ unsigned long long s_carry;
  if (threadIdx.x == 0) s_carry = 0ull;
  __syncthreads();
  for (unsigned base = 0; base < nblocks; base += 1024) {
    const unsigned q = base + threadIdx.x;
    const unsigned long long mine = q < nblocks ? ((unsigned long long)block_sum[2 * q + 1] << 32 | block_sum[2 * q]) : 0ull;
    const unsigned long long inc = warp_incl_scan_u64(mine);
    if (lane_id() == 31) s_warp[threadIdx.x >> 5] = inc;
    __syncthreads();
    unsigned long long woff = 0, tot = 0;
    for (int w = 0; w < 32; ++w) {
      if (w < (int)(threadIdx.x >> 5)) woff += s_warp[w];
      tot += s_warp[w];
    }
    const unsigned long long ex = s_carry + woff + inc - mine;
    if (q < nblocks) {
      block_sum[2 * q] = (unsigned)(ex & 0xffffffffull);
      block_sum[2 * q + 1] = (unsigned)(ex >> 32);
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    total[0] = (unsigned)(s_carry & 0xffffffffull);
    total[1] = (unsigned)(s_carry >> 32);
  }
}
__global__ void k_ps_add(unsigned* __restrict__ out, unsigned* __restrict__ nonzero_out, unsigned n, const unsigned* __restrict__ block_sum) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  out[q] += block_sum[2 * (q / PS_TILE)];
  if (nonzero_out) nonzero_out[q] += block_sum[2 * (q / PS_TILE) + 1];
}

int scan_u32(ctr_ctx* ctx, const unsigned* in, unsigned n, unsigned* out, unsigned* nonzero_out, unsigned* block_sum, unsigned* total) {
  cudaStream_t st = ctx->stream;
  const unsigned nb = (n + PS_TILE - 1) / PS_TILE;
  k_ps_local<<<nb, PS_THREADS, 0, st>>>(in, n, out, block_sum, nonzero_out);
  k_ps_blocks<<<1, 1024, 0, st>>>(block_sum, nb, total);
  k_ps_add<<<(n + 255) / 256, 256, 0, st>>>(out, nonzero_out, n, block_sum);
  ctx->launches += 3;
  return 0;
}
