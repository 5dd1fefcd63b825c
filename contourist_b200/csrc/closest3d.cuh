// Closest points on the 3D device mesh to query points (ctr_mt3d_closest): a linear BVH (Karras, HPG 2012) over the
// triangles, rebuilt on every call, and one nearest-triangle descent per point.
//
// Included into mesh3d.cu inside its anonymous namespace.  The definition is oracle/mt3d_closest.py:closest; the
// closest point of a triangle is one fixed-order fp64 formula (__dadd_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn: nothing
// contracts), and the winner is the smallest (d2, triangle index), so the device result equals it bit for bit.
//   k_cq_box    : thread per triangle: ids checked against [0, n_verts); the leaf box, padded by 2^-40 max|coordinate|
//                 of the triangle and rounded outward to fp32; the scene box of the box centres, reduced per block
//                 before one global atomic per bound;
//   k_cq_finite : thread per point (device points): a non-finite coordinate raises a flag.  Host wait: both flags and
//                 the scene box, so every error is reported before anything is written;
//   k_cq_morton : 63-bit Morton code (3 x 21 bits) of every box centre in the scene box, and the triangle index;
//   cub::DeviceRadixSort::SortPairs over 63 bits (stable: equal codes stay in triangle order);
//   k_cq_nodes  : the Karras internal nodes on the augmented key (code, then index: 64 + clz of the index xor for equal
//                 codes) and the parent links;
//   k_cq_refit  : bottom-up boxes, one arrival counter per node (the second arrival builds the node); the height;
//   k_cq_query  : thread per point: near child first (by the fp64 lower bound of the point-to-box distance, the left
//                 child on a tie), the stack in shared memory.
// Pruning is conservative.  Every computed closest point lies within a few fp64 rounding errors (< 2^-50 max|coordinate|)
// of its triangle (the definition's weights are all in [0, 1]), so it lies inside the padded leaf box, and a computed
// d2 <= best implies a computed lower bound <= best (1 + 10 2^-53).  A node is skipped only when its bound exceeds
// best (1 + 2^-40): no triangle whose computed d2 could tie or beat the best is ever skipped.
// The augmented key has 63 + 31 distinct prefix lengths and every level of a Karras tree lengthens the common prefix,
// so no leaf is deeper than 94 and the 96-entry stack cannot overflow.
// Node: one 64-byte line, both children's boxes (fp32) and links (>= 0: node; < 0: ~triangle).
// Scratch: AUX_SCRATCH0 (counters, leaf boxes, codes, the sort).  AUX_CLOSEST_TREE: nodes, parents, arrival counters.
// cq_build is the whole build; ctr_mt3d_raycast (raycast3d.cuh) builds the same tree through it.
// AUX_CLOSEST_RESULT: distance, triangle, point.  AUX_CLOSEST_POINTS: host points staged in their own type.

constexpr int CQ_THREADS = 128;                        // query block: 96 x 128 x 4 bytes of stack = 48 KiB
constexpr int CQ_STACK = 96;
constexpr int CQ_EMPTY = (int)0x80000000;              // root of a mesh with no triangles (~t is > INT_MIN for t < 2^31-1)

struct CqCounters {                                    // 64 bytes
  unsigned bad_ids, bad_points, n_found, height;
  unsigned lo[3], hi[3];                               // scene box of the box centres, order-preserving keys
  unsigned pad[6];
};
static_assert(sizeof(CqCounters) == 64, "CqCounters is one 64-byte head");

struct CqBox {
  float lo[3], hi[3];
};

struct __align__(16) CqNode {
  float4 a, b, c;                                      // left lo xyz, left hi xyz, right lo xyz, right hi xyz
  int4 d;                                              // left link, right link, height, unused
};
static_assert(sizeof(CqNode) == 64, "a node is one 64-byte line");

__device__ __forceinline__ unsigned cq_fkey(float f) {
  const unsigned u = __float_as_uint(f);
  return (u >> 31) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float cq_funkey(unsigned k) {
  const unsigned u = (k >> 31) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}

struct D3 {
  double x, y, z;
};
__device__ __forceinline__ D3 d3_sub(D3 a, D3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ double d3_dot(D3 a, D3 b) {
  return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ D3 d3_axpy(D3 u, double t, D3 w) {  // u + t * w per axis
  return {__dadd_rn(u.x, __dmul_rn(t, w.x)), __dadd_rn(u.y, __dmul_rn(t, w.y)), __dadd_rn(u.z, __dmul_rn(t, w.z))};
}
__device__ __forceinline__ double d3_dist2(D3 p, D3 q) {
  const D3 d = d3_sub(p, q);
  return d3_dot(d, d);
}

// closest point of segment (u, v): u + clamp(dot(p-u, w) / dot(w, w), 0, 1) * w with w = v-u; u where dot(w, w) == 0
__device__ __forceinline__ D3 cq_segment(D3 p, D3 u, D3 v) {
  const D3 w = d3_sub(v, u);
  const double ww = d3_dot(w, w);
  if (ww == 0.0) return u;
  return d3_axpy(u, fmin(fmax(__ddiv_rn(d3_dot(d3_sub(p, u), w), ww), 0.0), 1.0), w);
}

// the definition's closest point of triangle (a, b, c) to p: Ericson's region walk, or the segment rule
__device__ __forceinline__ D3 cq_triangle(D3 p, D3 a, D3 b, D3 c) {
  D3 q = a;
  bool seg = false;
  do {
    const D3 ab = d3_sub(b, a), ac = d3_sub(c, a), ap = d3_sub(p, a);
    const double d1 = d3_dot(ab, ap), d2 = d3_dot(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) break;
    const D3 bp = d3_sub(p, b);
    const double d3 = d3_dot(ab, bp), d4 = d3_dot(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) {
      q = b;
      break;
    }
    const double vc = __dsub_rn(__dmul_rn(d1, d4), __dmul_rn(d3, d2));
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
      const double den = __dsub_rn(d1, d3);
      if (den != 0.0) q = d3_axpy(a, __ddiv_rn(d1, den), ab);
      else seg = true;
      break;
    }
    const D3 cp = d3_sub(p, c);
    const double d5 = d3_dot(ab, cp), d6 = d3_dot(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) {
      q = c;
      break;
    }
    const double vb = __dsub_rn(__dmul_rn(d5, d2), __dmul_rn(d1, d6));
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
      const double den = __dsub_rn(d2, d6);
      if (den != 0.0) q = d3_axpy(a, __ddiv_rn(d2, den), ac);
      else seg = true;
      break;
    }
    const double va = __dsub_rn(__dmul_rn(d3, d6), __dmul_rn(d5, d4));
    const double e = __dsub_rn(d4, d3), f = __dsub_rn(d5, d6);
    if (va <= 0.0 && e >= 0.0 && f >= 0.0) {
      const double den = __dadd_rn(e, f);
      if (den != 0.0) q = d3_axpy(b, __ddiv_rn(e, den), d3_sub(c, b));
      else seg = true;
      break;
    }
    const double s = __dadd_rn(__dadd_rn(va, vb), vc);
    const double v = __ddiv_rn(vb, s), w = __ddiv_rn(vc, s);
    if (s > 0.0 && v >= 0.0 && w >= 0.0 && __dadd_rn(v, w) <= 1.0) q = d3_axpy(d3_axpy(a, v, ab), w, ac);
    else seg = true;
  } while (0);
  if (seg) {                                           // edges (a,b), (b,c), (c,a): the smallest d2, the first on a tie
    q = cq_segment(p, a, b);
    double bd = d3_dist2(p, q);
    D3 o = cq_segment(p, b, c);
    double od = d3_dist2(p, o);
    if (od < bd) {
      q = o;
      bd = od;
    }
    o = cq_segment(p, c, a);
    od = d3_dist2(p, o);
    if (od < bd) q = o;
  }
  return q;
}

template <typename G>
__device__ __forceinline__ D3 cq_vertex(const G* __restrict__ verts, int v) {
  const G* r = verts + (size_t)v * 3;
  return {(double)r[0], (double)r[1], (double)r[2]};
}

template <typename G>
__global__ void __launch_bounds__(256) k_cq_box(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                unsigned nv, CqBox* __restrict__ box, CqCounters* ctr) {
  __shared__ float s_red[8][6];
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  float cmin[3] = {INFINITY, INFINITY, INFINITY}, cmax[3] = {-INFINITY, -INFINITY, -INFINITY};
  if (t < nt) {
    const int i0 = tris[(size_t)t * 3], i1 = tris[(size_t)t * 3 + 1], i2 = tris[(size_t)t * 3 + 2];
    CqBox bx;
    if ((unsigned)i0 >= nv || (unsigned)i1 >= nv || (unsigned)i2 >= nv) {
      ctr->bad_ids = 1u;
#pragma unroll
      for (int k = 0; k < 3; ++k) bx.lo[k] = bx.hi[k] = 0.0f;
    } else {
      const D3 a = cq_vertex(verts, i0), b = cq_vertex(verts, i1), c = cq_vertex(verts, i2);
      const double lo[3] = {fmin(a.x, fmin(b.x, c.x)), fmin(a.y, fmin(b.y, c.y)), fmin(a.z, fmin(b.z, c.z))};
      const double hi[3] = {fmax(a.x, fmax(b.x, c.x)), fmax(a.y, fmax(b.y, c.y)), fmax(a.z, fmax(b.z, c.z))};
      double m = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) m = fmax(m, fmax(fabs(lo[k]), fabs(hi[k])));
      const double pad = __dmul_rn(m, 0x1p-40);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        bx.lo[k] = __double2float_rd(__dsub_rn(lo[k], pad));
        bx.hi[k] = __double2float_ru(__dadd_rn(hi[k], pad));
        const float cen = __fmul_rn(0.5f, __fadd_rn(bx.lo[k], bx.hi[k]));
        cmin[k] = cmax[k] = cen;
      }
    }
    box[t] = bx;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      cmin[k] = fminf(cmin[k], __shfl_xor_sync(0xffffffffu, cmin[k], o));
      cmax[k] = fmaxf(cmax[k], __shfl_xor_sync(0xffffffffu, cmax[k], o));
    }
  const unsigned w = threadIdx.x >> 5;
  if (lane_id() == 0)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      s_red[w][k] = cmin[k];
      s_red[w][3 + k] = cmax[k];
    }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int k = threadIdx.x;
    float mn = INFINITY, mx = -INFINITY;
    for (unsigned q = 0; q < blockDim.x / 32; ++q) {
      mn = fminf(mn, s_red[q][k]);
      mx = fmaxf(mx, s_red[q][3 + k]);
    }
    if (mn <= mx) {
      atomicMin(&ctr->lo[k], cq_fkey(mn));
      atomicMax(&ctr->hi[k], cq_fkey(mx));
    }
  }
}

template <typename P>
__global__ void __launch_bounds__(256) k_cq_finite(const P* __restrict__ pts, size_t n, CqCounters* ctr) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(isfinite(pts[i]))) ctr->bad_points = 1u;
}

__device__ __forceinline__ unsigned long long cq_spread(unsigned v) {   // 21 bits to every third bit
  unsigned long long x = v & 0x1fffffu;
  x = (x | x << 32) & 0x1f00000000ffffull;
  x = (x | x << 16) & 0x1f0000ff0000ffull;
  x = (x | x << 8) & 0x100f00f00f00f00full;
  x = (x | x << 4) & 0x10c30c30c30c30c3ull;
  x = (x | x << 2) & 0x1249249249249249ull;
  return x;
}

__global__ void __launch_bounds__(256) k_cq_morton(const CqBox* __restrict__ box, unsigned nt, double3 lo, double3 scale,
                                                   unsigned long long* __restrict__ code, unsigned* __restrict__ idx) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const CqBox b = box[t];
  const double l[3] = {lo.x, lo.y, lo.z}, s[3] = {scale.x, scale.y, scale.z};
  unsigned long long c = 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double cen = (double)__fmul_rn(0.5f, __fadd_rn(b.lo[k], b.hi[k]));
    const double u = fmin(fmax((cen - l[k]) * s[k], 0.0), 2097151.0);
    c |= cq_spread((unsigned)u) << (2 - k);
  }
  code[t] = c;
  idx[t] = t;
}

// the length of the common prefix of the augmented keys (code, index) of sorted leaves i and j; -1 outside [0, n)
__device__ __forceinline__ int cq_delta(const unsigned long long* __restrict__ code, int n, int i, long long j) {
  if (j < 0 || j >= n) return -1;
  const unsigned long long ci = code[i], cj = code[j];
  return ci != cj ? __clzll(ci ^ cj) : 64 + __clz(i ^ (int)j);
}

__global__ void __launch_bounds__(256) k_cq_nodes(const unsigned long long* __restrict__ code, const unsigned* __restrict__ tri,
                                                  int n, CqNode* __restrict__ node, int* __restrict__ node_parent,
                                                  int* __restrict__ leaf_parent) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  const int d = cq_delta(code, n, i, i + 1) - cq_delta(code, n, i, i - 1) >= 0 ? 1 : -1;
  const int dmin = cq_delta(code, n, i, i - d);
  long long lmax = 2;
  while (cq_delta(code, n, i, i + lmax * d) > dmin && lmax < (1ll << 32)) lmax <<= 1;
  long long l = 0;
  for (long long s = lmax >> 1; s >= 1; s >>= 1)
    if (cq_delta(code, n, i, i + (l + s) * d) > dmin) l += s;
  const int j = (int)(i + l * d);
  const int dnode = cq_delta(code, n, i, j);
  long long s = 0;
  for (long long div = 2, step;; div <<= 1) {
    step = (l + div - 1) / div;
    if (cq_delta(code, n, i, i + (s + step) * d) > dnode) s += step;
    if (step <= 1) break;
  }
  const int gamma = (int)(i + s * d) + min(d, 0);
  const int lo = min(i, j), hi = max(i, j);
  int left, right;
  if (lo == gamma) {
    left = ~(int)tri[gamma];
    leaf_parent[gamma] = i;
  } else {
    left = gamma;
    node_parent[gamma] = i;
  }
  if (hi == gamma + 1) {
    right = ~(int)tri[gamma + 1];
    leaf_parent[gamma + 1] = i;
  } else {
    right = gamma + 1;
    node_parent[gamma + 1] = i;
  }
  node[i].d = make_int4(left, right, 0, 0);
  if (i == 0) node_parent[0] = -1;
}

// the box (lo, hi) and height of child link `c`, read through L2 (another thread wrote a node child)
__device__ __forceinline__ int cq_child(const CqNode* node, const CqBox* __restrict__ box, int c, float lo[3], float hi[3]) {
  if (c < 0) {
    const CqBox b = box[~c];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = b.lo[k];
      hi[k] = b.hi[k];
    }
    return 0;
  }
  const float4 a = __ldcg(&node[c].a), b = __ldcg(&node[c].b), e = __ldcg(&node[c].c);
  const int h = __ldcg(&node[c].d.z);
  lo[0] = fminf(a.x, b.z);
  lo[1] = fminf(a.y, b.w);
  lo[2] = fminf(a.z, e.x);
  hi[0] = fmaxf(a.w, e.y);
  hi[1] = fmaxf(b.x, e.z);
  hi[2] = fmaxf(b.y, e.w);
  return h;
}

__global__ void __launch_bounds__(256) k_cq_refit(int n, const CqBox* __restrict__ box, CqNode* node,
                                                  const int* __restrict__ node_parent, const int* __restrict__ leaf_parent,
                                                  unsigned* arrive, CqCounters* ctr) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  int p = leaf_parent[k];
  while (p >= 0) {
    __threadfence();
    if (atomicAdd(&arrive[p], 1u) == 0u) return;       // the first arrival leaves; the second builds the node
    __threadfence();
    const int4 d = node[p].d;
    float l[3], h[3], r[3], s[3];
    const int hl = cq_child(node, box, d.x, l, h), hr = cq_child(node, box, d.y, r, s);
    const int ht = 1 + max(hl, hr);
    node[p].a = make_float4(l[0], l[1], l[2], h[0]);
    node[p].b = make_float4(h[1], h[2], r[0], r[1]);
    node[p].c = make_float4(r[2], s[0], s[1], s[2]);
    node[p].d.z = ht;
    if (p == 0) ctr->height = (unsigned)ht;
    p = node_parent[p];
  }
}

// the fp64 lower bound of the squared distance from p to box (lo, hi)
__device__ __forceinline__ double cq_box_d2(D3 p, float lx, float ly, float lz, float hx, float hy, float hz) {
  const double dx = fmax(fmax(__dsub_rn((double)lx, p.x), __dsub_rn(p.x, (double)hx)), 0.0);
  const double dy = fmax(fmax(__dsub_rn((double)ly, p.y), __dsub_rn(p.y, (double)hy)), 0.0);
  const double dz = fmax(fmax(__dsub_rn((double)lz, p.z), __dsub_rn(p.z, (double)hz)), 0.0);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

template <typename G, typename P>
__global__ void __launch_bounds__(CQ_THREADS) k_cq_query(const P* __restrict__ pts, unsigned np, const CqNode* __restrict__ node,
                                                         int root, const G* __restrict__ verts, const int* __restrict__ tris,
                                                         double best0, double* __restrict__ dist, int* __restrict__ tri_out,
                                                         double* __restrict__ pt_out, CqCounters* ctr) {
  __shared__ int s_stack[CQ_STACK * CQ_THREADS];       // entry e of thread x at e * CQ_THREADS + x: no bank conflicts
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  bool found = false;
  if (i < np) {
    const D3 p = {(double)pts[(size_t)i * 3], (double)pts[(size_t)i * 3 + 1], (double)pts[(size_t)i * 3 + 2]};
    double best = best0, lim = __dmul_rn(best0, 1.0 + 0x1p-40);
    int bt = 0x7fffffff;
    D3 bq = {0.0, 0.0, 0.0};
    int* stk = s_stack + threadIdx.x;
    int sp = 0, cur = root;
    while (cur != CQ_EMPTY) {
      if (cur >= 0) {
        const float4* nd = reinterpret_cast<const float4*>(node + cur);
        const float4 a = __ldg(nd), b = __ldg(nd + 1), c = __ldg(nd + 2);
        const int4 d = __ldg(reinterpret_cast<const int4*>(nd + 3));
        const double dl = cq_box_d2(p, a.x, a.y, a.z, a.w, b.x, b.y), dr = cq_box_d2(p, b.z, b.w, c.x, c.y, c.z, c.w);
        const bool vl = !(dl > lim), vr = !(dr > lim);
        if (vl && vr) {
          const bool rfirst = dr < dl;
          stk[sp * CQ_THREADS] = rfirst ? d.x : d.y;
          ++sp;
          cur = rfirst ? d.y : d.x;
          continue;
        }
        if (vl || vr) {
          cur = vl ? d.x : d.y;
          continue;
        }
      } else {
        const int t = ~cur;
        const int* tv = tris + (size_t)t * 3;
        const D3 q = cq_triangle(p, cq_vertex(verts, __ldg(tv)), cq_vertex(verts, __ldg(tv + 1)), cq_vertex(verts, __ldg(tv + 2)));
        const double d2 = d3_dist2(p, q);
        if (d2 < best || (d2 == best && t < bt)) {
          best = d2;
          bt = t;
          bq = q;
          lim = __dmul_rn(best, 1.0 + 0x1p-40);
        }
      }
      if (sp == 0) break;
      --sp;
      cur = stk[sp * CQ_THREADS];
    }
    found = bt != 0x7fffffff;
    dist[i] = found ? __dsqrt_rn(best) : INFINITY;
    tri_out[i] = found ? bt : -1;
    pt_out[(size_t)i * 3] = found ? bq.x : NAN;
    pt_out[(size_t)i * 3 + 1] = found ? bq.y : NAN;
    pt_out[(size_t)i * 3 + 2] = found ? bq.z : NAN;
  }
  const unsigned f = __ballot_sync(0xffffffffu, found);
  if (lane_id() == 0 && f) atomicAdd(&ctr->n_found, (unsigned)__popc(f));
}

// launches of cub::DeviceRadixSort::SortPairs on n (u64 code, u32 index) pairs over 63 bits: one single-tile kernel,
// or a histogram, an exclusive sum and one onesweep kernel per 8-bit digit and portion of the input
static inline int64_t cq_sort_launches(size_t n) {
  using Single = cub::detail::radix::policy_hub<unsigned long long, unsigned, uint32_t>::Policy1000::SingleTilePolicy;
  if (n <= (size_t)Single::BLOCK_THREADS * Single::ITEMS_PER_THREAD) return 1;
  const size_t portion = (size_t)1 << 28;
  return 2 + 8 * (int64_t)((n + portion - 1) / portion);
}

// The tree over the mesh as it stands, shared by ctr_mt3d_closest and ctr_mt3d_raycast: k_cq_box, the queries' own
// check kernels (`check` enqueues them on the counters and returns their launch count), the one host wait (the id flag,
// the query flag, the scene box: an error here is `bad_msg`, and nothing has been written), then k_cq_morton, the sort,
// k_cq_nodes and k_cq_refit.  Fills the root link, the nodes, the device counters and their host copy.
struct CqTree {
  int root;
  CqNode* node;
  CqCounters* ctr;
  CqCounters h;
};

template <typename G, typename Check>
int cq_build(ctr_ctx* ctx, Check&& check, const char* bad_msg, CqTree* tr) {
  cudaStream_t st = ctx->stream;
  const size_t nT = (size_t)ctx->last_counts[1], nV = (size_t)ctx->last_counts[0];
  const int* tris = (const int*)ctx->tris.p;
  const G* verts = (const G*)ctx->verts.p;
  // ---- scratch: counters, leaf boxes, codes and indices (both sort buffers), the sort's temporary storage
  size_t sort_bytes = 0;
  if (nT > 1)
    CTR_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long*)nullptr,
                                                  (unsigned long long*)nullptr, (const unsigned*)nullptr, (unsigned*)nullptr,
                                                  (int)nT, 0, 63, st));
  CqCounters* ctr;
  CqBox* box;
  unsigned long long *code, *code_s;
  unsigned *idx, *idx_s;
  void* sort_tmp;
  int rc;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH0], [&](ctr_carve& c) {
         c(ctr, sizeof(CqCounters));
         c(box, nT * sizeof(CqBox));
         c(code, nT * 8);
         c(code_s, nT * 8);
         c(idx, nT * 4);
         c(idx_s, nT * 4);
         c(sort_tmp, sort_bytes);
       })))
    return rc;
  CTR_CUDA(ctx, cudaMemsetAsync(ctr, 0, sizeof(CqCounters), st));
  CTR_CUDA(ctx, cudaMemsetAsync(ctr->lo, 0xff, sizeof ctr->lo, st));
  const unsigned tb = (unsigned)((nT + 255) / 256);
  if (nT) {
    k_cq_box<G><<<tb, 256, 0, st>>>(verts, tris, (unsigned)nT, (unsigned)nV, box, ctr);
    ctx->launches++;
  }
  ctx->launches += check(ctr);
  CTR_CUDA(ctx, cudaGetLastError());
  CqCounters& h = tr->h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.bad_ids) return fail_shifted_ids(ctx);
  if (h.bad_points) return ctr_fail(ctx, CTR_ERR_BAD_ARG, bad_msg);
  // ---- the tree
  CqNode* node = nullptr;
  int *node_parent, *leaf_parent;
  unsigned* arrive;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_CLOSEST_TREE], [&](ctr_carve& c) {
         c(node, (nT > 1 ? nT - 1 : 0) * sizeof(CqNode));
         c(node_parent, nT * 4);
         c(leaf_parent, nT * 4);
         c(arrive, nT * 4);
       })))
    return rc;
  if (nT > 1) {
    double3 lo, scale;
    double l[3], s[3];
    for (int k = 0; k < 3; ++k) {
      l[k] = (double)cq_funkey(h.lo[k]);
      const double ext = (double)cq_funkey(h.hi[k]) - l[k];
      s[k] = ext > 0.0 && isfinite(ext) ? 2097151.0 / ext : 0.0;
    }
    lo = make_double3(l[0], l[1], l[2]);
    scale = make_double3(s[0], s[1], s[2]);
    k_cq_morton<<<tb, 256, 0, st>>>(box, (unsigned)nT, lo, scale, code, idx);
    CTR_CUDA(ctx, cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, code, code_s, idx, idx_s, (int)nT, 0, 63, st));
    const unsigned nb = (unsigned)((nT - 1 + 255) / 256);
    k_cq_nodes<<<nb, 256, 0, st>>>(code_s, idx_s, (int)nT, node, node_parent, leaf_parent);
    CTR_CUDA(ctx, cudaMemsetAsync(arrive, 0, (nT - 1) * 4, st));
    k_cq_refit<<<tb, 256, 0, st>>>((int)nT, box, node, node_parent, leaf_parent, arrive, ctr);
    ctx->launches += 3 + cq_sort_launches(nT);
  }
  tr->root = nT == 0 ? CQ_EMPTY : nT == 1 ? ~0 : 0;
  tr->node = node;
  tr->ctr = ctr;
  return 0;
}

template <typename G, typename P>
int closest_run(ctr_ctx* ctx, const ctr_closest_params* cp, const P* pts, ctr_closest_counts* out) {
  cudaStream_t st = ctx->stream;
  const size_t nT = (size_t)ctx->last_counts[1], nP = (size_t)cp->n_points;
  const int* tris = (const int*)ctx->tris.p;
  const G* verts = (const G*)ctx->verts.p;
  const bool on_device = cp->flags & CTR_FIELD_ON_DEVICE;
  CqTree tr;
  int rc;
  if ((rc = cq_build<G>(ctx, [&](CqCounters* ctr) -> int64_t {
         if (!on_device || !nP) return 0;
         k_cq_finite<P><<<(unsigned)((nP * 3 + 255) / 256), 256, 0, st>>>(pts, nP * 3, ctr);
         return 1;
       }, "query points must be finite", &tr)))
    return rc;
  // ---- the queries
  double* dist;
  int* tri_out;
  double* pt_out;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_CLOSEST_RESULT], [&](ctr_carve& c) {
         c(dist, nP * 8);
         c(tri_out, nP * 4);
         c(pt_out, nP * 24);
       })))
    return rc;
  if (nP) {
    const double md = cp->max_distance;
    k_cq_query<G, P><<<(unsigned)((nP + CQ_THREADS - 1) / CQ_THREADS), CQ_THREADS, 0, st>>>(
        pts, (unsigned)nP, tr.node, tr.root, verts, tris, md * md, dist, tri_out, pt_out, tr.ctr);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CqCounters& h = tr.h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, tr.ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->closest_n = (int64_t)nP;
  out->n_found = h.n_found;
  out->height = nT > 1 ? (int64_t)h.height : 0;
  return 0;
}

template <typename G>
int closest_typed(ctr_ctx* ctx, const ctr_closest_params* cp, ctr_closest_counts* out) {
  const size_t nP = (size_t)cp->n_points, psz = cp->dtype == CTR_F64 ? 8 : 4;
  const void* pts = cp->points;
  if (!(cp->flags & CTR_FIELD_ON_DEVICE) && nP) {     // host points: staged in their own type
    if (int rc = ctr_ensure(ctx, ctx->aux[AUX_CLOSEST_POINTS], nP * 3 * psz)) return rc;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->aux[AUX_CLOSEST_POINTS].p, pts, nP * 3 * psz, cudaMemcpyHostToDevice, ctx->stream));
    pts = ctx->aux[AUX_CLOSEST_POINTS].p;
  }
  if (cp->dtype == CTR_F64) return closest_run<G, double>(ctx, cp, (const double*)pts, out);
  return closest_run<G, float>(ctx, cp, (const float*)pts, out);
}
