// Caps that close the 3D device mesh at the faces of the volume (ctr_mt3d_cap; included by mesh3d.cu inside its anonymous
// namespace, after decimate3d.cuh, whose k_d_ids it runs).  The definition is oracle/mt3d_cap.py:cap (exact; new
// normals within rounding of the normalisation).
//
// With the Kuhn decomposition each box face square (minimum corner m, in-face axes a < b) is cut along its min -> max
// diagonal into T0 = (m, m + e_a, m + e_a + e_b) and T1 = (m, m + e_b, m + e_a + e_b), so the surface's rim on the face is
// the contour of the face samples on those triangles and the cap is the part of each face triangle on the chosen side.
//   k_d_ids      : every triangle id in [0, n_verts) (read back at the one host wait, before anything is written);
//   k_cap_index  : thread per vertex; a vertex whose key names an in-face edge of a box face goes into the key -> id table;
//   k_cap_count  : thread per face square of the six faces (face-major, then row-major over (a, b)): the pieces of its two
//                  face triangles, their crossing vertices looked up (a missing one drops the face triangle, n_missing),
//                  one flag byte per piece slot (4 per square) and one flag per box-surface point a piece uses;
//   k_flag_scan x 2 : output index of every piece and of every used point; one host wait for the totals;
//   k_cap_verts  : thread per box-surface point (canonical index = rank in lin order): position, normal, key, lowmin;
//   k_cap_tris   : thread per face square with pieces: the triangles, ids looked up again.
// Scratch: AUX_SCRATCH2 only.  The output buffers grow with ctr_grow_keep, so device pointers handed out before may change.

struct CapCounters {                                   // head of the scan piece
  DecCounters ids;                                     // k_d_ids: bad_ids
  unsigned n_missing;
  unsigned ticket[2];                                  // tile tickets of the piece and point scans
  unsigned long long total[2];                         // pieces, used points
};
static_assert(sizeof(CapCounters) <= 64, "CapCounters fits the 64-byte head of the scan piece");

struct CapGrid {
  long long n[3];
  long long sq_base[7];                                // first face-square index of each face; sq_base[6]: all squares
  long long plane, ring;                               // points of a box plane (n1 n2) and of an interior plane's rim
  double value;
  int side;                                            // CTR_CAP_HIGH / CTR_CAP_LOW
  double origin[3], delta[3];
  int wsign[6];                                        // per face: sign of its cap triangles' world normal along e_axis
};

__device__ __forceinline__ void face_axes(int axis, int& a, int& b) {
  a = axis == 0 ? 1 : 0;
  b = axis == 2 ? 1 : 2;
}

__device__ __forceinline__ long long cap_lin(const CapGrid& g, const long long p[3]) {
  return (p[0] * g.n[1] + p[1]) * g.n[2] + p[2];
}

// rank of box-surface point p among the box-surface points in lin order: the full planes i = 0 and i = n0 - 1, and in
// between, per plane, the full rows j = 0 and j = n1 - 1 and two points (k = 0, k = n2 - 1) of every other row
__device__ __forceinline__ long long surf_index(const CapGrid& g, const long long p[3]) {
  if (p[0] == 0) return p[1] * g.n[2] + p[2];
  long long r = g.plane + (p[0] - 1) * g.ring;
  if (p[0] == g.n[0] - 1) return r + p[1] * g.n[2] + p[2];
  if (p[1] == 0) return r + p[2];
  if (p[1] == g.n[1] - 1) return r + g.n[2] + (g.n[1] - 2) * 2 + p[2];
  return r + g.n[2] + (p[1] - 1) * 2 + (p[2] == 0 ? 0 : 1);
}

__device__ __forceinline__ void surf_point(const CapGrid& g, long long s, long long p[3]) {
  if (s < g.plane) {
    p[0] = 0; p[1] = s / g.n[2]; p[2] = s % g.n[2];
    return;
  }
  s -= g.plane;
  if (s >= (g.n[0] - 2) * g.ring) {
    s -= (g.n[0] - 2) * g.ring;
    p[0] = g.n[0] - 1; p[1] = s / g.n[2]; p[2] = s % g.n[2];
    return;
  }
  p[0] = 1 + s / g.ring;
  s %= g.ring;
  if (s < g.n[2]) {
    p[1] = 0; p[2] = s;
  } else if ((s -= g.n[2]) < (g.n[1] - 2) * 2) {
    p[1] = 1 + s / 2; p[2] = (s & 1) ? g.n[2] - 1 : 0;
  } else {
    s -= (g.n[1] - 2) * 2;
    p[1] = g.n[1] - 1; p[2] = s;
  }
}

// a face square by global index q: its face and its minimum corner
__device__ __forceinline__ int face_square(const CapGrid& g, long long q, long long m[3], int& a, int& b) {
  int f = 0;
#pragma unroll
  for (int i = 1; i < 6; ++i) f += q >= g.sq_base[i];
  const int axis = f >> 1;
  face_axes(axis, a, b);
  const long long r = q - g.sq_base[f], nb = (b == 1 ? g.n[1] : g.n[2]) - 1;
  const long long fixed = (f & 1) ? (axis == 0 ? g.n[0] : axis == 1 ? g.n[1] : g.n[2]) - 1 : 0;
#pragma unroll
  for (int x = 0; x < 3; ++x) m[x] = x == axis ? fixed : x == a ? r / nb : r % nb;   // (selects: x is a constant)
  return f;
}

// The corners of face triangle t of the square at m and their on-side flags (bit i: corner i).  The piece on the side
// (oracle/mt3d_cap.py:polygon) walks i = 0, 1, 2: corner i if it is on the side, then the crossing of edge (i, i+1 mod 3)
// if exactly one of its ends is; the walk is unrolled wherever it is used, so nothing is indexed at run time.
template <typename T>
__device__ __forceinline__ unsigned cap_corners(const CapGrid& g, const T* __restrict__ f, const long long m[3], int a, int b,
                                                int t, long long c[3][3]) {
  const int e = t == 0 ? a : b;
#pragma unroll
  for (int x = 0; x < 3; ++x) {
    c[0][x] = m[x];
    c[1][x] = m[x] + (x == e);
    c[2][x] = m[x] + (x == a || x == b);
  }
  unsigned s = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) s |= (unsigned)(((double)f[cap_lin(g, c[i])] < g.value) == (g.side == CTR_CAP_LOW)) << i;
  return s;
}

// mesh vertex of the crossing on edge (c[i], c[i+1 mod 3]), or -1
template <int i>
__device__ __forceinline__ int cap_crossing(const CapGrid& g, const long long c[3][3], ufh::Slot* tab, size_t mask) {
  constexpr int j = (i + 1) % 3;
  long long lo[3];
  unsigned d = 0;
#pragma unroll
  for (int x = 0; x < 3; ++x) {
    lo[x] = min(c[i][x], c[j][x]);
    d |= (unsigned)(c[i][x] != c[j][x]) << (2 - x);
  }
  const unsigned long long key = ((unsigned long long)cap_lin(g, lo) << 3) | d;
  const ufh::Slot* s = ufh::hash_slot(tab, mask, key, false);
  return s->key == key ? s->tri : -1;
}

__device__ __forceinline__ bool edge_changes(unsigned s, int i) { return ((s >> i) ^ (s >> ((i + 1) % 3))) & 1u; }

// cross(c1 - c0, c2 - c0) of face triangle t is +sigma e_axis for T0, -sigma e_axis for T1 (e_a x e_b = sigma e_axis);
// the cap faces into the box for CTR_CAP_HIGH, out of it for CTR_CAP_LOW: reverse the pieces where the two differ
__device__ __forceinline__ bool cap_flip(const CapGrid& g, int f, int t) {
  const int axis = f >> 1;
  const int natural = (axis == 1 ? -1 : 1) * (t == 0 ? 1 : -1);
  const int out = (f & 1) ? 1 : -1;
  return natural != (g.side == CTR_CAP_HIGH ? -out : out);
}

__global__ void __launch_bounds__(256) k_cap_index(const unsigned long long* __restrict__ keys, unsigned nv, CapGrid g,
                                                   ufh::Slot* tab, size_t mask) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const unsigned long long key = keys[v];
  const unsigned d = (unsigned)key & 7u;
  const long long lin = (long long)(key >> 3);
  const long long p[3] = {lin / (g.n[1] * g.n[2]), (lin / g.n[2]) % g.n[1], lin % g.n[2]};
  bool in_face = false;
#pragma unroll
  for (int x = 0; x < 3; ++x)                            // both ends on face x = 0 or x = n - 1
    in_face |= ((d >> (2 - x)) & 1u) == 0u && (p[x] == 0 || p[x] == g.n[x] - 1);
  if (in_face && d != 0u) ufh::hash_slot(tab, mask, key, true)->tri = (int)v;
}

template <typename T>
__global__ void __launch_bounds__(256) k_cap_count(const T* __restrict__ f, CapGrid g, ufh::Slot* tab, size_t mask,
                                                   uint32_t* __restrict__ piece_flags, uint8_t* __restrict__ point_flags,
                                                   CapCounters* ctr) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.sq_base[6]) return;
  long long m[3], c[3][3];
  int a, b;
  face_square(g, q, m, a, b);
  uint32_t word = 0;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const unsigned sd = cap_corners(g, f, m, a, b, t, c);
    if (!sd) continue;
    bool ok = true;
    if (edge_changes(sd, 0)) ok = ok && cap_crossing<0>(g, c, tab, mask) >= 0;
    if (edge_changes(sd, 1)) ok = ok && cap_crossing<1>(g, c, tab, mask) >= 0;
    if (edge_changes(sd, 2)) ok = ok && cap_crossing<2>(g, c, tab, mask) >= 0;
    if (!ok) {
      atomicAdd(&ctr->n_missing, 1u);
      continue;
    }
    const int n = __popc(sd) + (sd == 7u ? 0 : 2);     // polygon vertices; n - 2 pieces
    word |= 1u << (16 * t);
    if (n == 4) word |= 1u << (16 * t + 8);
#pragma unroll
    for (int i = 0; i < 3; ++i)
      if ((sd >> i) & 1u) point_flags[surf_index(g, c[i])] = 1;
  }
  piece_flags[q] = word;
}

template <typename T, typename G>
__global__ void __launch_bounds__(256) k_cap_verts(const T* __restrict__ f, CapGrid g, unsigned long long n_points,
                                                   const uint8_t* __restrict__ point_flags, const uint32_t* __restrict__ point_idx,
                                                   size_t nv, G* __restrict__ verts, G* __restrict__ normals,
                                                   unsigned long long* __restrict__ keys, uint8_t* __restrict__ lowmin) {
  const unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_points || !point_flags[s]) return;
  const size_t id = nv + point_idx[s];
  long long p[3];
  surf_point(g, (long long)s, p);
  const long long lin = cap_lin(g, p);
#pragma unroll
  for (int x = 0; x < 3; ++x) verts[id * 3 + x] = add_rn(mul_rn((G)p[x], (G)g.delta[x]), (G)g.origin[x]);
  keys[id] = (unsigned long long)lin << 3;
  lowmin[id] = (double)f[lin] < g.value ? 1 : 0;
  if (normals) {
    G nn[3], len2 = (G)0;
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      nn[x] = (G)0;
      if (p[x] == 0) nn[x] = (G)g.wsign[2 * x];
      if (p[x] == g.n[x] - 1) nn[x] = (G)g.wsign[2 * x + 1];
      len2 = add_rn(len2, mul_rn(nn[x], nn[x]));
    }
    const G len = sqrt(len2);
#pragma unroll
    for (int x = 0; x < 3; ++x) normals[id * 3 + x] = nn[x] / len;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_cap_tris(const T* __restrict__ f, CapGrid g, ufh::Slot* tab, size_t mask,
                                                  const uint32_t* __restrict__ piece_flags, const uint32_t* __restrict__ piece_idx,
                                                  const uint32_t* __restrict__ point_idx, unsigned nv, unsigned nt,
                                                  int* __restrict__ tris) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.sq_base[6]) return;
  const uint32_t word = piece_flags[q];
  if (!word) return;
  long long m[3], c[3][3];
  int a, b;
  const int fc = face_square(g, q, m, a, b);
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    if (!((word >> (16 * t)) & 0xffffu)) continue;
    const unsigned sd = cap_corners(g, f, m, a, b, t, c);
    int v[4] = {0, 0, 0, 0}, n = 0;                    // the polygon's vertex ids, in walk order
    auto push = [&](int id) {
      v[3] = n == 3 ? id : v[3];
      v[2] = n == 2 ? id : v[2];
      v[1] = n == 1 ? id : v[1];
      v[0] = n == 0 ? id : v[0];
      ++n;
    };
    if (sd & 1u) push((int)(nv + point_idx[surf_index(g, c[0])]));
    if (edge_changes(sd, 0)) push(cap_crossing<0>(g, c, tab, mask));
    if (sd & 2u) push((int)(nv + point_idx[surf_index(g, c[1])]));
    if (edge_changes(sd, 1)) push(cap_crossing<1>(g, c, tab, mask));
    if (sd & 4u) push((int)(nv + point_idx[surf_index(g, c[2])]));
    if (edge_changes(sd, 2)) push(cap_crossing<2>(g, c, tab, mask));
    const bool flip = cap_flip(g, fc, t);
    // the fan from v[0]: (v0, v1, v2), and (v0, v2, v3) for a quad; reversed where the face triangle points the wrong way
    int* o = tris + ((size_t)nt + piece_idx[q * 4 + t * 2]) * 3;
    o[0] = v[0];
    o[1] = flip ? v[2] : v[1];
    o[2] = flip ? v[1] : v[2];
    if (n == 4) {
      o = tris + ((size_t)nt + piece_idx[q * 4 + t * 2 + 1]) * 3;
      o[0] = v[0];
      o[1] = flip ? v[3] : v[2];
      o[2] = flip ? v[2] : v[3];
    }
  }
}

template <typename T, typename G>
int cap_typed(ctr_ctx* ctx, const ctr_cap_params* cp, ctr_cap_counts* out) {
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  cudaStream_t st = ctx->stream;
  const size_t nV = (size_t)ctx->last_counts[0], nT = (size_t)ctx->last_counts[1];
  CapGrid g;
  g.n[0] = p->n0;
  g.n[1] = p->n1;
  g.n[2] = p->n2;
  g.sq_base[0] = 0;
  size_t edges = 0;                                    // in-face edges of the six faces (counted per face): table bound
  for (int fc = 0; fc < 6; ++fc) {
    const int axis = fc >> 1, a = axis == 0 ? 1 : 0, b = axis == 2 ? 1 : 2;
    g.sq_base[fc + 1] = g.sq_base[fc] + (g.n[a] - 1) * (g.n[b] - 1);
    edges += 3 * (size_t)g.n[a] * (size_t)g.n[b];
    const int outward = (fc & 1) ? 1 : -1;
    g.wsign[fc] = (cp->side == CTR_CAP_HIGH ? -outward : outward) * (p->delta[a] < 0 ? -1 : 1) * (p->delta[b] < 0 ? -1 : 1);
  }
  g.plane = g.n[1] * g.n[2];
  g.ring = g.plane - (g.n[1] - 2) * (g.n[2] - 2);
  const long long n_sq = g.sq_base[6], n_pts = 2 * g.plane + (g.n[0] - 2) * g.ring;
  if ((unsigned long long)n_sq * 4 > 0xfffff000ull || (unsigned long long)n_pts > 0xfffff000ull)
    return ctr_fail(ctx, CTR_ERR_OVERFLOW, "the box surface has more than 2^32 face-triangle pieces or points");
  g.value = p->isovalue;
  g.side = cp->side;
  for (int a = 0; a < 3; ++a) {
    g.origin[a] = p->origin[a];
    g.delta[a] = p->delta[a];
  }
  size_t nslots = 256;
  while (nslots < 2 * std::min(nV, edges)) nslots <<= 1;
  const int tiles_t = (int)((n_sq * 4 + SC_TILE - 1) / SC_TILE), tiles_p = (int)((n_pts + SC_TILE - 1) / SC_TILE);
  const size_t scan_bytes = 64 + ((size_t)tiles_t + 1 + (size_t)tiles_p + 1) * 8;
  char* scan;
  ufh::Slot* tab;
  uint32_t *piece_flags, *piece_idx, *point_idx;
  uint8_t* point_flags;
  int rc;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_SCRATCH2], [&](ctr_carve& c) {
         c(scan, scan_bytes);
         c(tab, nslots * sizeof(ufh::Slot));
         c(piece_flags, (size_t)n_sq * 4);
         c(piece_idx, (size_t)n_sq * 16);
         c(point_flags, (size_t)n_pts);
         c(point_idx, (size_t)n_pts * 4);
       })))
    return rc;
  CapCounters* ctr = (CapCounters*)scan;
  unsigned long long* st_t = (unsigned long long*)(scan + 64);
  unsigned long long* st_p = st_t + tiles_t + 1;
  CTR_CUDA(ctx, cudaMemsetAsync(scan, 0, scan_bytes, st));
  CTR_CUDA(ctx, cudaMemsetAsync(tab, 0xff, nslots * sizeof(ufh::Slot), st));
  CTR_CUDA(ctx, cudaMemsetAsync(point_flags, 0, (size_t)n_pts, st));
  const T* f = (p->flags & CTR_FIELD_ON_DEVICE) ? (const T*)p->field : (const T*)ctx->field.p;
  const size_t mask = nslots - 1;
  const unsigned sq_blocks = (unsigned)((n_sq + 255) / 256), pt_blocks = (unsigned)((n_pts + 255) / 256);
  if (nT) {
    k_d_ids<<<(unsigned)((nT * 3 + 255) / 256), 256, 0, st>>>((const int*)ctx->tris.p, nT * 3, (unsigned)nV, &ctr->ids);
    ctx->launches++;
  }
  if (nV) {
    k_cap_index<<<(unsigned)((nV + 255) / 256), 256, 0, st>>>((const unsigned long long*)ctx->keys.p, (unsigned)nV, g, tab, mask);
    ctx->launches++;
  }
  k_cap_count<T><<<sq_blocks, 256, 0, st>>>(f, g, tab, mask, piece_flags, point_flags, ctr);
  k_flag_scan<<<tiles_t, SC_THREADS, 0, st>>>((const uint8_t*)piece_flags, (unsigned)(n_sq * 4), piece_idx, st_t, &ctr->ticket[0],
                                              &ctr->total[0], tiles_t);
  k_flag_scan<<<tiles_p, SC_THREADS, 0, st>>>(point_flags, (unsigned)n_pts, point_idx, st_p, &ctr->ticket[1], &ctr->total[1], tiles_p);
  ctx->launches += 3;
  CTR_CUDA(ctx, cudaGetLastError());
  CapCounters h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (h.ids.bad_ids) return fail_shifted_ids(ctx);
  const size_t capT = (size_t)h.total[0], capV = (size_t)h.total[1];
  const size_t newV = nV + capV, newT = nT + capT;
  if (newV > 0x7fffffffull || newT > 0x7fffffffull)
    return ctr_fail(ctx, CTR_ERR_OVERFLOW, "the capped mesh would have 2^31 or more vertices or triangles");
  mesh_edited(ctx, EDIT_CAP);
  const size_t gsz = sizeof(G);
  if ((rc = ctr_grow_keep(ctx, ctx->verts, newV * 3 * gsz, nV * 3 * gsz))) return rc;
  if ((ctx->last_flags & CTR_WANT_NORMALS) && (rc = ctr_grow_keep(ctx, ctx->normals, newV * 3 * gsz, nV * 3 * gsz))) return rc;
  if ((rc = ctr_grow_keep(ctx, ctx->keys, newV * 8, nV * 8))) return rc;
  if ((rc = ctr_grow_keep(ctx, ctx->lowmin, newV, nV))) return rc;
  if ((rc = ctr_grow_keep(ctx, ctx->tris, newT * 12, nT * 12))) return rc;
  if (capV) {
    k_cap_verts<T, G><<<pt_blocks, 256, 0, st>>>(f, g, (unsigned long long)n_pts, point_flags, point_idx, nV, (G*)ctx->verts.p,
                                                 (ctx->last_flags & CTR_WANT_NORMALS) ? (G*)ctx->normals.p : nullptr,
                                                 (unsigned long long*)ctx->keys.p, (uint8_t*)ctx->lowmin.p);
    ctx->launches++;
  }
  if (capT) {
    k_cap_tris<T><<<sq_blocks, 256, 0, st>>>(f, g, tab, mask, piece_flags, piece_idx, point_idx, (unsigned)nV, (unsigned)nT,
                                             (int*)ctx->tris.p);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->last_counts[0] = (int64_t)newV;
  ctx->last_counts[1] = (int64_t)newT;
  out->n_verts = (int64_t)newV;
  out->n_tris = (int64_t)newT;
  out->n_cap_verts = (int64_t)capV;
  out->n_cap_tris = (int64_t)capT;
  out->n_missing = h.n_missing;
  return 0;
}
