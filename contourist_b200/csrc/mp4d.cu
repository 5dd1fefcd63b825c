// 4D marching pentatopes on sm_100a: f(x,y,z,t) = v over a regular 4D grid -> tetrahedra of a 3-manifold,
// then (morph stage) time-binning, instant/tiny filtering and slicing of every tetrahedron into morph triangles.
// Same bitplane-first architecture as mt3d.cu:
//   stage 1 (bitplane.cuh) : the field is streamed ONCE into low / near bitplanes (TMA bulk copies);
//   k4_count_scan          : per 32-hypervoxel word, from the bitplanes: distinct crossing edges (15 Kuhn
//                            directions per owner), tetrahedra (24 pentatopes x {1,3}), decoupled-lookback scan,
//                            compacted owner / hypervoxel lists;
//   k4_emit_verts          : edge crossings in 4D (tetrahedral.py:471-487); with CTR_MORPH also the fp64 grid-coordinate
//                            vertices with binned times, the bins and their range (pentatopes.py:162-169,336-337);
//   k4_emit_tets           : per hypervoxel, 24 pentatopes (pentatopes.py:15-26,223-291) -> tets of vertex ids;
//   k4_slice               : morph_geometry.py:145-237 slicing, single pass (look-back scan, smem-staged output), with
//                            the instant / tiny filter (pentatopes.py:171-189, tetrahedral.py:353-375) folded in when
//                            the integer time bins decide it; k4_tet_filter is the general (fp64) form of that filter.
#include <stdlib.h>

#include "bitplane.cuh"
#include "tables.h"

namespace {

__constant__ uint8_t c4_pent[24][5];
__constant__ uint8_t c4_edge_s[CTR_NEDGE4];
__constant__ uint8_t c4_edge_d[CTR_NEDGE4];
__constant__ uint32_t c4_pentmask[16][16];
__device__ uint8_t d4_tet_n[24][32];
__device__ __align__(4) uint8_t d4_tet_e[24][32][12];

struct Counters4 {
  unsigned long long min_key, max_key;
  unsigned int pad0, pad1;
  unsigned long long n_cells, n_cross, total_vt, total_act, v_emit;
  unsigned int n_own, n_cell;        // list slots handed out to the tiles (= lengths of the owner / hypervoxel lists)
};
constexpr size_t C4_STAGE2_OFFSET = 24;

template <typename T>
struct Grid4 {
  const T* f;
  const uint32_t* bits;
  const uint32_t* nbits;
  const uint8_t* rowflag;
  int n0, n1, n2, n3, W;
  double v, tolv;
  int any_near;
  FastDiv divW, divN2, divN1;
  __device__ __forceinline__ void word_coords(unsigned gw, int& i, int& j, int& k, int& w) const {
    unsigned row = divW.div(gw);
    w = (int)(gw - row * (unsigned)W);
    unsigned ij = divN2.div(row);
    k = (int)(row - ij * (unsigned)n2);
    unsigned ii = divN1.div(ij);
    i = (int)ii;
    j = (int)(ij - ii * (unsigned)n1);
  }
  __device__ __forceinline__ size_t row_of(int i, int j, int k) const { return ((size_t)i * n1 + j) * n2 + k; }
};

template <typename T>
__device__ __forceinline__ double sample4(const Grid4<T>& g, int i, int j, int k, int l) {
  return (double)g.f[g.row_of(i, j, k) * g.n3 + l];
}

__device__ __forceinline__ bool near_a4(double f, double v) {
  return fabs(v - f) <= __dadd_rn(1e-8, __dmul_rn(1e-5, fabs(f)));
}

// 24-bit mask of the pentatopes of hypervoxel (i,j,k,l) that emit tetrahedra (exact, fp64, from the samples)
template <typename T>
__device__ __noinline__ unsigned cell_emit_exact4(const Grid4<T> g, int i, int j, int k, int l, uint8_t* codes24) {
  if (i < 0 || j < 0 || k < 0 || l < 0 || i >= g.n0 - 1 || j >= g.n1 - 1 || k >= g.n2 - 1 || l >= g.n3 - 1) {
    if (codes24)
      for (int p = 0; p < 24; ++p) codes24[p] = 0;
    return 0;
  }
  bool all_a = true;
  unsigned low = 0, nb = 0;
  for (int c = 0; c < 16; ++c) {
    const double fv = sample4(g, i + ((c >> 3) & 1), j + ((c >> 2) & 1), k + ((c >> 1) & 1), l + (c & 1));
    all_a = all_a && near_a4(fv, g.v);
    low |= (fv < g.v ? 1u : 0u) << c;
    nb |= (fabs(fv - g.v) <= g.tolv ? 1u : 0u) << c;
  }
  unsigned emit = 0;
  for (int p = 0; p < 24; ++p) {
    unsigned m = 0, alln = 1;
    for (int b = 0; b < 5; ++b) {
      const int c = c4_pent[p][b];
      m |= ((low >> c) & 1u) << b;
      alln &= (nb >> c) & 1u;
    }
    if (codes24) codes24[p] = (uint8_t)(m | (alln << 5));
    if (m != 0 && m != 31 && !alln) emit |= 1u << p;
  }
  return all_a ? 0u : emit;
}

template <typename T>
__device__ __noinline__ bool edge_used_exact4(const Grid4<T> g, int i, int j, int k, int l, int d) {
  for (int s = 0; s < 16; ++s) {
    if (s & d) continue;
    const unsigned pm = c4_pentmask[d][s];
    if (!pm) continue;
    const unsigned e = cell_emit_exact4(g, i - ((s >> 3) & 1), j - ((s >> 2) & 1), k - ((s >> 1) & 1), l - (s & 1), nullptr);
    if (e & pm) return true;
  }
  return false;
}

// rows (i+a, j+b, k+c), a,b,c in {0,1}: P = bits at l, S = bits at l+1
struct Planes4 {
  uint32_t P[8], S[8];
  uint32_t kpt, kp1;
  bool has[8];                 // row abc exists
};

__device__ __forceinline__ uint32_t low_mask4(int n) { return n >= 32 ? 0xffffffffu : (n <= 0 ? 0u : ((1u << n) - 1u)); }

template <typename T>
__device__ __forceinline__ void load_planes4(const Grid4<T>& g, const uint32_t* __restrict__ plane, int i, int j, int k, int w,
                                             Planes4& pl) {
  const int rem = g.n3 - w * 32;
  pl.kpt = low_mask4(rem);
  pl.kp1 = low_mask4(rem - 1);
#pragma unroll
  for (int abc = 0; abc < 8; ++abc) {
    const int a = abc >> 2, b = (abc >> 1) & 1, c = abc & 1;
    const bool ok = (i + a < g.n0) && (j + b < g.n1) && (k + c < g.n2);
    uint32_t p = 0, nx = 0;
    if (ok) {
      const size_t base = g.row_of(i + a, j + b, k + c) * g.W + w;
      p = plane[base];
      if (w + 1 < g.W) nx = plane[base + 1];
    }
    pl.has[abc] = ok;
    pl.P[abc] = p;
    pl.S[abc] = (p >> 1) | (nx << 31);
  }
}

__device__ __forceinline__ uint32_t corner_plane4(const Planes4& pl, int c) { return (c & 1) ? pl.S[c >> 1] : pl.P[c >> 1]; }

// crossing words for the 15 edge directions of the owner row (index d-1), masked to edges inside the grid
__device__ __forceinline__ void cross_words4(const Planes4& pl, uint32_t x[15]) {
  const uint32_t A = pl.P[0];
#pragma unroll
  for (int d = 1; d <= 15; ++d) {
    const int abc = d >> 1;
    const uint32_t other = (d & 1) ? pl.S[abc] : pl.P[abc];
    const uint32_t valid = ((d & 1) ? pl.kp1 : pl.kpt) & (pl.has[abc] ? 0xffffffffu : 0u);
    x[d - 1] = (A ^ other) & valid;
  }
}

// per word: number of tetrahedra and mask of emitting hypervoxels (fast, bit-sliced; no allclose handling);
// cand = hypervoxels that have a crossing pentatope whose 5 corners are all near
__device__ __forceinline__ void pent_words4(const Planes4& pl, const Planes4* npl, uint32_t cellmask, unsigned& ntet,
                                            uint32_t& emitting, uint32_t& cand) {
  ntet = 0;
  emitting = 0;
  cand = 0;
#pragma unroll
  for (int p = 0; p < 24; ++p) {
    const uint32_t v0 = corner_plane4(pl, c4_pent[p][0]), v1 = corner_plane4(pl, c4_pent[p][1]),
                   v2 = corner_plane4(pl, c4_pent[p][2]), v3 = corner_plane4(pl, c4_pent[p][3]),
                   v4 = corner_plane4(pl, c4_pent[p][4]);
    const uint32_t dif = ((v0 ^ v1) | (v0 ^ v2) | (v0 ^ v3) | (v0 ^ v4)) & cellmask;
    // bit-sliced population count of the 5 low bits: n = s0 + 2*t0 + 4*t1
    const uint32_t a0 = v0 ^ v1 ^ v2, a1 = (v0 & v1) | (v2 & (v0 ^ v1));
    const uint32_t b0 = v3 ^ v4, b1 = v3 & v4;
    const uint32_t c = a0 & b0;
    const uint32_t t0 = a1 ^ b1 ^ c;                 // set <=> 2 or 3 low corners -> 3 tetrahedra, else 1
    ntet += __popc(dif) + 2 * __popc(dif & t0);
    emitting |= dif;
    if (npl) {
      const uint32_t nn = corner_plane4(*npl, c4_pent[p][0]) & corner_plane4(*npl, c4_pent[p][1]) &
                          corner_plane4(*npl, c4_pent[p][2]) & corner_plane4(*npl, c4_pent[p][3]) &
                          corner_plane4(*npl, c4_pent[p][4]);
      cand |= nn & dif;
    }
  }
}

// The out-of-line exact paths take and return their data BY VALUE: a reference to a kernel's registers (grid
// descriptor, bit planes, used-edge words) would pin those to local memory for the whole kernel (mt3d.cu, same note).
struct W15 {
  uint32_t x[15];
};

template <typename T>
__device__ __noinline__ W15 resolve_used_exact4(const Grid4<T> g, int i, int j, int k, int w, W15 in) {
  uint32_t used[15];
#pragma unroll
  for (int d = 0; d < 15; ++d) used[d] = in.x[d];
  Planes4 npl;
  load_planes4(g, g.nbits, i, j, k, w, npl);
  for (int d = 1; d <= 15; ++d) {
    const int abc = d >> 1;
    uint32_t c = used[d - 1] & npl.P[0] & ((d & 1) ? npl.S[abc] : npl.P[abc]);
    while (c) {
      const int b = __ffs(c) - 1;
      c &= c - 1;
      if (!edge_used_exact4(g, i, j, k, w * 32 + b, d)) used[d - 1] &= ~(1u << b);
    }
  }
  W15 out;
#pragma unroll
  for (int d = 0; d < 15; ++d) out.x[d] = used[d];
  return out;
}

template <typename T>
__device__ __forceinline__ void owner_used4(const Grid4<T>& g, const Planes4& pl, int i, int j, int k, int w, uint32_t used[15]) {
  cross_words4(pl, used);
  if (g.any_near) {
    W15 in;
#pragma unroll
    for (int d = 0; d < 15; ++d) in.x[d] = used[d];
    const W15 out = resolve_used_exact4(g, i, j, k, w, in);
#pragma unroll
    for (int d = 0; d < 15; ++d) used[d] = out.x[d];
  }
}

__device__ __forceinline__ unsigned gather15(const uint32_t u[15], int b) {
  unsigned m = 0;
#pragma unroll
  for (int d = 0; d < 15; ++d) m |= ((u[d] >> b) & 1u) << d;
  return m;
}

__device__ __forceinline__ unsigned pent_mask_of(unsigned corner16, int p) {
  unsigned m = 0;
#pragma unroll
  for (int b = 0; b < 5; ++b) m |= ((corner16 >> c4_pent[p][b]) & 1u) << b;
  return m;
}

__device__ __forceinline__ unsigned ntet_of_mask(unsigned m) {       // pentatopes.py:246-291
  const int n = __popc(m);
  return (n == 0 || n == 5) ? 0u : ((n == 1 || n == 4) ? 1u : 3u);
}

struct WordExact4 {
  unsigned ntet;
  uint32_t emitting;
};

template <typename T>
__device__ __noinline__ WordExact4 count_word_exact4(const Grid4<T> g, const Planes4 pl, int i, int j, int k, int w,
                                                     WordExact4 in, uint32_t cand) {
  unsigned ntet = in.ntet;
  uint32_t emitting = in.emitting;
  while (cand) {
    const int b = __ffs(cand) - 1;
    cand &= cand - 1;
    unsigned c16 = 0;
    for (int c = 0; c < 16; ++c) c16 |= ((corner_plane4(pl, c) >> b) & 1u) << c;
    for (int p = 0; p < 24; ++p) ntet -= ntet_of_mask(pent_mask_of(c16, p));
    emitting &= ~(1u << b);
    const unsigned e = cell_emit_exact4(g, i, j, k, w * 32 + b, nullptr);
    if (e) emitting |= 1u << b;
    for (int p = 0; p < 24; ++p)
      if ((e >> p) & 1u) ntet += ntet_of_mask(pent_mask_of(c16, p));
  }
  WordExact4 out;
  out.ntet = ntet;
  out.emitting = emitting;
  return out;
}

// ------------------------------------------------------------------------------------------------
// count + scan (same phase structure as k_count_scan in mt3d.cu)
// ------------------------------------------------------------------------------------------------
constexpr int C4_THREADS = 256;
constexpr int C4_ITEMS = 4;
constexpr int C4_TILE = C4_THREADS * C4_ITEMS;

struct C4Shared {
  uint32_t own[C4_TILE], emit[C4_TILE];
  uint32_t pv[C4_TILE], pt[C4_TILE], po[C4_TILE], pc[C4_TILE];
  unsigned short cv[C4_TILE], ct[C4_TILE];
  unsigned short list[C4_TILE];
  unsigned long long warp_vt[C4_THREADS / 32], warp_act[C4_THREADS / 32];
  unsigned long long excl_vt, excl_act;
  unsigned tile, nint;
};

template <typename T>
__global__ void __launch_bounds__(C4_THREADS, 2) k4_count_scan(Grid4<T> gin, unsigned nwords, uint32_t* __restrict__ vbase,
                                                               unsigned long long* __restrict__ own_id,
                                                               uint32_t* __restrict__ own_voff,
                                                               unsigned long long* __restrict__ cell_id,
                                                               uint32_t* __restrict__ cell_toff, unsigned cap_own,
                                                               unsigned cap_cell, unsigned long long* __restrict__ tile_vt,
                                                               Counters4* ctr, int ntiles) {
  __shared__ C4Shared sh;
  Grid4<T> g = gin;
  g.any_near = 0;
  if (threadIdx.x == 0) sh.nint = 0;
  __syncthreads();
  const int tile = (int)blockIdx.x;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned tile0 = (unsigned)tile * C4_TILE;
  // ---- A: quick test
#pragma unroll 1
  for (int q = 0; q < C4_ITEMS; ++q) {
    const unsigned wl = (unsigned)q * C4_THREADS + threadIdx.x;
    const unsigned gw = tile0 + wl;
    bool interesting = false;
    if (gw < nwords) {
      int i, j, k, w;
      g.word_coords(gw, i, j, k, w);
      Planes4 pl;
      load_planes4(g, g.bits, i, j, k, w, pl);
      uint32_t any = 0;
#pragma unroll
      for (int d = 1; d <= 15; ++d) {
        const int abc = d >> 1;
        const uint32_t other = (d & 1) ? pl.S[abc] : pl.P[abc];
        const uint32_t valid = ((d & 1) ? pl.kp1 : pl.kpt) & (pl.has[abc] ? 0xffffffffu : 0u);
        any |= (pl.P[0] ^ other) & valid;
      }
      interesting = any != 0;
    }
    sh.cv[wl] = 0;
    sh.ct[wl] = 0;
    sh.own[wl] = 0;
    sh.emit[wl] = 0;
    const unsigned m = __ballot_sync(0xffffffffu, interesting);
    unsigned base = 0;
    if (lane == 0 && m) base = atomicAdd(&sh.nint, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (interesting) sh.list[base + __popc(m & ((1u << lane) - 1u))] = (unsigned short)wl;
  }
  __syncthreads();
  const unsigned nint = sh.nint;
  // ---- B: counts
  unsigned ncross = 0, ncells = 0;
  for (unsigned idx = threadIdx.x; idx < nint; idx += C4_THREADS) {
    const unsigned wl = sh.list[idx];
    const unsigned gw = tile0 + wl;
    int i, j, k, w;
    g.word_coords(gw, i, j, k, w);
    g.any_near = g.rowflag[g.row_of(i, j, k)];
    Planes4 pl;
    load_planes4(g, g.bits, i, j, k, w, pl);
    uint32_t x[15];
    owner_used4(g, pl, i, j, k, w, x);
    unsigned v = 0;
    uint32_t any = 0;
#pragma unroll
    for (int d = 0; d < 15; ++d) {
      v += __popc(x[d]);
      any |= x[d];
    }
    const bool cells_ok = pl.has[7];
    unsigned t = 0;
    uint32_t em = 0;
    if (cells_ok) {
      uint32_t xs[15];
      cross_words4(pl, xs);
      Planes4 npl;
      if (g.any_near) load_planes4(g, g.nbits, i, j, k, w, npl);
#pragma unroll
      for (int d = 1; d <= 15; ++d) {
        uint32_t xd = xs[d - 1] & pl.kp1;
        ncross += __popc(xd);
        if (g.any_near) {           // not strict when the high endpoint equals the isovalue exactly
          const int abc = d >> 1;
          const uint32_t A = pl.P[0], O = (d & 1) ? pl.S[abc] : pl.P[abc];
          const uint32_t nO = (d & 1) ? npl.S[abc] : npl.P[abc];
          uint32_t c = xd & ((~A & npl.P[0]) | (~O & nO));
          while (c) {
            const int b = __ffs(c) - 1;
            c &= c - 1;
            const bool a_high = !((A >> b) & 1u);
            const int l = w * 32 + b;
            const double fh = a_high ? sample4(g, i, j, k, l)
                                     : sample4(g, i + ((d >> 3) & 1), j + ((d >> 2) & 1), k + ((d >> 1) & 1), l + (d & 1));
            if (fh == g.v) --ncross;
          }
        }
      }
      uint32_t cand;
      pent_words4(pl, g.any_near ? &npl : nullptr, pl.kp1, t, em, cand);
      if (cand) {
        WordExact4 we;
        we.ntet = t;
        we.emitting = em;
        we = count_word_exact4(g, pl, i, j, k, w, we, cand);
        t = we.ntet;
        em = we.emitting;
      }
    }
    sh.cv[wl] = (unsigned short)v;
    sh.ct[wl] = (unsigned short)t;
    sh.own[wl] = any;
    sh.emit[wl] = em;
    ncells += __popc(em);
  }
  unsigned long long cc = ((unsigned long long)ncross << 32) | ncells;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cc += __shfl_xor_sync(0xffffffffu, cc, o);
  if (lane == 0 && cc) {
    if (cc & 0xffffffffull) atomicAdd(&ctr->n_cells, cc & 0xffffffffull);
    if (cc >> 32) atomicAdd(&ctr->n_cross, cc >> 32);
  }
  __syncthreads();
  // ---- C: scan
  unsigned long long loc_vt = 0, loc_act = 0, item_vt[C4_ITEMS], item_act[C4_ITEMS];
#pragma unroll
  for (int it = 0; it < C4_ITEMS; ++it) {
    const unsigned wl = threadIdx.x * C4_ITEMS + it;
    item_vt[it] = ((unsigned long long)sh.ct[wl] << 31) | sh.cv[wl];
    item_act[it] = ((unsigned long long)__popc(sh.emit[wl]) << 31) | (unsigned)__popc(sh.own[wl]);
    loc_vt += item_vt[it];
    loc_act += item_act[it];
  }
  const unsigned long long inc_vt = warp_incl_scan_u64(loc_vt), inc_act = warp_incl_scan_u64(loc_act);
  if (lane == 31) {
    sh.warp_vt[warp] = inc_vt;
    sh.warp_act[warp] = inc_act;
  }
  __syncthreads();
  unsigned long long woff_vt = 0, woff_act = 0, blk_vt = 0, blk_act = 0;
#pragma unroll
  for (int q = 0; q < C4_THREADS / 32; ++q) {
    if (q < (int)warp) {
      woff_vt += sh.warp_vt[q];
      woff_act += sh.warp_act[q];
    }
    blk_vt += sh.warp_vt[q];
    blk_act += sh.warp_act[q];
  }
  // No tile waits for another: vertex ids / tetrahedron offsets are written RELATIVE to the tile (k4_tile_scan turns
  // the per-tile totals into tile offsets, k4_fix_vbase and the emit kernels add them), and the work-list slots come
  // from two atomic counters (the lists are unordered across tiles; the mesh does not depend on their order).  A
  // look-back scan here cost a quarter of the kernel's stall samples: blocks finish out of order and sat polling.
  if (threadIdx.x == 0) {
    tile_vt[tile] = blk_vt;
    const unsigned no = (unsigned)(blk_act & 0x7fffffffull), nc = (unsigned)(blk_act >> 31);
    const unsigned long long bo = no ? atomicAdd(&ctr->n_own, no) : 0u, bc = nc ? atomicAdd(&ctr->n_cell, nc) : 0u;
    sh.excl_vt = 0ull;
    sh.excl_act = bo | (bc << 31);
  }
  __syncthreads();
  unsigned long long run_vt = sh.excl_vt + woff_vt + inc_vt - loc_vt;
  unsigned long long run_act = sh.excl_act + woff_act + inc_act - loc_act;
#pragma unroll
  for (int it = 0; it < C4_ITEMS; ++it) {
    const unsigned wl = threadIdx.x * C4_ITEMS + it;
    sh.pv[wl] = (uint32_t)(run_vt & 0x7fffffffull);
    sh.pt[wl] = (uint32_t)(run_vt >> 31);
    sh.po[wl] = (uint32_t)(run_act & 0x7fffffffull);
    sh.pc[wl] = (uint32_t)(run_act >> 31);
    if (tile0 + wl < nwords) vbase[tile0 + wl] = sh.pv[wl];
    run_vt += item_vt[it];
    run_act += item_act[it];
  }
  __syncthreads();
  // ---- D: lists
  for (unsigned idx = threadIdx.x; idx < nint; idx += C4_THREADS) {
    const unsigned wl = sh.list[idx];
    uint32_t mo = sh.own[wl], me = sh.emit[wl];
    if (!(mo | me)) continue;
    const unsigned gw = tile0 + wl;
    int i, j, k, w;
    g.word_coords(gw, i, j, k, w);
    g.any_near = g.rowflag[g.row_of(i, j, k)];
    Planes4 pl;
    load_planes4(g, g.bits, i, j, k, w, pl);
    if (mo) {
      uint32_t x[15];
      owner_used4(g, pl, i, j, k, w, x);
      unsigned vrun = sh.pv[wl], orun = sh.po[wl];
      while (mo) {
        const int b = __ffs(mo) - 1;
        mo &= mo - 1;
        const unsigned m15 = gather15(x, b);
        if (orun < cap_own) {
          own_id[orun] = ((unsigned long long)gw << 21) | ((unsigned)b << 16) | (((pl.P[0] >> b) & 1u) << 15) | m15;
          own_voff[orun] = vrun;
        }
        ++orun;
        vrun += __popc(m15);
      }
    }
    if (me) {
      unsigned trun = sh.pt[wl], crun = sh.pc[wl];
      Planes4 npl;
      if (g.any_near) load_planes4(g, g.nbits, i, j, k, w, npl);
      while (me) {
        const int b = __ffs(me) - 1;
        me &= me - 1;
        unsigned c16 = 0;
#pragma unroll
        for (int c = 0; c < 16; ++c) c16 |= ((corner_plane4(pl, c) >> b) & 1u) << c;
        unsigned nt = 0;
        bool cand = false;
        if (g.any_near) {
          unsigned n16 = 0;
          for (int c = 0; c < 16; ++c) n16 |= ((corner_plane4(npl, c) >> b) & 1u) << c;
          for (int p = 0; p < 24; ++p) {
            const unsigned m = pent_mask_of(c16, p);
            cand = cand || (m != 0 && m != 31 && pent_mask_of(n16, p) == 31);
          }
        }
        if (cand) {
          const unsigned e = cell_emit_exact4(g, i, j, k, w * 32 + b, nullptr);
          for (int p = 0; p < 24; ++p)
            if ((e >> p) & 1u) nt += ntet_of_mask(pent_mask_of(c16, p));
        } else {
#pragma unroll 1
          for (int p = 0; p < 24; ++p) nt += ntet_of_mask(pent_mask_of(c16, p));
        }
        if (crun < cap_cell) {
          cell_id[crun] = ((unsigned long long)gw << 22) | ((unsigned)b << 17) | ((cand ? 1u : 0u) << 16) | c16;
          cell_toff[crun] = trun;
        }
        ++crun;
        trun += nt;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// vertices: one thread per (owner, owned edge) pair, dealt out per warp as in mt3d.cu
// ------------------------------------------------------------------------------------------------
// exclusive scan of the per-tile (vertices | tetrahedra << 31) totals: one block, a few thousand tiles
__global__ void __launch_bounds__(1024) k4_tile_scan(const unsigned long long* __restrict__ tile_vt, int ntiles,
                                                     unsigned long long* __restrict__ tile_off, Counters4* ctr) {
  constexpr int PER = 4;                               // consecutive tiles per thread: 4096 tiles in one round
  __shared__ unsigned long long s_warp[32];
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  unsigned long long carry = 0;
  for (int base = 0; base < ntiles; base += 1024 * PER) {
    const int q = base + (int)threadIdx.x * PER;
    unsigned long long c[PER], mine = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      c[u] = q + u < ntiles ? tile_vt[q + u] : 0ull;
      mine += c[u];
    }
    const unsigned long long inc = warp_incl_scan_u64(mine);
    __syncthreads();
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    unsigned long long woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) {
      if (w < (int)warp) woff += s_warp[w];
      tot += s_warp[w];
    }
    unsigned long long run = carry + woff + inc - mine;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      if (q + u < ntiles) tile_off[q + u] = run;
      run += c[u];
    }
    carry += tot;
  }
  if (threadIdx.x == 0) {
    ctr->total_vt = carry;
    ctr->total_act = (unsigned long long)ctr->n_own | ((unsigned long long)ctr->n_cell << 31);
  }
}

// vbase[word]: tile-relative -> absolute first vertex id of the word
__global__ void k4_fix_vbase(uint32_t* __restrict__ vbase, unsigned nwords, const unsigned long long* __restrict__ tile_off) {
  const unsigned w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < nwords) vbase[w] += (uint32_t)(tile_off[w / C4_TILE] & 0x7fffffffull);
}

struct Xform4 {
  double origin[4], delta[4];
};
__device__ __forceinline__ double mul_rn4(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn4(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn4(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn4(float a, float b) { return __fadd_rn(a, b); }

// One thread per owner point: its 1..15 crossing edges (tetrahedral.py:471-487 in 4D), world transform.
// With mverts != nullptr the morph stage's inputs come out of the same visit of the samples: the fp64 grid-coordinate
// vertex with its time snapped down to a bin (pentatopes.py:162-169 bin_times), the bin itself, and the range of the
// binned times (for the zero-duration threshold, pentatopes.py:336-337).
template <typename T, typename G>
__global__ void __launch_bounds__(256) k4_emit_verts(Grid4<T> g, const unsigned long long* __restrict__ own_id,
                                                     const uint32_t* __restrict__ own_voff, unsigned n_own, Xform4 xf,
                                                     G* __restrict__ verts, unsigned long long* __restrict__ keys,
                                                     uint8_t* __restrict__ lowmin, double* __restrict__ mverts,
                                                     int* __restrict__ tbin, double bin_width, MinMaxKeys* mm,
                                                     const unsigned long long* __restrict__ tile_off) {
  const unsigned a = blockIdx.x * blockDim.x + threadIdx.x;
  double tmn = INFINITY, tmx = -INFINITY;
  if (a < n_own) {
    const unsigned long long oid = own_id[a];
    unsigned id = own_voff[a] + (unsigned)(tile_off[(unsigned)(oid >> 21) / C4_TILE] & 0x7fffffffull);   // tile-relative -> absolute
    const unsigned m15 = (unsigned)oid & 0x7fffu;
    const bool p_low = (oid >> 15) & 1u;
    int i, j, k, w;
    g.word_coords((unsigned)(oid >> 21), i, j, k, w);
    const int l = w * 32 + (int)((oid >> 16) & 31u);
    const T fp_raw = g.f[g.row_of(i, j, k) * g.n3 + l];
    const G fp = (G)fp_raw;
    const G v = (G)g.v;
    const unsigned long long lin = (unsigned long long)(g.row_of(i, j, k) * g.n3 + l);
#pragma unroll 1
    for (int d = 1; d <= 15; ++d) {
      if (!((m15 >> (d - 1)) & 1u)) continue;
      const int dd[4] = {(d >> 3) & 1, (d >> 2) & 1, (d >> 1) & 1, d & 1};
      const T fq_raw = g.f[g.row_of(i + dd[0], j + dd[1], k + dd[2]) * g.n3 + l + dd[3]];
      const int p0[4] = {i, j, k, l};
      {
        const G fq = (G)fq_raw;
        const G flow = p_low ? fp : fq, fhigh = p_low ? fq : fp;
        const G den = fhigh - flow;
        const G ratio = (fabs((double)den) <= 1e-8) ? (G)0.5 : (v - flow) / den;
        const G step = p_low ? ratio : -ratio;
#pragma unroll
        for (int ax = 0; ax < 4; ++ax) {
          const G b0 = (G)(p_low ? p0[ax] : p0[ax] + dd[ax]);
          const G x = dd[ax] ? add_rn4(b0, step) : b0;
          verts[(size_t)id * 4 + ax] = add_rn4(mul_rn4(x, (G)xf.delta[ax]), (G)xf.origin[ax]);
        }
      }
      if (mverts) {
        const double fpd = (double)fp_raw, fqd = (double)fq_raw;
        const double flow = p_low ? fpd : fqd, fhigh = p_low ? fqd : fpd;
        const double den = fhigh - flow;
        const double ratio = (fabs(den) <= 1e-8) ? 0.5 : (g.v - flow) / den;
        const double step = p_low ? ratio : -ratio;
        double x[4];
#pragma unroll
        for (int ax = 0; ax < 4; ++ax) {
          const double b0 = (double)(p_low ? p0[ax] : p0[ax] + dd[ax]);
          x[ax] = dd[ax] ? __dadd_rn(b0, step) : b0;
        }
        const double b = trunc(x[3] / bin_width);
        x[3] = __dmul_rn(b, bin_width);                                             // pentatopes.py:168-169
        tbin[id] = (int)fmax(fmin(b, 1.0e9), -1.0e9);
        reinterpret_cast<double2*>(mverts + (size_t)id * 4)[0] = make_double2(x[0], x[1]);
        reinterpret_cast<double2*>(mverts + (size_t)id * 4)[1] = make_double2(x[2], x[3]);
        tmn = fmin(tmn, x[3]);
        tmx = fmax(tmx, x[3]);
      }
      if (keys) {
        keys[id] = (lin << 4) | (unsigned)d;
        lowmin[id] = p_low ? 1 : 0;
      }
      ++id;
    }
  }
  if (mverts) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      tmn = fmin(tmn, __shfl_xor_sync(0xffffffffu, tmn, o));
      tmx = fmax(tmx, __shfl_xor_sync(0xffffffffu, tmx, o));
    }
    if (lane_id() == 0 && tmn <= tmx) {
      atomicMin(&mm->min_key, order_key(tmn));
      atomicMax(&mm->max_key, order_key(tmx));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// tetrahedra: one thread per hypervoxel
// ------------------------------------------------------------------------------------------------
constexpr int E4_THREADS = 64;

#ifndef CTR_E4_MINB
#define CTR_E4_MINB 8           // 128 registers: 0.565 ms (unbounded 161: 0.615; 10 -> 96: 0.681; 12 -> 80: 0.744)
#endif
#define CTR_E4_BOUNDS __launch_bounds__(E4_THREADS, CTR_E4_MINB)
template <typename T>
__global__ void CTR_E4_BOUNDS k4_emit_tets(Grid4<T> gin, const unsigned long long* __restrict__ cell_id,
                                                           const uint32_t* __restrict__ cell_toff, unsigned n_cells,
                                                           const uint32_t* __restrict__ vbase, int* __restrict__ tets,
                                                           uint8_t* __restrict__ codes,
                                                           const unsigned long long* __restrict__ tile_off) {
  __shared__ unsigned s_ids[CTR_NEDGE4][E4_THREADS];
  Grid4<T> g = gin;
  const unsigned a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_cells) return;
  const unsigned long long cid = cell_id[a];
  const unsigned c16 = (unsigned)cid & 0xffffu;
  const bool cand = (cid >> 16) & 1u;
  const int b = (int)((cid >> 17) & 31u);
  int i, j, k, w;
  g.word_coords((unsigned)(cid >> 22), i, j, k, w);
  g.any_near = g.rowflag[g.row_of(i, j, k)];
  // owner (first vertex id, mask15) for the 16 corners: owner rows abc (8) x {l, l+1}
  unsigned idb[16], msk[16];
  const uint32_t below = (1u << b) - 1u;
#pragma unroll 1
  for (int abc = 0; abc < 8; ++abc) {
    const int ii = i + (abc >> 2), jj = j + ((abc >> 1) & 1), kk = k + (abc & 1);
    Planes4 pl;
    load_planes4(g, g.bits, ii, jj, kk, w, pl);
    uint32_t u[15];
    owner_used4(g, pl, ii, jj, kk, w, u);
    const size_t wi = g.row_of(ii, jj, kk) * g.W + w;
    unsigned rank = 0;
#pragma unroll
    for (int d = 0; d < 15; ++d) rank += __popc(u[d] & below);
    const unsigned m0 = gather15(u, b);
    const unsigned id0 = vbase[wi] + rank;
    unsigned m1, id1;
    if (b < 31) {
      m1 = gather15(u, b + 1);
      id1 = id0 + __popc(m0);
    } else {
      Planes4 pn;
      load_planes4(g, g.bits, ii, jj, kk, w + 1, pn);
      uint32_t un[15];
      owner_used4(g, pn, ii, jj, kk, w + 1, un);
      m1 = gather15(un, 0);
      id1 = vbase[wi + 1];
    }
    idb[abc * 2 + 0] = id0;
    msk[abc * 2 + 0] = m0;
    idb[abc * 2 + 1] = id1;
    msk[abc * 2 + 1] = m1;
  }
#pragma unroll
  for (int e = 0; e < CTR_NEDGE4; ++e) {
    const int s = c4_edge_s[e], d = c4_edge_d[e];
    s_ids[e][threadIdx.x] = idb[s] + __popc(msk[s] & ((1u << (d - 1)) - 1u));
  }
  unsigned emit = 0xffffffu;
  if (cand) emit = cell_emit_exact4(g, i, j, k, w * 32 + b, nullptr);
  if (codes) cell_emit_exact4(g, i, j, k, w * 32 + b, codes + (size_t)a * 24);
  size_t o = (size_t)cell_toff[a] + (size_t)(tile_off[(unsigned)(cid >> 22) / C4_TILE] >> 31);   // tile-relative -> absolute
#pragma unroll 1
  for (int p = 0; p < 24; ++p) {
    const unsigned m = pent_mask_of(c16, p);
    if (m == 0 || m == 31 || !((emit >> p) & 1u)) continue;
    const int n = d4_tet_n[p][m];
    for (int q = 0; q < n; ++q) {
      // the four edge slots of the tetrahedron in one 32-bit load, its four vertex ids in one 128-bit store
      const uint32_t e4 = *reinterpret_cast<const uint32_t*>(&d4_tet_e[p][m][q * 4]);
      int4 t4;
      t4.x = (int)s_ids[e4 & 255u][threadIdx.x];
      t4.y = (int)s_ids[(e4 >> 8) & 255u][threadIdx.x];
      t4.z = (int)s_ids[(e4 >> 16) & 255u][threadIdx.x];
      t4.w = (int)s_ids[e4 >> 24][threadIdx.x];
      *reinterpret_cast<int4*>(tets + o * 4) = t4;
      ++o;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// morph stage (grid coordinates, fp64): pentatopes.py:162-189, tetrahedral.py:353-375, morph_geometry.py:145-237
// ------------------------------------------------------------------------------------------------
struct MorphParams {
  double inv_corner[4];
  double eps_instant, eps_tiny, eps_gap, eps_in, t_eps;
};

// keep[t] = 1 unless the tet is instantaneous (t extent < eps_instant) or tiny (every extent/corner < eps_tiny).
// Both verdicts need the (z, t) halves of the four vertices; x and y only matter when z and t are already tiny, which
// almost never happens: they are loaded on that path only (half the gather traffic, half the instructions).
__global__ void k4_tet_filter(const double* __restrict__ verts, const int* __restrict__ tets, unsigned nt, MorphParams mp,
                              uint8_t* __restrict__ keep) {
  const unsigned a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= nt) return;
  const int4 t4 = *reinterpret_cast<const int4*>(tets + (size_t)a * 4);
  const int tv[4] = {t4.x, t4.y, t4.z, t4.w};
  double2 zt[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) zt[r] = reinterpret_cast<const double2*>(verts + (size_t)tv[r] * 4)[1];
  const double zmn = fmin(fmin(zt[0].x, zt[1].x), fmin(zt[2].x, zt[3].x)), zmx = fmax(fmax(zt[0].x, zt[1].x), fmax(zt[2].x, zt[3].x));
  const double tmn = fmin(fmin(zt[0].y, zt[1].y), fmin(zt[2].y, zt[3].y)), tmx = fmax(fmax(zt[0].y, zt[1].y), fmax(zt[2].y, zt[3].y));
  const bool instant = (tmx - tmn) < mp.eps_instant;
  double ext = fmax(__dmul_rn(zmx - zmn, mp.inv_corner[2]), __dmul_rn(tmx - tmn, mp.inv_corner[3]));
  bool tiny = false;
  if (!instant && ext < mp.eps_tiny) {
    double2 xy[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) xy[r] = reinterpret_cast<const double2*>(verts + (size_t)tv[r] * 4)[0];
    const double xmn = fmin(fmin(xy[0].x, xy[1].x), fmin(xy[2].x, xy[3].x)), xmx = fmax(fmax(xy[0].x, xy[1].x), fmax(xy[2].x, xy[3].x));
    const double ymn = fmin(fmin(xy[0].y, xy[1].y), fmin(xy[2].y, xy[3].y)), ymx = fmax(fmax(xy[0].y, xy[1].y), fmax(xy[2].y, xy[3].y));
    ext = fmax(ext, fmax(__dmul_rn(xmx - xmn, mp.inv_corner[0]), __dmul_rn(ymx - ymn, mp.inv_corner[1])));
    tiny = ext < mp.eps_tiny;
  }
  keep[a] = (instant || tiny) ? 0 : 1;
}

// slices of one tetrahedron: returns the number of morph triangles; if out != nullptr writes them as
// 3 segments x (low id, high id) with the deterministic 4-edge split (first edge in (ab,ac,ad,bc,bd,cd) order
// of the id-sorted vertices + the edge disjoint from it are the shared pair).
// Slicing of one tetrahedron at the midpoints of its t-gaps (morph_geometry.py:145-237), done ONCE per tetrahedron:
// the result is a 64-bit code (up to 6 morph triangles x 3 tetrahedron edges x 3 bits) that the emit step only decodes.
// Edge e joins corners EA(e), EB(e) of the id-sorted tetrahedron; opposite edges are e and 5 - e.
__device__ __forceinline__ constexpr int EA(int e) { return e < 3 ? 0 : e < 5 ? 1 : 2; }
__device__ __forceinline__ constexpr int EB(int e) { return e == 0 ? 1 : e == 1 ? 2 : e == 2 ? 3 : e == 3 ? 2 : 3; }

// per 6-bit mask of the edges cut by a slice: triangle count | (e0 | e1<<3 | e2<<6) << 2 | second triangle << 11
__device__ __forceinline__ unsigned slice_entry(unsigned mask) {
  int inter[6], ni = 0;
  for (int e = 0; e < 6; ++e)
    if ((mask >> e) & 1u) inter[ni++] = e;
  if (ni == 3) return 1u | ((unsigned)(inter[0] | (inter[1] << 3) | (inter[2] << 6)) << 2);
  if (ni == 4) {                                                   // morph_geometry.py:176-186
    const int p1 = inter[0], p2 = 5 - p1;                          // the edge sharing no corner with p1
    if (!((mask >> p2) & 1u)) return 0u;
    unsigned out = 0, ntri = 0;
    for (int q = 1; q < 4; ++q)
      if (inter[q] != p2) {
        out |= (unsigned)(p1 | (p2 << 3) | (inter[q] << 6)) << (2 + 9 * ntri);
        ++ntri;
      }
    return out | ntri;
  }
  return 0u;
}

constexpr int SL_THREADS = 256;


// The time comparisons of the slicing, on the binned times themselves (fp64, the reference's tolerances) or -- when
// the bin width dwarfs every tolerance, i.e. always in practice -- on the integer bins: binned times are bin * width, so
// "gap > 1e-4" is "bins differ", "mid +- 1e-5 inside [lo, hi]" is "2 lo < a + b < 2 hi" (a slice midpoint never
// coincides with a corner time: the two sorted times it lies between are adjacent), "|dt| <= 1e-7 range" is "bins equal".
template <typename TT>
struct TimeOps;
template <>
struct TimeOps<double> {
  static __device__ __forceinline__ double mn(double a, double b) { return fmin(a, b); }
  static __device__ __forceinline__ double mx(double a, double b) { return fmax(a, b); }
  static __device__ __forceinline__ bool gap(double a, double b, const MorphParams& mp) { return (b - a) > mp.eps_gap; }
  static __device__ __forceinline__ bool cut(double lo, double hi, double a, double b, const MorphParams& mp) {
    const double mid = 0.5 * (b + a);
    return !(mid + mp.eps_in < lo || mid - mp.eps_in > hi);                         // morph_geometry.py:218
  }
  static __device__ __forceinline__ bool same(double a, double b, const MorphParams& mp) { return fabs(a - b) <= mp.t_eps; }
  static __device__ __forceinline__ double load(const double* verts, const int*, int v) { return verts[(size_t)v * 4 + 3]; }
};
template <>
struct TimeOps<int> {
  static __device__ __forceinline__ int mn(int a, int b) { return min(a, b); }
  static __device__ __forceinline__ int mx(int a, int b) { return max(a, b); }
  static __device__ __forceinline__ bool gap(int a, int b, const MorphParams&) { return b > a; }
  static __device__ __forceinline__ bool cut(int lo, int hi, int a, int b, const MorphParams&) {
    const int s2 = a + b;
    return !(s2 < 2 * lo || s2 > 2 * hi);
  }
  static __device__ __forceinline__ bool same(int a, int b, const MorphParams&) { return a == b; }
  static __device__ __forceinline__ int load(const double*, const int* tbin, int v) { return tbin[v]; }
};

// returns the number of morph triangles of the tetrahedron and their code; v = corner ids sorted, tv = their t
template <typename TT>
__device__ __forceinline__ int slice_code(const TT tv[4], const MorphParams& mp, const unsigned* __restrict__ s_tab,
                                          unsigned long long& code) {
  typedef TimeOps<TT> Op;
  TT ts[4] = {tv[0], tv[1], tv[2], tv[3]};
#define CTR_CSWAP(a, b)            \
  {                                \
    const TT lo = Op::mn(a, b);    \
    b = Op::mx(a, b);              \
    a = lo;                        \
  }
  CTR_CSWAP(ts[0], ts[1]) CTR_CSWAP(ts[2], ts[3]) CTR_CSWAP(ts[0], ts[2]) CTR_CSWAP(ts[1], ts[3]) CTR_CSWAP(ts[1], ts[2])
#undef CTR_CSWAP
  // edges whose two ends are (nearly) simultaneous: a morph triangle using one is dropped (pentatopes.py:339-348)
  unsigned killmask = 0;
#pragma unroll
  for (int e = 0; e < 6; ++e)
    if (Op::same(tv[EA(e)], tv[EB(e)], mp)) killmask |= 1u << e;
  // t-extent of every edge, once (the three slices test the same six intervals)
  TT e_lo[6], e_hi[6];
#pragma unroll
  for (int e = 0; e < 6; ++e) {
    e_lo[e] = Op::mn(tv[EA(e)], tv[EB(e)]);
    e_hi[e] = Op::mx(tv[EA(e)], tv[EB(e)]);
  }
  int n = 0;
  code = 0ull;
#pragma unroll
  for (int gap = 0; gap < 3; ++gap) {
    if (!Op::gap(ts[gap], ts[gap + 1], mp)) continue;
    unsigned mask = 0;
#pragma unroll
    for (int e = 0; e < 6; ++e)
      if (Op::cut(e_lo[e], e_hi[e], ts[gap], ts[gap + 1], mp)) mask |= 1u << e;
    unsigned ent = s_tab[mask];
    const unsigned ntri = ent & 3u;
    ent >>= 2;
    for (unsigned q = 0; q < ntri; ++q, ent >>= 9) {
      const unsigned t9 = ent & 511u;
      const unsigned em = (1u << (t9 & 7u)) | (1u << ((t9 >> 3) & 7u)) | (1u << (t9 >> 6));
      if (em & killmask) continue;
      code |= (unsigned long long)t9 << (9 * n);
      ++n;
    }
  }
  return n;
}

// On integer time bins the whole slicing of a tetrahedron depends only on how its four bins compare pairwise: a weak
// ordering of four elements (75 of them).  The pattern -- 2 bits (less, equal) per pair (0,1),(0,2),(0,3),(1,2),(1,3),(2,3)
// -- indexes a table built once by running slice_code on one representative per pattern:
//   entry = triangle code (54 bits) | triangle count << 54 | low-t-first flags of the six edges << 57.
__device__ __forceinline__ unsigned order_pattern(const int tv[4]) {
  unsigned p = 0;
#pragma unroll
  for (int e = 0; e < 6; ++e) {
    const int a = tv[EA(e)], b = tv[EB(e)];
    p |= ((a < b ? 1u : 0u) | (a == b ? 2u : 0u)) << (2 * e);
  }
  return p;
}

__global__ void k4_slice_table(unsigned long long* __restrict__ tab, MorphParams mp) {
  __shared__ unsigned s_tab[64];
  if (threadIdx.x < 64) s_tab[threadIdx.x] = slice_entry(threadIdx.x);
  __syncthreads();
  const int tv[4] = {(int)(threadIdx.x & 3u), (int)((threadIdx.x >> 2) & 3u), (int)((threadIdx.x >> 4) & 3u), (int)(threadIdx.x >> 6)};
  unsigned long long code;
  const int n = slice_code<int>(tv, mp, s_tab, code);
  unsigned swapm = 0;
#pragma unroll
  for (int e = 0; e < 6; ++e)
    if (tv[EA(e)] > tv[EB(e)]) swapm |= 1u << e;
  tab[order_pattern(tv)] = code | ((unsigned long long)n << 54) | ((unsigned long long)swapm << 57);   // equal patterns, equal entries
}

struct SlCounters {
  unsigned long long total;
  unsigned int ticket, pad;
};

constexpr int SL_PER = 4;                            // consecutive tetrahedra per thread (10^5 tiles of 256 would
constexpr int SL_TILE = SL_THREADS * SL_PER;         // serialise on the ticket atomic and on the look-back)
constexpr int SL_MAXTRI = SL_TILE * 6;               // a tetrahedron gives at most 3 slices x 2 triangles

// What the write-out needs of one tetrahedron, as arrays over the tile's tetrahedra (structure of arrays: a round of
// the write-out reads the records of ~32 consecutive tetrahedra, one word per lane and field -> no bank conflicts):
// id-sorted corners v[0..3], triangle code (two halves), low-t-first flags | first triangle << 8.
constexpr int SL_FIELDS = 7;
constexpr int SL_SMEM = SL_TILE * SL_FIELDS * 4 + SL_MAXTRI * 2;        // records + the tetrahedron of every triangle

template <typename TT>
__device__ __forceinline__ bool slice_load(const double* __restrict__ verts, const int* __restrict__ tbin,
                                           const int* __restrict__ tets, unsigned a, int v[4], TT tv[4]) {
  const int4 t4 = *reinterpret_cast<const int4*>(tets + (size_t)a * 4);
  v[0] = t4.x; v[1] = t4.y; v[2] = t4.z; v[3] = t4.w;
#define CTR_ISWAP(a, b)          \
  {                              \
    const int lo = min(a, b);    \
    b = max(a, b);               \
    a = lo;                      \
  }
  CTR_ISWAP(v[0], v[1]) CTR_ISWAP(v[2], v[3]) CTR_ISWAP(v[0], v[2]) CTR_ISWAP(v[1], v[3]) CTR_ISWAP(v[1], v[2])
#undef CTR_ISWAP
#pragma unroll
  for (int r = 0; r < 4; ++r) tv[r] = TimeOps<TT>::load(verts, tbin, v[r]);
  return !(v[0] == v[1] || v[1] == v[2] || v[2] == v[3]);
}

// fp64 times: the reference's tolerances, evaluated; integer bins: the pattern table
template <typename TT>
__device__ __forceinline__ void slice_lookup(const TT tv[4], const MorphParams& mp, const unsigned* __restrict__ s_tab,
                                             const unsigned long long* __restrict__, unsigned long long& code, int& cnt, unsigned& swapm) {
  cnt = slice_code<TT>(tv, mp, s_tab, code);
#pragma unroll
  for (int e = 0; e < 6; ++e)
    if (tv[EA(e)] > tv[EB(e)]) swapm |= 1u << e;                  // morph_geometry.py:13-17: low t first
}
template <>
__device__ __forceinline__ void slice_lookup<int>(const int tv[4], const MorphParams&, const unsigned* __restrict__,
                                                  const unsigned long long* __restrict__ pattern_tab, unsigned long long& code,
                                                  int& cnt, unsigned& swapm) {
  const unsigned long long ent = __ldg(pattern_tab + order_pattern(tv));
  code = ent & ((1ull << 54) - 1ull);
  cnt = (int)((ent >> 54) & 7ull);
  swapm = (unsigned)(ent >> 57) & 63u;
}

template <typename TT>
__global__ void __launch_bounds__(SL_THREADS) k4_slice(const double* __restrict__ verts, const int* __restrict__ tbin,
                                                       const int* __restrict__ tets,
                                                       const uint8_t* __restrict__ keep, uint8_t* __restrict__ keep_out,
                                                       unsigned nt, MorphParams mp,
                                                       unsigned long long* status, SlCounters* ctr, int ntiles,
                                                       int* __restrict__ out, unsigned cap,
                                                       const unsigned long long* __restrict__ pattern_tab) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  unsigned* s_f = reinterpret_cast<unsigned*>(s_dyn);                        // [SL_FIELDS][SL_TILE]
  unsigned short* s_own = reinterpret_cast<unsigned short*>(s_dyn + SL_TILE * SL_FIELDS * 4);   // [SL_MAXTRI]
  __shared__ unsigned s_tile;
  __shared__ unsigned s_tab[64];
  __shared__ unsigned long long s_warp[SL_THREADS / 32], s_excl;
  if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket, 1u);
  if (threadIdx.x < 64) s_tab[threadIdx.x] = slice_entry(threadIdx.x);
  __syncthreads();
  const int tile = (int)s_tile;
  const unsigned tile0 = (unsigned)tile * SL_TILE;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  // tetrahedron u of this thread is number u * 256 + thread in the tile: consecutive lanes, consecutive tetrahedra
  unsigned long long code[SL_PER];
  int cnt[SL_PER];
  int vv[SL_PER][4];                                  // id-sorted corners and low-t-first flags, kept for the write phase
  unsigned swapm[SL_PER];
  unsigned long long n4 = 0;                          // the four counts, 16 bits each (a quarter tile has <= 1536 triangles)
#pragma unroll
  for (int u = 0; u < SL_PER; ++u) {
    cnt[u] = 0;
    code[u] = 0ull;
    swapm[u] = 0;
    vv[u][0] = vv[u][1] = vv[u][2] = vv[u][3] = 0;
    const unsigned a = tile0 + (unsigned)u * SL_THREADS + threadIdx.x;
    if (a < nt && (keep_out || keep[a])) {
      TT tv[4];
      const bool distinct = slice_load<TT>(verts, tbin, tets, a, vv[u], tv);
      bool kept = true;
      if (keep_out) {
        // the instant / tiny filter folded in (host guarantees: a tetrahedron spanning two bins is neither): keep
        // unless all four vertices share a time bin
        typedef TimeOps<TT> Op;
        kept = Op::gap(Op::mn(Op::mn(tv[0], tv[1]), Op::mn(tv[2], tv[3])), Op::mx(Op::mx(tv[0], tv[1]), Op::mx(tv[2], tv[3])), mp);
        keep_out[a] = kept ? 1 : 0;
      }
      if (distinct && kept) slice_lookup<TT>(tv, mp, s_tab, pattern_tab, code[u], cnt[u], swapm[u]);
    }
    n4 |= (unsigned long long)cnt[u] << (16 * u);
  }
  // one packed scan gives the prefix of every quarter (threads of one u) at once
  const unsigned long long inc = warp_incl_scan_u64(n4);
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  unsigned long long woff = 0, tot4 = 0;
#pragma unroll
  for (int q = 0; q < SL_THREADS / 32; ++q) {
    if (q < (int)warp) woff += s_warp[q];
    tot4 += s_warp[q];
  }
  const unsigned long long excl4 = woff + inc - n4;           // per quarter: triangles of the threads before this one
  unsigned qbase[SL_PER], blk = 0;
#pragma unroll
  for (int u = 0; u < SL_PER; ++u) {
    qbase[u] = blk;                                            // triangles of the quarters before quarter u
    blk += (unsigned)(tot4 >> (16 * u)) & 0xffffu;
  }
  // The tile's aggregate is published at once; the look-back is resolved after the records below have been staged: by
  // then the predecessors have published theirs and the warp does not sit polling.
  if (warp == 0) lb_publish(status, tile, (unsigned long long)blk);
  // A thread that wrote its own triangles would run as long as the warp's busiest lane with most lanes idle; instead
  // every tetrahedron leaves a record in shared memory and marks its triangles with its number, and the tile's
  // triangles are then dealt out one per thread per round.
#pragma unroll
  for (int u = 0; u < SL_PER; ++u) {
    const unsigned tl = (unsigned)u * SL_THREADS + threadIdx.x;
    const unsigned loc = qbase[u] + ((unsigned)(excl4 >> (16 * u)) & 0xffffu);
    s_f[0 * SL_TILE + tl] = (unsigned)vv[u][0];
    s_f[1 * SL_TILE + tl] = (unsigned)vv[u][1];
    s_f[2 * SL_TILE + tl] = (unsigned)vv[u][2];
    s_f[3 * SL_TILE + tl] = (unsigned)vv[u][3];
    s_f[4 * SL_TILE + tl] = (unsigned)(code[u] & 0xffffffffull);
    s_f[5 * SL_TILE + tl] = (unsigned)(code[u] >> 32);
    s_f[6 * SL_TILE + tl] = swapm[u] | (loc << 8);
    for (int q = 0; q < cnt[u]; ++q) s_own[loc + q] = (unsigned short)tl;
  }
  if (warp == 0) {
    unsigned long long e = lb_resolve(status, tile, (unsigned long long)blk);
    if (lane == 0) s_excl = e;
  }
  __syncthreads();
  const unsigned long long base = s_excl;
  for (unsigned q = threadIdx.x; q < blk; q += SL_THREADS) {
    if (base + q >= cap) break;
    const unsigned tl = s_own[q];
    const unsigned sf = s_f[6 * SL_TILE + tl];
    const unsigned idx = q - (sf >> 8);
    const unsigned long long c = ((unsigned long long)s_f[5 * SL_TILE + tl] << 32) | s_f[4 * SL_TILE + tl];
    const unsigned t9 = (unsigned)(c >> (9 * idx)) & 511u;
    int2* o = reinterpret_cast<int2*>(out + (base + q) * 6);
#pragma unroll
    for (int rr = 0; rr < 3; ++rr) {
      const unsigned e = (t9 >> (3 * rr)) & 7u;
      // corners of edge e: EA = {0,0,0,1,1,2}, EB = {1,2,3,2,3,3} as 2-bit fields
      const int i0 = (int)s_f[((0x940u >> (2 * e)) & 3u) * SL_TILE + tl], i1 = (int)s_f[((0xfb9u >> (2 * e)) & 3u) * SL_TILE + tl];
      const bool swap = (sf >> e) & 1u;
      o[rr] = swap ? make_int2(i1, i0) : make_int2(i0, i1);
    }
  }
  if (tile == ntiles - 1 && threadIdx.x == 0) ctr->total = s_excl + blk;
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
bool g4_tables_loaded[64] = {};

int load_tables4(ctr_ctx* ctx) {
  if (ctx->device < 64 && g4_tables_loaded[ctx->device]) return 0;
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c4_pent, CTR_PENT4_H, sizeof(CTR_PENT4_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c4_edge_s, CTR_EDGE4_S_H, sizeof(CTR_EDGE4_S_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c4_edge_d, CTR_EDGE4_D_H, sizeof(CTR_EDGE4_D_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c4_pentmask, CTR_PENTMASK4_H, sizeof(CTR_PENTMASK4_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(d4_tet_n, CTR_TET4_N_H, sizeof(CTR_TET4_N_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(d4_tet_e, CTR_TET4_E_H, sizeof(CTR_TET4_E_H)));
  if (ctx->device < 64) g4_tables_loaded[ctx->device] = true;
  return 0;
}

// buffers of the 4D path: generic slots 12.. of the context
struct Bufs4 {
  DevBuf &own_id, &own_voff, &cell_id, &cell_toff, &rowflag, &verts, &keys, &lowmin, &tets, &codes, &keep, &mverts, &mtris,
      &slstate, &tbin;
  explicit Bufs4(ctr_ctx* c)
      : own_id(c->aux[12]), own_voff(c->aux[13]), cell_id(c->aux[14]), cell_toff(c->aux[15]), rowflag(c->aux[16]),
        verts(c->aux[17]), keys(c->aux[18]), lowmin(c->aux[19]), tets(c->aux[20]), codes(c->aux[21]), keep(c->aux[22]),
        mverts(c->aux[23]), mtris(c->aux[24]), slstate(c->aux[25]), tbin(c->aux[26]) {}
};

template <typename T>
int run4d(ctr_ctx* ctx, const ctr_mp4d_params* p, ctr_mp4d_counts* out) {
  const int n0 = (int)p->n0, n1 = (int)p->n1, n2 = (int)p->n2, n3 = (int)p->n3;
  const int W = (n3 + 31) / 32;
  const long long nrows = (long long)n0 * n1 * n2;
  const long long nwords = nrows * W;
  const size_t nsamp = (size_t)nrows * n3;
  cudaStream_t st = ctx->stream;
  if (nwords >= (1ll << 31) - 64) return ctr_fail(ctx, CTR_ERR_UNSUPPORTED, "4D field too large for 32-bit word indices");
  Bufs4 B(ctx);
  int rc;
  if ((rc = load_tables4(ctx))) return rc;
  ctr_stage_mark(ctx, 0);
  const T* df;
  if (p->flags & CTR_FIELD_ON_DEVICE) {
    df = (const T*)p->field;
  } else {
    if ((rc = ctr_ensure(ctx, ctx->field, nsamp * sizeof(T)))) return rc;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->field.p, p->field, nsamp * sizeof(T), cudaMemcpyHostToDevice, st));
    df = (const T*)ctx->field.p;
  }
  ctr_stage_mark(ctx, 1);
  if ((rc = ctr_ensure(ctx, ctx->bits, (size_t)(nwords + 4) * 4))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->nbits, (size_t)(nwords + 4) * 4))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->vbase, (size_t)(nwords + 4) * 4))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->counters, 256))) return rc;
  if ((rc = ctr_ensure(ctx, B.rowflag, (size_t)nrows + 16))) return rc;
  if (!ctx->counters_host) CTR_CUDA(ctx, cudaMallocHost(&ctx->counters_host, 1024));
  Counters4 init;
  memset(&init, 0, sizeof init);
  init.min_key = ~0ull;
  memcpy(ctx->counters_host, &init, sizeof init);
  CTR_CUDA(ctx, cudaMemcpyAsync(ctx->counters.p, ctx->counters_host, sizeof init, cudaMemcpyHostToDevice, st));
  Counters4* dctr = (Counters4*)ctx->counters.p;
  rc = launch_bitplane<T>(ctx, df, (unsigned)nrows, n3, W, n1, n2, p->isovalue, (uint32_t*)ctx->bits.p, (uint32_t*)ctx->nbits.p,
                          (uint8_t*)B.rowflag.p, (MinMaxKeys*)dctr, (p->flags & CTR_WANT_MINMAX) != 0);
  if (rc) return rc;
  ctr_stage_mark(ctx, 2);
  Grid4<T> g;
  g.f = df;
  g.bits = (const uint32_t*)ctx->bits.p;
  g.nbits = (const uint32_t*)ctx->nbits.p;
  g.rowflag = (const uint8_t*)B.rowflag.p;
  g.n0 = n0; g.n1 = n1; g.n2 = n2; g.n3 = n3; g.W = W;
  g.v = p->isovalue;
  g.tolv = 1e-8 + 1e-5 * fabs(p->isovalue);
  g.any_near = 0;
  g.divW.init((unsigned)W);
  g.divN2.init((unsigned)n2);
  g.divN1.init((unsigned)n1);
  const int ntiles = (int)((nwords + C4_TILE - 1) / C4_TILE);
  if ((rc = ctr_ensure(ctx, ctx->tile_state, (size_t)ntiles * 16 + 16))) return rc;
  unsigned long long* st_vt = (unsigned long long*)ctx->tile_state.p;       // per-tile totals
  unsigned long long* tile_off = st_vt + ntiles;                              // their exclusive prefix
  size_t want_own = std::max<size_t>((size_t)nwords / 2, 1 << 14), want_cell = want_own;
  Counters4 h;
  unsigned long long totV = 0, totT = 0, nOwn = 0, nCell = 0;
  for (int attempt = 0; attempt < 3; ++attempt) {
    if ((rc = ctr_ensure(ctx, B.own_id, want_own * 8))) return rc;
    if ((rc = ctr_ensure(ctx, B.own_voff, want_own * 4))) return rc;
    if ((rc = ctr_ensure(ctx, B.cell_id, want_cell * 8))) return rc;
    if ((rc = ctr_ensure(ctx, B.cell_toff, want_cell * 4))) return rc;
    const unsigned cap_own = (unsigned)std::min<size_t>(std::min(B.own_id.cap / 8, B.own_voff.cap / 4), 0x7fffffffu);
    const unsigned cap_cell = (unsigned)std::min<size_t>(std::min(B.cell_id.cap / 8, B.cell_toff.cap / 4), 0x7fffffffu);
    CTR_CUDA(ctx, cudaMemsetAsync((char*)dctr + C4_STAGE2_OFFSET, 0, sizeof(Counters4) - C4_STAGE2_OFFSET, st));
    k4_count_scan<T><<<ntiles, C4_THREADS, 0, st>>>(g, (unsigned)nwords, (uint32_t*)ctx->vbase.p,
                                                    (unsigned long long*)B.own_id.p, (uint32_t*)B.own_voff.p,
                                                    (unsigned long long*)B.cell_id.p, (uint32_t*)B.cell_toff.p, cap_own,
                                                    cap_cell, st_vt, dctr, ntiles);
    k4_tile_scan<<<1, 1024, 0, st>>>(st_vt, ntiles, tile_off, dctr);
    k4_fix_vbase<<<(unsigned)((nwords + 255) / 256), 256, 0, st>>>((uint32_t*)ctx->vbase.p, (unsigned)nwords, tile_off);
    ctx->launches += 3;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->counters_host, dctr, sizeof(Counters4), cudaMemcpyDeviceToHost, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    memcpy(&h, ctx->counters_host, sizeof h);
    totV = h.total_vt & 0x7fffffffull;
    totT = h.total_vt >> 31;
    nOwn = h.total_act & 0x7fffffffull;
    nCell = h.total_act >> 31;
    if (nOwn <= cap_own && nCell <= cap_cell) break;
    if (attempt == 2) return ctr_fail(ctx, CTR_ERR_STATE, "list capacity did not converge");
    want_own = std::max<size_t>(nOwn, want_own);
    want_cell = std::max<size_t>(nCell, want_cell);
  }
  ctr_stage_mark(ctx, 3);
  if (totV >= 0x7ffffff0ull || totT >= 0x7ffffff0ull)
    return ctr_fail(ctx, CTR_ERR_OVERFLOW, "more than 2^31 vertices or tetrahedra in one call; shard the field");
  out->n_verts = (int64_t)totV;
  out->n_tets = (int64_t)totT;
  out->n_active_cells = (int64_t)h.n_cells;
  out->n_crossings = (int64_t)h.n_cross;
  out->n_morph_tris = 0;
  const bool mm = (p->flags & CTR_WANT_MINMAX) && h.min_key != ~0ull;
  out->fmin = mm ? key_to_double(h.min_key) : NAN;
  out->fmax = mm ? key_to_double(h.max_key) : NAN;
  out->t_min = out->t_max = NAN;
  const bool f64 = (p->flags & CTR_GEOM_F64) != 0;
  const size_t gsz = f64 ? 8 : 4;
  if (!(p->flags & CTR_NO_GEOMETRY)) {
    if ((rc = ctr_ensure(ctx, B.verts, (size_t)totV * 4 * gsz + 16))) return rc;
    if ((rc = ctr_ensure(ctx, B.tets, (size_t)totT * 16 + 16))) return rc;
    if (p->flags & CTR_WANT_KEYS) {
      if ((rc = ctr_ensure(ctx, B.keys, (size_t)totV * 8 + 16))) return rc;
      if ((rc = ctr_ensure(ctx, B.lowmin, (size_t)totV + 16))) return rc;
    }
    if (p->flags & CTR_WANT_CODES)
      if ((rc = ctr_ensure(ctx, B.codes, (size_t)nCell * 24 + 16))) return rc;
    Xform4 xf;
    for (int a = 0; a < 4; ++a) {
      xf.origin[a] = p->origin[a];
      xf.delta[a] = p->delta[a];
    }
    unsigned long long* dkeys = (p->flags & CTR_WANT_KEYS) ? (unsigned long long*)B.keys.p : nullptr;
    uint8_t* dlow = (p->flags & CTR_WANT_KEYS) ? (uint8_t*)B.lowmin.p : nullptr;
    // morph stage inputs (grid coordinates, fp64: its thresholds are defined there) come out of the same kernel
    const bool morph = (p->flags & CTR_MORPH) && totV && totT;
    const double corner_t = (double)(n3 - 1);
    const double bin_width = corner_t * (1.0 / p->nbins);
    if (morph) {
      if ((rc = ctr_ensure(ctx, B.mverts, (size_t)totV * 32 + 16))) return rc;
      if ((rc = ctr_ensure(ctx, B.tbin, (size_t)totV * 4 + 16))) return rc;
      if ((rc = ctr_ensure(ctx, B.keep, (size_t)totT + 16))) return rc;
      MinMaxKeys mk0;                                  // t range of the binned vertices, filled by k4_emit_verts
      mk0.min_key = ~0ull;
      mk0.max_key = 0ull;
      memcpy(ctx->counters_host, &mk0, sizeof mk0);
      CTR_CUDA(ctx, cudaMemcpyAsync(dctr, ctx->counters_host, sizeof mk0, cudaMemcpyHostToDevice, st));
    }
    if (nOwn) {
      const int blocks = (int)((nOwn + 255) / 256);
      double* dmv = morph ? (double*)B.mverts.p : nullptr;
      int* dtb = morph ? (int*)B.tbin.p : nullptr;
      if (f64)
        k4_emit_verts<T, double><<<blocks, 256, 0, st>>>(g, (const unsigned long long*)B.own_id.p, (const uint32_t*)B.own_voff.p,
                                                         (unsigned)nOwn, xf, (double*)B.verts.p, dkeys, dlow, dmv, dtb, bin_width,
                                                         (MinMaxKeys*)dctr, tile_off);
      else
        k4_emit_verts<T, float><<<blocks, 256, 0, st>>>(g, (const unsigned long long*)B.own_id.p, (const uint32_t*)B.own_voff.p,
                                                        (unsigned)nOwn, xf, (float*)B.verts.p, dkeys, dlow, dmv, dtb, bin_width,
                                                        (MinMaxKeys*)dctr, tile_off);
      ctx->launches++;
    }
    ctr_stage_mark(ctx, 4);
    if (nCell) {
      const int blocks = (int)((nCell + E4_THREADS - 1) / E4_THREADS);
      k4_emit_tets<T><<<blocks, E4_THREADS, 0, st>>>(g, (const unsigned long long*)B.cell_id.p, (const uint32_t*)B.cell_toff.p,
                                                     (unsigned)nCell, (const uint32_t*)ctx->vbase.p, (int*)B.tets.p,
                                                     (p->flags & CTR_WANT_CODES) ? (uint8_t*)B.codes.p : nullptr, tile_off);
      ctx->launches++;
    }
    ctr_stage_mark(ctx, 5);
    // ---- morph stage
    if (morph) {
      MinMaxKeys mk;
      CTR_CUDA(ctx, cudaMemcpyAsync(ctx->counters_host, dctr, sizeof mk, cudaMemcpyDeviceToHost, st));
      CTR_CUDA(ctx, cudaStreamSynchronize(st));
      memcpy(&mk, ctx->counters_host, sizeof mk);
      const double tmin = key_to_double(mk.min_key), tmax = key_to_double(mk.max_key);
      out->t_min = tmin;
      out->t_max = tmax;
      MorphParams mp;
      const int nn[4] = {n0, n1, n2, n3};
      for (int a = 0; a < 4; ++a) mp.inv_corner[a] = 1.0 / (double)(nn[a] - 1);
      mp.eps_instant = 1e-7;
      mp.eps_tiny = 1e-3;
      mp.eps_gap = 1e-4;
      mp.eps_in = 1e-5;
      mp.t_eps = 1e-7 * (tmax - tmin);
      // integer bins decide exactly like the fp64 tolerances when the bin width dwarfs them (CTR_SLICE_FP64=1: never)
      const bool int_times = bin_width > 100.0 * std::max(mp.eps_gap, std::max(mp.eps_in, mp.t_eps)) &&
                             fabs(tmax) < 1.0e9 * bin_width && fabs(tmin) < 1.0e9 * bin_width && !getenv("CTR_SLICE_FP64");
      // ... and then the filter is a by-product of the slicing: vertices in different bins are >= one bin apart, which
      // is neither "instant" (1e-7) nor, with a bin wider than eps_tiny of the t axis, "tiny"; equal bins are instant
      const bool fused_filter = int_times && bin_width * mp.inv_corner[3] > 2.0 * mp.eps_tiny;
      if (!fused_filter) {
        k4_tet_filter<<<(int)((totT + 255) / 256), 256, 0, st>>>((const double*)B.mverts.p, (const int*)B.tets.p, (unsigned)totT,
                                                                 mp, (uint8_t*)B.keep.p);
        ctx->launches++;
      }
      const int sl_tiles = (int)((totT + SL_TILE - 1) / SL_TILE);
      if ((rc = ctr_ensure(ctx, B.slstate, (size_t)sl_tiles * 8 + 64 + 256 + 4096 * 8))) return rc;      // + the pattern table
      size_t want = std::max<size_t>((size_t)totT * 2, 1 << 14);
      unsigned long long nmt = 0;
      for (int attempt = 0; attempt < 3; ++attempt) {
        if ((rc = ctr_ensure(ctx, B.mtris, want * 24))) return rc;
        const unsigned cap = (unsigned)std::min<size_t>(B.mtris.cap / 24, 0x7fffffffu);
        CTR_CUDA(ctx, ctr_smem_optin(ctx, k4_slice<double>, SL_SMEM));
        CTR_CUDA(ctx, ctr_smem_optin(ctx, k4_slice<int>, SL_SMEM));
        SlCounters* slc = (SlCounters*)((char*)B.slstate.p + (size_t)sl_tiles * 8);
        unsigned long long* ptab = (unsigned long long*)((char*)B.slstate.p + (((size_t)sl_tiles * 8 + 64 + 255) & ~(size_t)255));
        CTR_CUDA(ctx, cudaMemsetAsync(B.slstate.p, 0, (size_t)sl_tiles * 8 + 32, st));
        if (int_times) {
          k4_slice_table<<<1, 256, 0, st>>>(ptab, mp);
          ctx->launches++;
        }
        if (int_times)
          k4_slice<int><<<sl_tiles, SL_THREADS, SL_SMEM, st>>>(
              (const double*)B.mverts.p, (const int*)B.tbin.p, (const int*)B.tets.p,
              fused_filter ? nullptr : (const uint8_t*)B.keep.p, fused_filter ? (uint8_t*)B.keep.p : nullptr, (unsigned)totT, mp,
              (unsigned long long*)B.slstate.p, slc, sl_tiles, (int*)B.mtris.p, cap, ptab);
        else
          k4_slice<double><<<sl_tiles, SL_THREADS, SL_SMEM, st>>>(
              (const double*)B.mverts.p, (const int*)B.tbin.p, (const int*)B.tets.p, (const uint8_t*)B.keep.p, nullptr,
              (unsigned)totT, mp, (unsigned long long*)B.slstate.p, slc, sl_tiles, (int*)B.mtris.p, cap, ptab);
        ctx->launches++;
        CTR_CUDA(ctx, cudaMemcpyAsync(ctx->counters_host, slc, sizeof(SlCounters), cudaMemcpyDeviceToHost, st));
        CTR_CUDA(ctx, cudaStreamSynchronize(st));
        SlCounters hs;
        memcpy(&hs, ctx->counters_host, sizeof hs);
        nmt = hs.total;
        if (nmt <= cap) break;
        if (attempt == 2) return ctr_fail(ctx, CTR_ERR_STATE, "morph triangle capacity did not converge");
        want = nmt;
      }
      out->n_morph_tris = (int64_t)nmt;
    }
    ctr_stage_mark(ctx, 6);
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  if (ctx->timing) {
    for (int s = 0; s < 6; ++s) {
      ctx->stage_ms[s] = 0.f;
      if (ctx->ev_set[s] && ctx->ev_set[s + 1]) cudaEventElapsedTime(&ctx->stage_ms[s], ctx->ev[s], ctx->ev[s + 1]);
    }
  }
  ctx->last_kind = 4;
  ctx->last_flags = p->flags;
  ctx->last_counts[0] = (int64_t)totV;
  ctx->last_counts[1] = (int64_t)totT;
  ctx->last_counts[2] = (p->flags & CTR_WANT_CODES) ? (int64_t)nCell : 0;
  ctx->last_counts[3] = out->n_morph_tris;
  out->n_codes = ctx->last_counts[2];
  return 0;
}

}  // namespace

extern "C" int ctr_mp4d_run(ctr_ctx* ctx, const ctr_mp4d_params* p, ctr_mp4d_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!p || !out || !p->field) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (p->n0 < 2 || p->n1 < 2 || p->n2 < 2 || p->n3 < 2) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "grid must have at least 2 samples per axis");
  if (!(p->isovalue == p->isovalue)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "isovalue is NaN");
  if ((p->flags & CTR_MORPH) && p->nbins < 1) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "nbins must be >= 1");
  for (int a = 0; a < 4; ++a)
    if (p->delta[a] == 0.0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "delta must be non-zero");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  memset(out, 0, sizeof *out);
  ctx->last_kind = 0;
  if (p->dtype == CTR_F32) return run4d<float>(ctx, p, out);
  if (p->dtype == CTR_F64) return run4d<double>(ctx, p, out);
  return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32 or CTR_F64");
}

extern "C" int ctr_mp4d_fetch(ctr_ctx* ctx, void* verts, int32_t* tets, uint64_t* keys, uint8_t* lowmin, uint8_t* codes,
                              int64_t* cells, double* morph_verts, uint8_t* keep, int32_t* morph_tris) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 4) return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mp4d_run to fetch from");
  if (ctx->last_flags & CTR_NO_GEOMETRY) return ctr_fail(ctx, CTR_ERR_STATE, "run had CTR_NO_GEOMETRY");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  Bufs4 B(ctx);
  const uint32_t fl = ctx->last_flags;
  const size_t gsz = (fl & CTR_GEOM_F64) ? 8 : 4;
  const size_t nV = (size_t)ctx->last_counts[0], nT = (size_t)ctx->last_counts[1], nC = (size_t)ctx->last_counts[2],
               nM = (size_t)ctx->last_counts[3];
  cudaStream_t st = ctx->stream;
  if (verts && nV) CTR_CUDA(ctx, cudaMemcpyAsync(verts, B.verts.p, nV * 4 * gsz, cudaMemcpyDeviceToHost, st));
  if (tets && nT) CTR_CUDA(ctx, cudaMemcpyAsync(tets, B.tets.p, nT * 16, cudaMemcpyDeviceToHost, st));
  if (keys || lowmin) {
    if (!(fl & CTR_WANT_KEYS)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not compute keys");
    if (keys && nV) CTR_CUDA(ctx, cudaMemcpyAsync(keys, B.keys.p, nV * 8, cudaMemcpyDeviceToHost, st));
    if (lowmin && nV) CTR_CUDA(ctx, cudaMemcpyAsync(lowmin, B.lowmin.p, nV, cudaMemcpyDeviceToHost, st));
  }
  if (codes || cells) {
    if (!(fl & CTR_WANT_CODES)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not compute case codes");
    if (codes && nC) CTR_CUDA(ctx, cudaMemcpyAsync(codes, B.codes.p, nC * 24, cudaMemcpyDeviceToHost, st));
    if (cells && nC) CTR_CUDA(ctx, cudaMemcpyAsync(cells, B.cell_id.p, nC * 8, cudaMemcpyDeviceToHost, st));
  }
  if (morph_verts || keep || morph_tris) {
    if (!(fl & CTR_MORPH)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not include the morph stage");
    if (morph_verts && nV) CTR_CUDA(ctx, cudaMemcpyAsync(morph_verts, B.mverts.p, nV * 32, cudaMemcpyDeviceToHost, st));
    if (keep && nT) CTR_CUDA(ctx, cudaMemcpyAsync(keep, B.keep.p, nT, cudaMemcpyDeviceToHost, st));
    if (morph_tris && nM) CTR_CUDA(ctx, cudaMemcpyAsync(morph_tris, B.mtris.p, nM * 24, cudaMemcpyDeviceToHost, st));
  }
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}
