// 3D marching tetrahedra on sm_100a -- bitplane-first design (DESIGN.md sections 3-4).
//
//   k_reset3     : counters, row flags, tile aggregates.
//   k_bitplane   : stream the scalar field ONCE (the only pass that touches all of it; TMA bulk copies into a shared
//                  memory ring, bitplane.cuh), write two bitplanes (1 bit/sample each): low = f < v
//                  (tetrahedral.py:572) and near = conservative hull of the two np.allclose tests
//                  (tetrahedral.py:391,576); min/max (grid_field.py:79-80).
//   k_count_a/_b : from the bitplanes (L2 resident), per 32-sample word: used-edge words of the 7 Kuhn directions,
//                  per-tet words, vertex / triangle counts (the scan records), per-direction vertex prefix (dirpack),
//                  strict crossings (grid_field.py:81) -- and, in the same visit, the work lists of stages 3 / 4
//                  (owner points, emitting voxels) into slots handed out by atomic counters; tile aggregates, scanned
//                  by the last block.
//   k_scan       : records -> vbase[word] (first vertex id), tbase[word] (first triangle).
//   k_emit_verts : thread per owner point, its 1..7 edges dealt out over the warp: crossings
//                  (tetrahedral.py:471-487), gradient normals, world transform (grid_field.py:89-93); vertex id =
//                  vbase[word] + dirbase + rank (the reference's dict dedup, tetrahedral.py:184-188, as a perfect hash).
//   k_emit_tris  : thread per emitting voxel: 6 Kuhn tets (tetrahedral.py:32-39,554-595) -> triangles of vertex ids,
//                  wound so the normal points to the high side.
//   k_codes      : optional parity output: (voxel, 30-bit case code) recomputed from the raw samples.
//
// Exactness: voxels / tets / edges whose outcome could depend on an np.allclose test are detected from the
// near bitplane and re-evaluated from the samples in fp64 (cell_emit_exact / edge_used_exact); everything
// else is decided by bit logic.  There is no CPU fallback anywhere.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "bitplane.cuh"
#include "tables.h"
#include "uf_hash.cuh"

namespace {

__constant__ uint8_t c_tetmask[8][8];
__constant__ uint8_t c_tet[6][4];
__constant__ unsigned short c_vox[256];   // corner bits -> emitting tets (6 bits) | triangle count << 8

struct Counters {                    // device counter block (mirrored to pinned host memory)
  // stage 1 (bitplane)
  unsigned long long min_key;        // order-preserving encoding of fmin
  unsigned long long max_key;        // order-preserving encoding of fmax
  unsigned int any_near;
  unsigned int pad0;
  // stage 2 (count + scan): zeroed before every launch
  unsigned long long n_cells;        // emitting voxels
  unsigned long long n_cross;        // strict crossings
  unsigned long long total_vt;       // packed totals over the scanned range: T << 31 | V
  unsigned long long v_emit;         // vertex count at the start of plane i_hi (vertices this call emits)
  unsigned int ticket;
  unsigned long long tot_v, tot_t;   // the same totals, accumulated unpacked (a vertex total >= 2^31 would carry into T above)
  // every tile of k_count_a adds to each of these three: one 128-byte line each, so that the atomics of different
  // counters go to different L2 slices instead of queueing behind one address line
  alignas(128) unsigned int n_word;  // interesting words listed by k_count_a
  alignas(128) unsigned int n_own;   // slots handed out in the owner / voxel work lists (their lengths at the end)
  alignas(128) unsigned int n_cell;
};


template <typename T>
struct Grid {
  const T* f;
  const uint32_t* bits;
  const uint32_t* nbits;
  int n0, n1, n2, W;
  int i_lo, i_hi, i_hiv;             // emit planes [i_lo, i_hi); scanned owner planes [i_lo, i_hiv)
  long long plane_offset;
  unsigned id_base;                  // added to every vertex id written into the triangles
  double v;                          // isovalue
  double tolv;                       // 1e-8 + 1e-5*|v|
  // allclose handling is local: rowflag[i*n1+j] != 0 iff some sample of rows (i..i+2, j..j+2) lies inside the
  // conservative allclose hull; kernels copy it into any_near before touching a word of row (i, j).
  int any_near;
  const uint8_t* rowflag;
  // per row, one bit per group of 2^wshift words (a group = one word up to 1024 samples per row):
  //   wordflag  : some near sample within rows +-2 and words w-1..w+1 (stage 1) -> stage 2 looks at the near plane;
  //   exactflag : the exact used-edge words of some word among rows (i..i+1, j..j+1) of this group differ from the
  //               plain crossing words (stage 2) -> stage 4 recomputes them exactly.  Practically never set.
  const uint32_t* wordflag;
  uint32_t* exactflag;
  int wshift;
  __device__ __forceinline__ int near_word(unsigned row, unsigned w) const { return (int)((wordflag[row] >> (w >> wshift)) & 1u); }
  __device__ __forceinline__ int exact_word(unsigned row, unsigned w) const { return (int)((exactflag[row] >> (w >> wshift)) & 1u); }
  FastDiv divW, divN1;
  __device__ __forceinline__ void word_coords(unsigned gw, int& i, int& j, int& w) const {
    unsigned row = divW.div(gw);
    w = (int)(gw - row * (unsigned)W);
    unsigned ii = divN1.div(row);
    i = (int)ii;
    j = (int)(row - ii * (unsigned)n1);
  }
};


// ------------------------------------------------------------------------------------------------
// Exact (fp64) evaluation from the samples -- only for voxels/edges flagged by the near bitplane.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool near_a(double f, double v) {   // np.allclose(value, f): tetrahedral.py:391
  return fabs(v - f) <= __dadd_rn(1e-8, __dmul_rn(1e-5, fabs(f)));
}

template <typename T>
__device__ __forceinline__ double sample(const Grid<T>& g, int i, int j, int k) {
  return (double)g.f[((long long)i * g.n1 + j) * g.n2 + k];
}

// 6-bit mask of the tets of voxel (i,j,k) that emit triangles; also returns the 30-bit case code.
template <typename T>
__device__ __noinline__ unsigned cell_emit_exact(const Grid<T> g, int i, int j, int k, unsigned* code_out) {
  if (code_out) *code_out = 0;
  if (i < 0 || j < 0 || k < 0 || i >= g.n0 - 1 || j >= g.n1 - 1 || k >= g.n2 - 1) return 0;
  double fv[8];
  bool all_a = true;
  unsigned low = 0, nb = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    fv[c] = sample(g, i + ((c >> 2) & 1), j + ((c >> 1) & 1), k + (c & 1));
    all_a = all_a && near_a(fv[c], g.v);
    low |= (fv[c] < g.v ? 1u : 0u) << c;
    nb |= (fabs(fv[c] - g.v) <= g.tolv ? 1u : 0u) << c;       // np.allclose(values, value): tetrahedral.py:576
  }
  unsigned emit = 0, code = 0;
#pragma unroll
  for (int t = 0; t < 6; ++t) {
    unsigned m = 0, alln = 1;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      int c = c_tet[t][b];
      m |= ((low >> c) & 1u) << b;
      alln &= (nb >> c) & 1u;
    }
    code |= (m | (alln << 4)) << (5 * t);
    if (m != 0 && m != 15 && !alln) emit |= 1u << t;
  }
  if (code_out) *code_out = code;
  // border_voxel (tetrahedral.py:391-394): the min<=v<=max half is implied by any crossing tet
  return all_a ? 0u : emit;
}

// Is the crossing edge p -> p+d used by any emitted triangle?  (OR over the voxels / tets that contain it.)
template <typename T>
__device__ __noinline__ bool edge_used_exact(const Grid<T> g, int i, int j, int k, int d) {
  for (int s = 0; s < 8; ++s) {
    if (s & d) continue;
    unsigned tm = c_tetmask[d][s];
    if (!tm) continue;
    unsigned e = cell_emit_exact(g, i - ((s >> 2) & 1), j - ((s >> 1) & 1), k - (s & 1), nullptr);
    if (e & tm) return true;
  }
  return false;
}

// ------------------------------------------------------------------------------------------------
// Bit-sliced neighbourhood of one word: rows (i+a, j+b), a,b in {0,1}; P = bits at k, S = bits at k+1.
// ------------------------------------------------------------------------------------------------
struct Planes {
  uint32_t P[4];    // index a*2+b
  uint32_t S[4];
  uint32_t kpt;     // bits with k < n2
  uint32_t kp1;     // bits with k+1 < n2
  bool has_i1, has_j1;
};

__device__ __forceinline__ uint32_t low_mask(int n) {   // n lowest bits set, n in [0,32]
  return n >= 32 ? 0xffffffffu : ((1u << n) - 1u);
}

template <typename T>
__device__ __forceinline__ void load_planes(const Grid<T>& g, const uint32_t* __restrict__ plane, int i, int j, int w,
                                            Planes& pl) {
  pl.has_i1 = (i + 1 < g.n0);
  pl.has_j1 = (j + 1 < g.n1);
  int rem = g.n2 - w * 32;                   // samples from this word's first bit to the end of the row
  pl.kpt = low_mask(rem < 0 ? 0 : rem);
  pl.kp1 = low_mask(rem - 1 < 0 ? 0 : rem - 1);
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      bool ok = (a == 0 || pl.has_i1) && (b == 0 || pl.has_j1);
      uint32_t p = 0, nx = 0;
      if (ok) {
        const unsigned base = ((unsigned)(i + a) * (unsigned)g.n1 + (unsigned)(j + b)) * (unsigned)g.W + (unsigned)w;
        p = plane[base];
        if (w + 1 < g.W) nx = plane[base + 1];
      }
      pl.P[a * 2 + b] = p;
      pl.S[a * 2 + b] = (p >> 1) | (nx << 31);
    }
}

// crossing words for the 7 edge directions of the owner row (index d-1), masked to edges inside the grid
__device__ __forceinline__ void cross_words(const Planes& pl, uint32_t x[7]) {
  uint32_t A = pl.P[0];
  uint32_t vj = pl.has_j1 ? 0xffffffffu : 0u, vi = pl.has_i1 ? 0xffffffffu : 0u;
  x[0] = (A ^ pl.S[0]) & pl.kp1;                 // d=1 (0,0,1)
  x[1] = (A ^ pl.P[1]) & pl.kpt & vj;            // d=2 (0,1,0)
  x[2] = (A ^ pl.S[1]) & pl.kp1 & vj;            // d=3 (0,1,1)
  x[3] = (A ^ pl.P[2]) & pl.kpt & vi;            // d=4 (1,0,0)
  x[4] = (A ^ pl.S[2]) & pl.kp1 & vi;            // d=5 (1,0,1)
  x[5] = (A ^ pl.P[3]) & pl.kpt & vi & vj;       // d=6 (1,1,0)
  x[6] = (A ^ pl.S[3]) & pl.kp1 & vi & vj;       // d=7 (1,1,1)
}

// the "other endpoint" plane for direction d (1..7) out of a Planes
__device__ __forceinline__ uint32_t dir_plane(const Planes& pl, int d) {
  int ab = d >> 1;
  return (d & 1) ? pl.S[ab] : pl.P[ab];
}

// corner planes of the voxel row: corner c = a*4+b*2+dk
__device__ __forceinline__ uint32_t corner_plane(const Planes& pl, int c) {
  return (c & 1) ? pl.S[c >> 1] : pl.P[c >> 1];
}

// Per-tet words: odd = 1-3 split (1 triangle), two = 2-2 split (2 triangles); cand = crossing & all four near.
__device__ __forceinline__ void tet_words(const Planes& pl, const Planes* npl, uint32_t cellmask, uint32_t odd[6],
                                          uint32_t two[6], uint32_t& cand) {
  const uint32_t A = pl.P[0], H = pl.S[3];
  const int xs[6] = {1, 3, 2, 6, 4, 5};          // tets [A,H,x,y]: (B,D),(D,C),(C,G),(G,E),(E,F),(F,B)
  const int ys[6] = {3, 2, 6, 4, 5, 1};
  cand = 0;
#pragma unroll
  for (int t = 0; t < 6; ++t) {
    uint32_t X = corner_plane(pl, xs[t]), Y = corner_plane(pl, ys[t]);
    uint32_t par = A ^ H ^ X ^ Y;
    uint32_t dif = (A ^ H) | (A ^ X) | (A ^ Y);
    odd[t] = par & cellmask;
    two[t] = ~par & dif & cellmask;
    if (npl) {
      uint32_t nn = npl->P[0] & npl->S[3] & corner_plane(*npl, xs[t]) & corner_plane(*npl, ys[t]);
      cand |= nn & dif & cellmask;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// used-edge words of an owner word (index d-1), allclose-ambiguous edges resolved exactly (serial, rare)
// ------------------------------------------------------------------------------------------------
// The out-of-line exact paths take and return their data BY VALUE: a reference or pointer to a kernel's registers
// (the grid descriptor, the bit planes, the used-edge words) would pin those to local memory for the whole kernel --
// measured: 1.9 M local-memory wave-fronts per extraction in k_emit_tris, 1.6 M in k_count_b, on paths that never run.
struct W7 {
  uint32_t x[7];
};

template <typename T>
__device__ __noinline__ W7 resolve_used_exact(const Grid<T> g, int i, int j, int w, W7 in) {
  uint32_t used[7];
#pragma unroll
  for (int d = 0; d < 7; ++d) used[d] = in.x[d];
  Planes npl;
  load_planes(g, g.nbits, i, j, w, npl);
  for (int d = 1; d <= 7; ++d) {
    uint32_t c = used[d - 1] & npl.P[0] & dir_plane(npl, d);
    while (c) {
      int b = __ffs(c) - 1;
      c &= c - 1;
      if (!edge_used_exact(g, i, j, w * 32 + b, d)) used[d - 1] &= ~(1u << b);
    }
  }
  W7 out;
#pragma unroll
  for (int d = 0; d < 7; ++d) out.x[d] = used[d];
  return out;
}

template <typename T>
__device__ __forceinline__ void owner_used(const Grid<T>& g, const Planes& pl, int i, int j, int w, uint32_t used[7]) {
  cross_words(pl, used);
  if (g.any_near) {
    W7 in;
#pragma unroll
    for (int d = 0; d < 7; ++d) in.x[d] = used[d];
    const W7 out = resolve_used_exact(g, i, j, w, in);
#pragma unroll
    for (int d = 0; d < 7; ++d) used[d] = out.x[d];
  }
}

__device__ __forceinline__ unsigned gather7(const uint32_t u[7], int b) {
  unsigned m = 0;
#pragma unroll
  for (int d = 0; d < 7; ++d) m |= ((u[d] >> b) & 1u) << d;
  return m;
}

__device__ __forceinline__ unsigned tet_mask_of(unsigned corner8, int t) {
  // tets [A,H,x,y] with (x,y) = (B,D),(D,C),(C,G),(G,E),(E,F),(F,B)  (tetrahedral.py:32-39)
  const int xs[6] = {1, 3, 2, 6, 4, 5};
  const int ys[6] = {3, 2, 6, 4, 5, 1};
  return (corner8 & 1u) | (((corner8 >> 7) & 1u) << 1) | (((corner8 >> xs[t]) & 1u) << 2) | (((corner8 >> ys[t]) & 1u) << 3);
}

// strict-crossing correction and exact tet counts of one word: the rare, allclose-dependent part of stage 2
struct WordExact {
  unsigned ncross, ntri;
  uint32_t emitting;
};

template <typename T>
__device__ __noinline__ WordExact count_word_exact(const Grid<T> g, const Planes pl, int i, int j, int w, bool cells_ok,
                                                   WordExact in) {
  unsigned ncross = in.ncross, ntri = in.ntri;
  uint32_t emitting = in.emitting;
  Planes npl;
  load_planes(g, g.nbits, i, j, w, npl);
  if (cells_ok) {
    uint32_t xs[7];
    cross_words(pl, xs);
    for (int d = 1; d <= 7; ++d) {
      // not strict when the HIGH endpoint equals the isovalue exactly (then (f0-v)*(f1-v) == 0)
      uint32_t A = pl.P[0], O = dir_plane(pl, d);
      uint32_t c = xs[d - 1] & pl.kp1 & ((~A & npl.P[0]) | (~O & dir_plane(npl, d)));
      while (c) {
        int b = __ffs(c) - 1;
        c &= c - 1;
        bool a_high = !((A >> b) & 1u);
        int k = w * 32 + b;
        double fh = a_high ? sample(g, i, j, k) : sample(g, i + ((d >> 2) & 1), j + ((d >> 1) & 1), k + (d & 1));
        if (fh == g.v) --ncross;
      }
    }
    uint32_t odd[6], two[6], cand;
    tet_words(pl, &npl, pl.kp1, odd, two, cand);
    while (cand) {
      int b = __ffs(cand) - 1;
      cand &= cand - 1;
      // remove the fast-path contribution of this voxel, add the exact one
      for (int q = 0; q < 6; ++q) ntri -= ((odd[q] >> b) & 1u) + 2u * ((two[q] >> b) & 1u);
      emitting &= ~(1u << b);
      unsigned e = cell_emit_exact(g, i, j, w * 32 + b, nullptr);
      if (e) emitting |= 1u << b;
      for (int q = 0; q < 6; ++q)
        if ((e >> q) & 1u) ntri += ((odd[q] >> b) & 1u) ? 1u : 2u;
    }
  }
  WordExact out;
  out.ncross = ncross;
  out.ntri = ntri;
  out.emitting = emitting;
  return out;
}

// ------------------------------------------------------------------------------------------------
// Stage 2: per-word counts from the bitplanes + fused single-pass decoupled-lookback scan.
//   A  every thread tests 4 words of the tile (does anything cross here?) and the block compacts the
//      interesting ones in shared memory;
//   B  interesting words are dealt out evenly: vertex / triangle / owner / voxel counts per word;
//   C  block scan + decoupled look-back across tiles -> exclusive offsets per word;
//   D  interesting words again: write vbase and the compacted, ordered lists of
//        active owners (16-byte entries: word<<13 | bit<<8 | p_low<<7 | mask7, and the 7 x 5-bit ranks)
//        active voxels (cell_id = word<<28 | first triangle<<19 | bit<<14 | emit6<<8 | corner8).
// ------------------------------------------------------------------------------------------------
constexpr int CS_THREADS = 256;
constexpr int CS_ITEMS = 4;
constexpr int CS_TILE = CS_THREADS * CS_ITEMS;

// Vertex order inside a word: direction-major, then bit (k).  dirpack byte q-1 (q = 1..6) = number of used edges of
// the word in the directions before direction index q (index = d-1); id = vbase[word] + dirbase(q) + rank of the bit
// among the used edges of that direction.  Kept as two 32-bit halves so that every extraction is a 32-bit shift.
__device__ __forceinline__ uint2 dir_pack(const uint32_t x[7]) {
  unsigned c = 0;
  uint2 dp = make_uint2(0u, 0u);
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    c += __popc(x[q]);
    if (q < 4) dp.x |= c << (8 * q);
    else dp.y |= c << (8 * (q - 4));
  }
  return dp;
}
__device__ __forceinline__ unsigned dir_base(uint2 dp, int q) {   // q = d-1 in 0..6, compile-time constant when unrolled
  return q == 0 ? 0u : q <= 4 ? (dp.x >> (8 * (q - 1))) & 255u : (dp.y >> (8 * (q - 5))) & 255u;
}

// Quick test of 4 consecutive words of one row (W % 4 == 0, gw % 4 == 0): does any of their 7 x 32 owned edges cross?
// 128-bit loads of the four rows the words touch; returns a 4-bit mask.
// The quick test of stage 2a for words gw .. gw+3 of one row (gw a multiple of 4, W a multiple of 4): bit q of the
// result = word gw+q owns a crossing edge.  For such a word byte q of own4 / cell4 is the number of its owner points
// (points with a crossing owned edge, planes below i_hi) and of its emitting voxels (corner bits not all equal) by the
// plain bit logic -- the slots the word needs in the two work lists.  A word under a near flag gets none here: its
// exact counts may be smaller, k_count_b takes its slots itself.
template <typename T>
__device__ __forceinline__ unsigned words4_interesting(const Grid<T>& g, unsigned gw, unsigned plane_words, unsigned& own4,
                                                       unsigned& cell4) {
  const unsigned row = g.divW.div(gw);
  const unsigned w = gw - row * (unsigned)g.W;
  const unsigned i = g.divN1.div(row);
  const unsigned j = row - i * (unsigned)g.n1;
  const bool hi = (int)i + 1 < g.n0, hj = (int)j + 1 < g.n1, hw = (int)w + 4 < g.W;
  const uint32_t* p = g.bits + gw;
  uint32_t a[5], b[5] = {0, 0, 0, 0, 0}, c[5] = {0, 0, 0, 0, 0}, d[5] = {0, 0, 0, 0, 0};
  {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
    a[4] = hw ? p[4] : 0u;
  }
  if (hj) {
    const uint4 v = *reinterpret_cast<const uint4*>(p + g.W);
    b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
    b[4] = hw ? p[g.W + 4] : 0u;
  }
  if (hi) {
    const uint4 v = *reinterpret_cast<const uint4*>(p + plane_words);
    c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
    c[4] = hw ? p[plane_words + 4] : 0u;
    if (hj) {
      const uint4 u = *reinterpret_cast<const uint4*>(p + plane_words + g.W);
      d[0] = u.x; d[1] = u.y; d[2] = u.z; d[3] = u.w;
      d[4] = hw ? p[plane_words + g.W + 4] : 0u;
    }
  }
  const uint32_t mj = hj ? 0xffffffffu : 0u, mi = hi ? 0xffffffffu : 0u, mij = mi & mj;
  unsigned out = 0;
  uint32_t any[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int rem = g.n2 - (int)(w + q) * 32;
    const uint32_t kpt = low_mask(rem), kp1 = low_mask(rem - 1);
    const uint32_t A = a[q];
    const uint32_t t = ((A ^ b[q]) & mj) | ((A ^ c[q]) & mi) | ((A ^ d[q]) & mij);
    const uint32_t u = (A ^ __funnelshift_r(a[q], a[q + 1], 1)) | ((A ^ __funnelshift_r(b[q], b[q + 1], 1)) & mj) |
                       ((A ^ __funnelshift_r(c[q], c[q + 1], 1)) & mi) | ((A ^ __funnelshift_r(d[q], d[q + 1], 1)) & mij);
    any[q] = (t & kpt) | (u & kp1);                     // OR of the seven crossing words (cross_words)
    if (any[q] != 0) out |= 1u << q;
  }
  own4 = cell4 = 0;
  if (out && (int)i < g.i_hi) {                         // planes from i_hi on are scanned for their vertex ids only
    const uint32_t nf = g.wordflag[row];
    if (nf) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if ((nf >> ((w + q) >> g.wshift)) & 1u) any[q] = 0u;
    }
    own4 = (unsigned)__popc(any[0]) | ((unsigned)__popc(any[1]) << 8) | ((unsigned)__popc(any[2]) << 16) | ((unsigned)__popc(any[3]) << 24);
    // voxels: the same points, except the row's last sample (k + 1 == n2), which can only sit in the row's last word
    if (hi && hj) cell4 = own4 - (hw ? 0u : (unsigned)__popc(any[3] & ~low_mask(g.n2 - (int)(w + 3) * 32 - 1)) << 24);
  }
  return out;
}

// the same for one word of any grid (rows whose word count is no multiple of 4)
template <typename T>
__device__ __forceinline__ bool word_interesting(const Grid<T>& g, unsigned gw, unsigned& own, unsigned& cell) {
  int i, j, w;
  g.word_coords(gw, i, j, w);
  Planes pl;
  load_planes(g, g.bits, i, j, w, pl);
  uint32_t x[7];
  cross_words(pl, x);
  const uint32_t any = x[0] | x[1] | x[2] | x[3] | x[4] | x[5] | x[6];
  own = cell = 0;
  if (any && i < g.i_hi && !g.near_word((unsigned)i * (unsigned)g.n1 + (unsigned)j, (unsigned)w)) {
    own = (unsigned)__popc(any);
    if (pl.has_i1 && pl.has_j1) cell = (unsigned)__popc(any & pl.kp1);
  }
  return any != 0;
}

// per-word record of the scan: vertices | triangles << 8
__device__ __forceinline__ unsigned long long rec_vt(uint32_t r) {
  return ((unsigned long long)(r >> 8) << 31) | (r & 255u);
}

// ------------------------------------------------------------------------------------------------
// Stage 2a: counts and work lists, in two kernels whose threads are all busy.
//   k_count_a : every word: 128-bit quick test, record zeroed, interesting words appended to a global list (one atomic
//               per tile; the list is ordered inside a tile's chunk);
//   k_count_b : one interesting word per thread, dense: counts, dirpack, owner / voxel work lists (slots: one block
//               scan and one atomicAdd per list and block), record, tile aggregate by atomicAdd;
//   k_tile_scan3 : one block: tile aggregates -> exclusive tile prefixes.
// (As ONE kernel per tile of 1024 words -- quick test, then the ~70 interesting words of the tile one per thread -- three
// quarters of every block idled through the second phase and every tile paid the latency chain planes -> counts -> two
// global atomics -> list writes on its own: 133 us against 17 + 104 us for the pair, measured under ncu.)
// Owner entries (16 bytes):  .x = word<<13 | bit<<8 | p_low<<7 | mask7, .y = 7 x 5-bit ranks within the directions.
// Voxel entries (8 bytes):  word<<28 | toff<<19 | bit<<14 | emit6<<8 | corner8, toff (9 bits, <= 31 x 12) = first triangle
// RELATIVE to tbase[word].  One store per entry in k_count_b, one load per entry in stages 3 / 4.
// Neither needs the scan: vertex ids are vbase[word] + dirbase + rank, triangle offsets tbase[word] + relative.
// The lists are ordered inside a block and unordered across blocks; the mesh does not depend on their order.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(CS_THREADS) k_count_a(Grid<T> g, unsigned word0, unsigned nwords_scan,
                                                     uint32_t* __restrict__ wlist, uint2* __restrict__ wslot,
                                                     uint2* __restrict__ tile_chunk, unsigned cap_w, Counters* ctr) {
  // the tile's interesting words in ascending word order, each with the first slot of its owner points and of its
  // emitting voxels in the work lists: one block prefix over (words, owner points, voxels) and three atomics per tile
  __shared__ unsigned long long s_warp[CS_THREADS / 32];
  __shared__ unsigned s_base[3];
  __shared__ unsigned short s_list[CS_TILE];
  __shared__ unsigned s_slot[CS_TILE];                 // tile-relative (owner slot | voxel slot << 16) of a listed word
  ctr_pdl_enter();
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned plane_words = (unsigned)g.n1 * (unsigned)g.W;
  const unsigned rel = blockIdx.x * CS_TILE + threadIdx.x * CS_ITEMS;      // this thread's four consecutive words
  unsigned m4 = 0, own4 = 0, cell4 = 0;
  if ((g.W & 3) == 0) {
    if (rel < nwords_scan) m4 = words4_interesting(g, word0 + rel, plane_words, own4, cell4);
  } else {
#pragma unroll
    for (int q = 0; q < CS_ITEMS; ++q) {
      unsigned o = 0, c = 0;
      if (rel + q < nwords_scan && word_interesting(g, word0 + rel + q, o, c)) m4 |= 1u << q;
      own4 |= o << (8 * q);
      cell4 |= c << (8 * q);
    }
  }
  // byte sums: a word has at most 32 owner points / 31 voxels, four words stay below 256
  const unsigned own_n = (own4 * 0x01010101u) >> 24, cell_n = (cell4 * 0x01010101u) >> 24;
  const unsigned long long mine = (unsigned long long)__popc(m4) | ((unsigned long long)own_n << 16) | ((unsigned long long)cell_n << 32);
  const unsigned long long inc = warp_incl_scan_u64(mine);
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  unsigned long long before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < CS_THREADS / 32; ++w) {
    const unsigned long long c = s_warp[w];
    if (w < (int)warp) before += c;
    total += c;
  }
  const unsigned nint = (unsigned)total & 0xffffu, n_own = (unsigned)(total >> 16) & 0xffffu, n_cell = (unsigned)(total >> 32);
  if (threadIdx.x == 0) {                              // three warps, one atomic each: the round trips overlap
    const unsigned b0 = nint ? atomicAdd(&ctr->n_word, nint) : 0u;
    s_base[0] = b0;
    tile_chunk[blockIdx.x] = make_uint2(b0, nint);
  } else if (threadIdx.x == 32) {
    s_base[1] = n_own ? atomicAdd(&ctr->n_own, n_own) : 0u;
  } else if (threadIdx.x == 64) {
    s_base[2] = n_cell ? atomicAdd(&ctr->n_cell, n_cell) : 0u;
  }
  if (!nint) return;
  {
    const unsigned long long ex = before + inc - mine;
    unsigned base = (unsigned)ex & 0xffffu, orun = (unsigned)(ex >> 16) & 0xffffu, crun = (unsigned)(ex >> 32);
#pragma unroll
    for (int q = 0; q < CS_ITEMS; ++q)
      if ((m4 >> q) & 1u) {
        s_list[base] = (unsigned short)(threadIdx.x * CS_ITEMS + q);
        s_slot[base] = orun | (crun << 16);
        ++base;
        orun += (own4 >> (8 * q)) & 255u;
        crun += (cell4 >> (8 * q)) & 255u;
      }
  }
  __syncthreads();
  const unsigned b0 = s_base[0], o0 = s_base[1], c0 = s_base[2];
  for (unsigned q = threadIdx.x; q < nint; q += CS_THREADS)
    if (b0 + q < cap_w) {
      wlist[b0 + q] = word0 + blockIdx.x * CS_TILE + s_list[q];
      const unsigned sl = s_slot[q];
      wslot[b0 + q] = make_uint2(o0 + (sl & 0xffffu), c0 + (sl >> 16));
    }
}

// The word flag of stage 1 is dilated; every exact path of stage 2 starts from the near bits of the eight words a word
// touches, so without any of those the plain bit logic is already exact.
template <typename T>
__device__ __noinline__ int near_bits_around(const Grid<T> g, int i, int j, int w, uint32_t kpt) {
  Planes npl;
  load_planes(g, g.nbits, i, j, w, npl);
  return ((npl.P[0] | npl.P[1] | npl.P[2] | npl.P[3] | npl.S[0] | npl.S[1] | npl.S[2] | npl.S[3]) & kpt) != 0u;
}

// Exact used-edge words that differ from the crossing words: stage 4 ranks the edges of rows (i..i+1, j..j+1) by these
// words, so the voxel rows that read this one are told to recompute them exactly.
template <typename T>
__device__ __noinline__ void flag_exact_words(const Grid<T> g, const Planes pl, int i, int j, int w, const W7 x7) {
  const uint32_t* x = x7.x;
  uint32_t xs[7];
  cross_words(pl, xs);
  uint32_t dif = 0;
#pragma unroll
  for (int d = 0; d < 7; ++d) dif |= xs[d] ^ x[d];
  if (!dif) return;
  const uint32_t m = 1u << ((unsigned)w >> g.wshift);
  for (int di = 0; di < 2; ++di)
    for (int dj = 0; dj < 2; ++dj)
      if (i - di >= 0 && j - dj >= 0) atomicOr(&g.exactflag[(size_t)(i - di) * g.n1 + (j - dj)], m);
}

#ifndef CTR_CB_THREADS
#define CTR_CB_THREADS 128          // without the slot barrier the block size is free: 128 x 5 blocks: stage 2 110.7 -> 106.5 us
#endif
constexpr int CB_THREADS = CTR_CB_THREADS;

struct CountBShared {
  unsigned long long spread[128];     // 7-bit direction mask -> 7 x 5-bit fields with a one where the mask has a bit
  unsigned short vox[256];
};

#ifndef CTR_CB_MINB
#define CTR_CB_MINB 5          // 96 registers (128 threads x 6 -> 80: 108.3 us; x 4 -> 128: 109.2; 64 threads x 10: 107.8)
#endif
template <typename T>
__global__ void __launch_bounds__(CB_THREADS, CTR_CB_MINB) k_count_b(Grid<T> gin, unsigned word0, const uint32_t* __restrict__ wlist,
                                                        const uint2* __restrict__ wslot,
                                                        unsigned cap_w, uint32_t* __restrict__ recc, uint4* __restrict__ wrec,
                                                        ulonglong2* __restrict__ own,
                                                        unsigned long long* __restrict__ cell_id,
                                                        unsigned cap_own, unsigned cap_cell,
                                                        unsigned long long* __restrict__ tile_vt, Counters* ctr, int ntiles) {
  __shared__ CountBShared sh;
  Grid<T> g = gin;
  g.any_near = 0;
  for (unsigned q = threadIdx.x; q < 256u; q += CB_THREADS) sh.vox[q] = c_vox[q];
  for (unsigned q = threadIdx.x; q < 128u; q += CB_THREADS) {
    unsigned long long sp = 0;
#pragma unroll
    for (int d = 0; d < 7; ++d) sp |= (unsigned long long)((q >> d) & 1u) << (5 * d);
    sh.spread[q] = sp;
  }
  __syncthreads();
  ctr_pdl_enter();                                     // the tables above come from constants: filled while k_count_a drains
  const unsigned lane = lane_id();
  const unsigned plane_words = (unsigned)g.n1 * (unsigned)g.W;
  const unsigned emit_end = (unsigned)g.i_hi * plane_words;
  const unsigned nint = min(ctr->n_word, cap_w);
  const unsigned idx = blockIdx.x * CB_THREADS + threadIdx.x;
  const bool have = idx < nint;
  unsigned ncross = 0, ncells = 0;
  unsigned gw = 0;
  int i = 0, j = 0, w = 0;
  Planes pl;
  uint32_t x[7] = {0, 0, 0, 0, 0, 0, 0};
  uint32_t any = 0, em = 0;
  uint2 slot = make_uint2(0u, 0u);
  bool flagged = false;
  uint32_t r = 0;
  if (have) {
    gw = wlist[idx];
    slot = wslot[idx];
    g.word_coords(gw, i, j, w);
    g.any_near = g.near_word((unsigned)i * (unsigned)g.n1 + (unsigned)j, (unsigned)w);
    flagged = g.any_near != 0;
    load_planes(g, g.bits, i, j, w, pl);
    if (g.any_near) g.any_near = near_bits_around(g, i, j, w, pl.kpt);
    owner_used(g, pl, i, j, w, x);
    if (g.any_near) {
      W7 x7;
#pragma unroll
      for (int d = 0; d < 7; ++d) x7.x[d] = x[d];
      flag_exact_words(g, pl, i, j, w, x7);
    }
    unsigned v = 0;
#pragma unroll
    for (int d = 0; d < 7; ++d) {
      v += __popc(x[d]);
      any |= x[d];
    }
    const bool cells_ok = pl.has_i1 && pl.has_j1 && i < g.i_hi;
    unsigned t = 0;
    if (cells_ok) {
      if (!g.any_near) {
#pragma unroll
        for (int d = 0; d < 7; ++d) ncross += __popc(x[d] & pl.kp1);
      } else {
        uint32_t xs[7];
        cross_words(pl, xs);
#pragma unroll
        for (int d = 0; d < 7; ++d) ncross += __popc(xs[d] & pl.kp1);
      }
      uint32_t odd[6], two[6], cand;
      tet_words(pl, nullptr, pl.kp1, odd, two, cand);
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        t += __popc(odd[q]) + 2 * __popc(two[q]);
        em |= odd[q] | two[q];
      }
    }
    if (g.any_near) {
      WordExact we;
      we.ncross = ncross;
      we.ntri = t;
      we.emitting = em;
      we = count_word_exact(g, pl, i, j, w, cells_ok, we);
      ncross = we.ncross;
      t = we.ntri;
      em = we.emitting;
    }
    r = v | (t << 8);
    recc[idx] = r;                                        // record of list entry idx (k_scan walks the list, not the words)
  }
  // The tile aggregate, one atomic per tile and warp: a tile's entries are one contiguous chunk of the list, so the
  // entries of a warp's tiles are runs of consecutive lanes (the lanes without an entry form the last run).  One atomic
  // per word put ~100 atomics on the address of every tile: 0.322 against 0.312 ms per 512^3 step (B200, 1000 W).
  {
    const unsigned tix = have ? (gw - word0) / CS_TILE : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, tix);
    unsigned long long sum = rec_vt(r);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {                   // suffix sums inside the run
      const unsigned long long u = __shfl_down_sync(0xffffffffu, sum, o);
      if (lane + o < 32u && ((peers >> (lane + o)) & 1u)) sum += u;
    }
    if (have && (int)lane == __ffs(peers) - 1 && sum) atomicAdd(&tile_vt[tix], sum);
  }
  if (have) {
    const unsigned v = r & 255u;
    if (v) {
      const uint2 dp = dir_pack(x);
      *reinterpret_cast<uint2*>(&wrec[gw].z) = dp;        // (.x, .y) = (vbase, tbase): k_scan
    }
    if (gw >= emit_end) any = 0u;
    ncells += __popc(em);
  }
  // The slots of the word's owner points and voxels in the work lists come from k_count_a (prefix over the tile's
  // words: no block scan and no barrier here; with them a fifth of this kernel's stall samples sat at the barrier in
  // front of the slot allocation).  A word under a near flag has none -- its exact counts may be smaller than the
  // plain ones -- and takes them from the counters itself (rare).
  unsigned orun = slot.x, crun = slot.y;
  if (flagged) {
    orun = any ? atomicAdd(&ctr->n_own, (unsigned)__popc(any)) : 0u;
    crun = em ? atomicAdd(&ctr->n_cell, (unsigned)__popc(em)) : 0u;
  }
  if (any) {
    uint32_t mo = any;
    // the ranks of an owner's edges within their directions = how many used edges of each direction came before it in
    // the word: seven 5-bit running counts, bumped per owner through a 128-entry table (a count reaches 32 only behind
    // the word's last owner)
    unsigned long long run = 0;
    while (mo) {
      const int b = __ffs(mo) - 1;
      mo &= mo - 1;
      const unsigned m7 = gather7(x, b);
      if (orun < cap_own) {
        own[orun] = make_ulonglong2(((unsigned long long)gw << 13) | ((unsigned)b << 8) | (((pl.P[0] >> b) & 1u) << 7) | m7, run);
      }
      run += sh.spread[m7];
      ++orun;
    }
  }
  if (em) {
    uint32_t me = em;
    unsigned trun = 0;
    Planes npl;
    if (g.any_near) load_planes(g, g.nbits, i, j, w, npl);
    // corner bits (k, k+1) of row ab = bits (b, b+1) of the row's 33-bit window: one funnel shift per row
    const uint32_t hi[4] = {pl.S[0] >> 31, pl.S[1] >> 31, pl.S[2] >> 31, pl.S[3] >> 31};
    while (me) {
      const int b = __ffs(me) - 1;
      me &= me - 1;
      unsigned c8 = 0;
#pragma unroll
      for (int ab = 0; ab < 4; ++ab) c8 |= (__funnelshift_r(pl.P[ab], hi[ab], b) & 3u) << (2 * ab);
      const unsigned en = sh.vox[c8];
      unsigned emit = en & 63u, nt = en >> 8;
      if (g.any_near) {
        unsigned n8 = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) n8 |= ((corner_plane(npl, c) >> b) & 1u) << c;
        bool cand = false;
#pragma unroll
        for (int t = 0; t < 6; ++t) cand = cand || (((emit >> t) & 1u) && tet_mask_of(n8, t) == 15);
        if (cand) {
          emit = cell_emit_exact(g, i, j, w * 32 + b, nullptr);
          nt = 0;
#pragma unroll
          for (int t = 0; t < 6; ++t)
            if ((emit >> t) & 1u) nt += (__popc(tet_mask_of(c8, t)) == 2) ? 2u : 1u;
        }
      }
      if (crun < cap_cell) {
        cell_id[crun] = ((unsigned long long)gw << 28) | ((unsigned long long)trun << 19) | ((unsigned)b << 14) | (emit << 8) | c8;
      }
      ++crun;
      trun += nt;
    }
  }
  unsigned long long cc = ((unsigned long long)ncross << 32) | ncells;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cc += __shfl_xor_sync(0xffffffffu, cc, o);
  if (lane == 0 && cc) {
    if (cc & 0xffffffffull) atomicAdd(&ctr->n_cells, cc & 0xffffffffull);
    if (cc >> 32) atomicAdd(&ctr->n_cross, cc >> 32);
  }
}

// exclusive scan of the tile aggregates (vertices | triangles << 31), in place: one block, a few thousand tiles.
// (As the last act of the last block of k_count_b this cost every block two barriers, a fence and a ticket atomic:
// a quarter of that kernel's stall samples.)
__global__ void __launch_bounds__(1024) k_tile_scan3(unsigned long long* __restrict__ tile_vt, int ntiles, Counters* ctr) {
  __shared__ unsigned long long s_warp[32], s_tot, s_v, s_t;
  ctr_pdl_enter();
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  unsigned long long carry = 0, my_v = 0, my_t = 0;
  if (threadIdx.x == 0) s_v = s_t = 0ull;
  for (int base = 0; base < ntiles; base += 4096) {   // 4 consecutive tiles per thread: 4 K tiles per round
    const int q = base + 4 * (int)threadIdx.x;
    unsigned long long a[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      a[u] = q + u < ntiles ? tile_vt[q + u] : 0ull;
      my_v += a[u] & 0x7fffffffull;                    // a tile's own aggregate is far below 2^31 in both halves
      my_t += a[u] >> 31;
    }
    const unsigned long long mine = a[0] + a[1] + a[2] + a[3];
    const unsigned long long ia = warp_incl_scan_u64(mine);
    __syncthreads();                                  // s_warp / s_tot of the previous round are consumed
    if (lane == 31) s_warp[warp] = ia;
    __syncthreads();
    if (warp == 0) {
      const unsigned long long w = s_warp[lane], iw = warp_incl_scan_u64(w);
      s_warp[lane] = iw - w;                          // exclusive prefix of the warps
      if (lane == 31) s_tot = iw;
    }
    __syncthreads();
    unsigned long long run = carry + s_warp[warp] + ia - mine;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (q + u < ntiles) tile_vt[q + u] = run;
      run += a[u];
    }
    carry += s_tot;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    my_v += __shfl_xor_sync(0xffffffffu, my_v, o);
    my_t += __shfl_xor_sync(0xffffffffu, my_t, o);
  }
  if (lane == 0) {
    atomicAdd(&s_v, my_v);
    atomicAdd(&s_t, my_t);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    ctr->total_vt = carry;
    ctr->tot_v = s_v;
    ctr->tot_t = s_t;
  }
}

// Stage 2b: offsets.  One warp per tile walks the tile's chunk of the interesting-word list (ascending words, k_count_a)
// from the tile's exclusive prefix: vbase[word] (first vertex id of the word), tbase[word] (first triangle of the word)
// -- for interesting words only; nothing reads the others.  (A dense scan over all words read and wrote 48 MB to serve
// the 10 % that matter.)
// The tile prefix: up to SCAN_FUSE_TILES tiles every block sums the aggregates of the tiles in front of its own (a few
// KB from L2, all loads independent) instead of waiting for a one-block scan kernel in front of it (k_tile_scan3:
// 7 us of pure latency in a 0.36 ms step); that is quadratic in the tile count, so larger volumes keep the scan kernel.
constexpr int SCAN_WARPS = 8;
constexpr int SCAN_FUSE_TILES = 8192;              // 512^3 has 4096
template <typename T>
__global__ void __launch_bounds__(SCAN_WARPS * 32) k_scan(Grid<T> g, unsigned word0, int ntiles, const uint32_t* __restrict__ wlist,
                                                         const uint32_t* __restrict__ recc, const uint2* __restrict__ tile_chunk,
                                                         unsigned cap_w, const unsigned long long* __restrict__ tile_vt,
                                                         uint4* __restrict__ wrec, Counters* ctr, int fused) {
  __shared__ unsigned long long s_acc[SCAN_WARPS], s_av[SCAN_WARPS];
  ctr_pdl_enter();
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const int first = (int)(blockIdx.x * SCAN_WARPS);
  const int tile = first + (int)warp;
  unsigned long long run = 0;
  if (fused) {
    // packed (vertices | triangles << 31) and, for the overflow check, the vertices alone:
    // the tiles in front of the block, strided over all its threads ...
    unsigned long long acc = 0, av = 0;
    for (int q = (int)threadIdx.x; q < first; q += SCAN_WARPS * 32) {
      const unsigned long long a = tile_vt[q];
      acc += a;
      av += a & 0x7fffffffull;
    }
    // ... and the block's own tiles in front of this warp's
    unsigned long long own_acc = (lane < warp && first + (int)lane < ntiles) ? tile_vt[first + (int)lane] : 0ull;
    unsigned long long own_av = own_acc & 0x7fffffffull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      acc += __shfl_xor_sync(0xffffffffu, acc, o);
      av += __shfl_xor_sync(0xffffffffu, av, o);
      own_acc += __shfl_xor_sync(0xffffffffu, own_acc, o);
      own_av += __shfl_xor_sync(0xffffffffu, own_av, o);
    }
    if (lane == 0) {
      s_acc[warp] = acc;
      s_av[warp] = av;
    }
    __syncthreads();
    unsigned long long base = 0, base_v = 0;
#pragma unroll
    for (int w = 0; w < SCAN_WARPS; ++w) {
      base += s_acc[w];
      base_v += s_av[w];
    }
    run = base + own_acc;
    if (tile == ntiles - 1 && lane == 0) {             // totals of the run: everything in front of the last tile + the last tile
      const unsigned long long a = tile_vt[tile];
      const unsigned long long tot = run + a, tv = base_v + own_av + (a & 0x7fffffffull);
      ctr->total_vt = tot;
      ctr->tot_v = tv;
      ctr->tot_t = (tot - tv) >> 31;
    }
    if (tile >= ntiles) return;
  } else {
    if (tile >= ntiles) return;
    run = tile_vt[tile];                               // scanned in place by k_tile_scan3
  }
  const unsigned long long run0 = run;
  const unsigned plane_words = (unsigned)g.n1 * (unsigned)g.W;
  const unsigned emit_end = (unsigned)g.i_hi * plane_words;
  const bool want_vemit = g.i_hiv > g.i_hi && (emit_end - word0) / CS_TILE == (unsigned)tile;
  const uint2 ch = tile_chunk[tile];
  unsigned long long below = 0;                        // records of this tile's words in front of emit_end
  for (unsigned q0 = 0; q0 < ch.y; q0 += 64) {         // two rounds per trip: the loads of the second do not wait for the first
    unsigned gw[2];
    unsigned long long item[2];
    bool have[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned q = q0 + 32u * u + lane;
      have[u] = q < ch.y && ch.x + q < cap_w;
      gw[u] = have[u] ? wlist[ch.x + q] : 0u;
      item[u] = have[u] ? rec_vt(recc[ch.x + q]) : 0ull;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const unsigned long long inc = warp_incl_scan_u64(item[u]);
      if (have[u]) {
        const unsigned long long mine = run + inc - item[u];
        // (first vertex id, first triangle) of the word; (.z, .w) is k_count_b's dirpack
        *reinterpret_cast<uint2*>(&wrec[gw[u]].x) = make_uint2((uint32_t)(mine & 0x7fffffffull), (uint32_t)(mine >> 31));
        if (want_vemit && gw[u] < emit_end) below += item[u];
      }
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  if (want_vemit) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
    if (lane == 0) ctr->v_emit = (run0 + below) & 0x7fffffffull;
  }
}

// ------------------------------------------------------------------------------------------------
// Stage 3: vertices.  A warp takes 32 active owner points, then deals their 1..7 owned edges out to its
// lanes one vertex per lane per round (balanced; consecutive lanes write consecutive vertex ids).
// ------------------------------------------------------------------------------------------------
template <typename T, typename G>
__device__ __forceinline__ void grad_at(const Grid<T>& g, int i, int j, int k, G out[3]) {
  const long long s1 = g.n2, s0 = (long long)g.n1 * g.n2;
  const T* c = g.f + ((long long)i * g.n1 + j) * g.n2 + k;
  if (i > 0 && i < g.n0 - 1 && j > 0 && j < g.n1 - 1 && k > 0 && k < g.n2 - 1) {   // interior: plain central differences
    out[0] = ((G)c[s0] - (G)c[-s0]) * (G)0.5;
    out[1] = ((G)c[s1] - (G)c[-s1]) * (G)0.5;
    out[2] = ((G)c[1] - (G)c[-1]) * (G)0.5;
    return;
  }
  {
    const bool lo = i > 0, hi = i < g.n0 - 1;
    G a = (G)c[hi ? s0 : 0], b = (G)c[lo ? -s0 : 0];
    out[0] = (a - b) * ((lo && hi) ? (G)0.5 : (G)1);
  }
  {
    const bool lo = j > 0, hi = j < g.n1 - 1;
    G a = (G)c[hi ? s1 : 0], b = (G)c[lo ? -s1 : 0];
    out[1] = (a - b) * ((lo && hi) ? (G)0.5 : (G)1);
  }
  {
    const bool lo = k > 0, hi = k < g.n2 - 1;
    G a = (G)c[hi ? 1 : 0], b = (G)c[lo ? -1 : 0];
    out[2] = (a - b) * ((lo && hi) ? (G)0.5 : (G)1);
  }
}

__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double shfl_g(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ float shfl_g(float v, int src) { return __shfl_sync(0xffffffffu, v, src); }

struct Xform {
  double origin[3], delta[3], inv_delta[3];
};

// geometry-mode arithmetic: IEEE in fp64 mode (positions bit-exact vs the oracle); fast approximations in fp32 mode (1e-4 rel)
__device__ __forceinline__ double quot(double a, double b) { return a / b; }
__device__ __forceinline__ float quot(float a, float b) { return __fdividef(a, b); }
__device__ __forceinline__ double inv_sqrt(double a) { return 1.0 / sqrt(a); }
__device__ __forceinline__ float inv_sqrt(float a) { return rsqrtf(a); }
// n-th (0-based) set bit of a 7-bit mask (__fns costs ~50 instructions)
__device__ __forceinline__ int nth_set_bit7(unsigned m, unsigned n) {
  int b = 0;
  if ((unsigned)__popc(m & 0xfu) <= n) b = 4;
  if ((unsigned)__popc(m & ((1u << (b + 2)) - 1u)) <= n) b += 2;
  if ((unsigned)__popc(m & ((1u << (b + 1)) - 1u)) <= n) b += 1;
  return b;
}

#ifdef CTR_EV_MINB
#define CTR_EV_BOUNDS __launch_bounds__(256, CTR_EV_MINB)
#else
#define CTR_EV_BOUNDS __launch_bounds__(256)
#endif
template <typename T, typename G>
__global__ void CTR_EV_BOUNDS k_emit_verts(Grid<T> g, const ulonglong2* __restrict__ own,
                                                    const uint4* __restrict__ wrec,
                                                    const Counters* __restrict__ ctr, unsigned cap_own, unsigned cap_v, unsigned w_bound, Xform xf,
                                                    G* __restrict__ verts, G* __restrict__ normals,
                                                    unsigned long long* __restrict__ keys, uint8_t* __restrict__ lowmin) {
  ctr_pdl_enter();
  // more interesting words than k_count_b went through: some slots of the work lists were never written (the host
  // redoes the run with larger pools); nothing to do here
  if (ctr->n_word > w_bound) return;
  // the list length comes from the device counters: the launch may precede the host's read of the counts
  const unsigned n_own = min(ctr->n_own, cap_own);
  const unsigned lane = lane_id();
  const unsigned a = blockIdx.x * blockDim.x + threadIdx.x;          // owner index of this lane
  const unsigned warp_first = a - lane;
  if (warp_first >= n_own) return;
  const bool have = a < n_own;
  const ulonglong2 oent = have ? own[a] : make_ulonglong2(0ull, 0ull);
  const unsigned long long oid = oent.x, ork = oent.y;
  const unsigned ogw = (unsigned)(oid >> 13);
  const uint4 orec = have ? wrec[ogw] : make_uint4(0u, 0u, 0u, 0u);
  const unsigned vb = orec.x;
  const uint2 odp = make_uint2(orec.z, orec.w);
  const unsigned long long dp64 = ((unsigned long long)odp.y << 32) | odp.x;
  const unsigned m7 = (unsigned)oid & 127u;
  int i = 0, j = 0, w = 0;
  g.word_coords(ogw, i, j, w);
  const int k = w * 32 + (int)((oid >> 8) & 31u);
  G fp = (G)0, gp[3] = {(G)0, (G)0, (G)0};
  if (have) {
    fp = (G)g.f[((long long)i * g.n1 + j) * g.n2 + k];
    if (normals) grad_at<T, G>(g, i, j, k, gp);
  }
  const unsigned cnt = __popc(m7);
  const unsigned incl = warp_incl_scan_u32(cnt);
  const unsigned excl = incl - cnt;
  const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
  const G v = (G)g.v;
  // what a vertex lane needs to know about its owner, in one word: prefix (8 bits) | edge mask (7) | low flag (1) | bit (5)
  const unsigned opack = excl | (((unsigned)oid & 0xffu) << 8) | ((unsigned)((oid >> 8) & 31u) << 16);
  for (unsigned base = 0; base < total; base += 32) {
    const unsigned vtx = base + lane;
    const bool act = vtx < total;
    // owner o = last lane whose exclusive prefix <= vtx.  Every listed owner has at least one vertex, so the prefixes
    // are strictly increasing and the owners (lanes 0 .. m-1) are counted by their first vertices: those in front of
    // this round (one ballot) plus those up to this lane's vertex (one warp OR of start bits) -- instead of a
    // five-step binary search by shuffles
    const bool starts_here = cnt > 0 && excl >= base && excl < base + 32u;
    const unsigned starts = __reduce_or_sync(0xffffffffu, starts_here ? 1u << (excl - base) : 0u);
    const unsigned before = __popc(__ballot_sync(0xffffffffu, cnt > 0 && excl < base));
    const int o = (int)(before + __popc(starts & (0xffffffffu >> (31u - lane)))) - 1;
    const unsigned op = __shfl_sync(0xffffffffu, opack, o);
    const unsigned o_excl = op & 255u, o_m7 = (op >> 8) & 127u, o_lo = (op >> 15) & 1u;
    int oi, oj, ow;
    g.word_coords(__shfl_sync(0xffffffffu, ogw, o), oi, oj, ow);
    const int ok = ow * 32 + (int)((op >> 16) & 31u);
    const G ofp = shfl_g(fp, o);
    G ogp[3];
    if (normals) {
      ogp[0] = shfl_g(gp[0], o);
      ogp[1] = shfl_g(gp[1], o);
      ogp[2] = shfl_g(gp[2], o);
    }
    const unsigned o_vb = __shfl_sync(0xffffffffu, vb, o);
    const unsigned long long o_dp = __shfl_sync(0xffffffffu, dp64, o), o_rk = __shfl_sync(0xffffffffu, ork, o);
    if (!act) continue;
    const int d = nth_set_bit7(o_m7, vtx - o_excl) + 1;               // (n+1)-th set bit -> direction 1..7
    const bool p_low = o_lo != 0;
    // id = word base + edges of the word in earlier directions + rank of the point in this direction
    const size_t id = (size_t)o_vb + (d == 1 ? 0u : (unsigned)(o_dp >> (8 * (d - 2))) & 255u) + ((unsigned)(o_rk >> (5 * (d - 1))) & 31u);
    if (id >= cap_v) continue;
    const int di = (d >> 2) & 1, dj = (d >> 1) & 1, dk = d & 1;
    const G fq = (G)g.f[((long long)(oi + di) * g.n1 + (oj + dj)) * g.n2 + (ok + dk)];
    // tetrahedral.py:476-487: key oriented (low, high) by value; ratio = (z-flow)/(fhigh-flow), 0.5 if ~0
    const G flow = p_low ? ofp : fq, fhigh = p_low ? fq : ofp;
    const G den = fhigh - flow;
    const G ratio = (fabs((double)den) <= 1e-8) ? (G)0.5 : quot(v - flow, den);
    // x = low + ratio*(high - low); (high-low) is +-1 or 0 per axis so the product is exact
    const G step = p_low ? ratio : -ratio;
    const int pl[3] = {p_low ? oi : oi + di, p_low ? oj : oj + dj, p_low ? ok : ok + dk};
    const int dd[3] = {di, dj, dk};
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
      const G b0 = (ax == 0) ? (G)((long long)pl[0] + g.plane_offset) : (G)pl[ax];
      const G x = dd[ax] ? add_rn(b0, step) : b0;
      verts[id * 3 + ax] = add_rn(mul_rn(x, (G)xf.delta[ax]), (G)xf.origin[ax]);   // grid_field.py:93
    }
    if (normals) {
      G gq[3];
      grad_at<T, G>(g, oi + di, oj + dj, ok + dk, gq);
      G nn[3], len2 = 0;
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) {
        const G gl = p_low ? ogp[ax] : gq[ax], gh = p_low ? gq[ax] : ogp[ax];
        nn[ax] = add_rn(gl, mul_rn(ratio, gh - gl)) * (G)xf.inv_delta[ax];
        len2 = add_rn(len2, mul_rn(nn[ax], nn[ax]));
      }
      const G inv = len2 > (G)0 ? inv_sqrt(len2) : (G)0;
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) normals[id * 3 + ax] = nn[ax] * inv;
    }
    if (keys) {
      const long long lin = (((long long)oi + g.plane_offset) * g.n1 + oj) * g.n2 + ok;
      keys[id] = ((unsigned long long)lin << 3) | (unsigned)d;
      lowmin[id] = p_low ? 1 : 0;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Stage 4: triangles.  One thread per active voxel.  The ids of the voxel's 19 edges come from
// vbase[word] + rank of the edge among the used edges of its owner's word (popcounts of crossing words).
// ------------------------------------------------------------------------------------------------
constexpr int ET_THREADS = 128;
__constant__ uint32_t c_tri_packed[6 * 16];    // n | slot0<<2 | slot1<<7 | ... (6 slots x 5 bits)

// edge slot e (tables.h CTR_EDGE3_*): owner corner s = a*4 + c*2 + dk and direction d, as compile-time constants
__device__ __forceinline__ constexpr int edge_s(int e) {
  return e < 7 ? 0 : e < 10 ? 1 : e < 13 ? 2 : e < 14 ? 3 : e < 17 ? 4 : e < 18 ? 5 : 6;
}
__device__ __forceinline__ constexpr int edge_d(int e) {
  return e < 7 ? e + 1 : e == 7 ? 2 : e == 8 ? 4 : e == 9 ? 6 : e == 10 ? 1 : e == 11 ? 4 : e == 12 ? 5 : e == 13 ? 4
         : e == 14 ? 1 : e == 15 ? 2 : e == 16 ? 3 : e == 17 ? 2 : 1;
}

// used-edge words of the voxel's four owner rows when some sample nearby is allclose to the isovalue (rare)
struct W28 {
  uint32_t x[4][7];
};

template <typename T>
__device__ __noinline__ W28 rows_used_exact(Grid<T> g, int i, int j, int w) {
  W28 out;
  g.any_near = 1;
  for (int ab = 0; ab < 4; ++ab) {
    Planes pl;
    load_planes(g, g.bits, i + (ab >> 1), j + (ab & 1), w, pl);
    owner_used(g, pl, i + (ab >> 1), j + (ab & 1), w, out.x[ab]);
  }
  return out;
}

// One thread per emitting voxel.  The id of each of the voxel's 19 edges is vbase[owner word] + dirbase + rank of the
// owner bit in that direction's used-edge word -- all from the 2x2 rows of bit words the voxel touches (8 loads) and
// the (vbase, dirpack) records of those rows.
#ifndef CTR_ET_MINB
#define CTR_ET_MINB 10          // 48 registers: 56.4 us (12 -> 40: 57.3; 8 -> 64: 59.5; 7: 60.5; 6 -> 80 registers: 64.5; 5 -> 96: 68.6; unbounded 124: 72.7)
#endif
#define CTR_ET_BOUNDS __launch_bounds__(ET_THREADS, CTR_ET_MINB)
template <typename T>
__global__ void CTR_ET_BOUNDS k_emit_tris(Grid<T> g, const unsigned long long* __restrict__ cell_id,
                                                          const Counters* __restrict__ ctr,
                                                          unsigned cap_cell, unsigned cap_t, unsigned w_bound,
                                                          const uint4* __restrict__ wrec, const uint32_t* __restrict__ vox_tab,
                                                          int* __restrict__ tris) {
  // No wait here: this kernel reads what stage 2 left (lists, records, counters) and nothing that k_emit_verts, the
  // kernel in front of it, writes.  Its blocks are released once every block of k_emit_verts has passed ITS wait, i.e.
  // once stage 2 is complete (common.cuh, rule 2), and fill the SMs that k_emit_verts' last wave leaves idle.  Whatever
  // follows in the stream reads the counters only (k_counts_out) or waits for both kernels (copies, events, plain launches).
  ctr_pdl_trigger();
  if (ctr->n_word > w_bound) return;                  // work lists incomplete (see k_emit_verts)
  const unsigned n_cells = min(ctr->n_cell, cap_cell);
  // per warp: the 19 edge ids of its 32 voxels (row stride 33: a round of the write-out below reads arbitrary
  // (edge, voxel) pairs, and with stride 32 all the edges of one voxel share a bank), and the voxel of each of the
  // warp's triangles
  __shared__ unsigned s_ids[ET_THREADS / 32][19 * 33];
  __shared__ uint8_t s_own[ET_THREADS / 32][32 * 12];
  unsigned a = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned warp_first = a - (threadIdx.x & 31u);
  if (warp_first >= n_cells) return;                  // warp-uniform
  const bool valid = a < n_cells;
  const unsigned long long cid = valid ? cell_id[a] : 0ull;   // lanes past the end run voxel 0 with nothing to emit
  const unsigned c8 = (unsigned)cid & 255u, emit = (unsigned)(cid >> 8) & 63u;
  const int b = (int)((cid >> 14) & 31u);
  const unsigned gw0 = (unsigned)(cid >> 28);
  const unsigned uW = (unsigned)g.W, plane_words = (unsigned)g.n1 * uW;
  const unsigned row = g.divW.div(gw0);
  const unsigned w = gw0 - row * uW;
  const bool near = g.exact_word(row, w) != 0;
  // the voxel's 2x2 rows: word w (P) and the same rows shifted by one sample in k (S)
  const bool next_ok = (w + 1 < uW);
  const unsigned wi[4] = {gw0, gw0 + uW, gw0 + plane_words, gw0 + plane_words + uW};
  uint32_t P[4], S[4];
  unsigned vb[4], vb1[4], tb0 = 0;
  uint2 dp[4], dp1[4];
#pragma unroll
  for (int ab = 0; ab < 4; ++ab) {
    P[ab] = g.bits[wi[ab]];
    const uint32_t nx = next_ok ? g.bits[wi[ab] + 1] : 0u;
    S[ab] = __funnelshift_r(P[ab], nx, 1);
    const uint4 r = wrec[wi[ab]];
    vb[ab] = r.x + g.id_base;
    dp[ab] = make_uint2(r.z, r.w);
    if (ab == 0) tb0 = r.y;
  }
  // used-edge words per owner row (index ab) and direction (index d-1); only the 14 that voxel edges use.  No masks:
  // bits below a valid edge's bit are valid edges of the same direction
  // (registers: only ever indexed by compile-time constants, and never handed out by address)
  uint32_t X[4][7];
  X[0][0] = P[0] ^ S[0]; X[0][1] = P[0] ^ P[1]; X[0][2] = P[0] ^ S[1]; X[0][3] = P[0] ^ P[2];
  X[0][4] = P[0] ^ S[2]; X[0][5] = P[0] ^ P[3]; X[0][6] = P[0] ^ S[3];
  X[1][0] = P[1] ^ S[1]; X[1][3] = P[1] ^ P[3]; X[1][4] = P[1] ^ S[3];
  X[2][0] = P[2] ^ S[2]; X[2][1] = P[2] ^ P[3]; X[2][2] = P[2] ^ S[3];
  X[3][0] = P[3] ^ S[3];
  if (near) {
    const unsigned i = g.divN1.div(row);
    const W28 e = rows_used_exact(g, (int)i, (int)(row - i * (unsigned)g.n1), (int)w);
    X[0][0] = e.x[0][0]; X[0][1] = e.x[0][1]; X[0][2] = e.x[0][2]; X[0][3] = e.x[0][3];
    X[0][4] = e.x[0][4]; X[0][5] = e.x[0][5]; X[0][6] = e.x[0][6];
    X[1][0] = e.x[1][0]; X[1][3] = e.x[1][3]; X[1][4] = e.x[1][4];
    X[2][0] = e.x[2][0]; X[2][1] = e.x[2][1]; X[2][2] = e.x[2][2];
    X[3][0] = e.x[3][0];
  }
  // owner points at k+1: bit b+1 of the same word, or (b == 31) bit 0 of the next word, which has rank 0
  const uint32_t below = (1u << b) - 1u;
  uint32_t below1 = below | (1u << b);
  if (b == 31) {
    below1 = 0u;
#pragma unroll
    for (int ab = 0; ab < 3; ++ab) {
      const uint4 r = wrec[wi[ab] + 1];
      vb1[ab] = r.x + g.id_base;
      dp1[ab] = make_uint2(r.z, r.w);
    }
  } else {
#pragma unroll
    for (int ab = 0; ab < 3; ++ab) {
      vb1[ab] = vb[ab];
      dp1[ab] = dp[ab];
    }
  }
#pragma unroll
  for (int e = 0; e < 19; ++e) {
    const int s = edge_s(e), d = edge_d(e);
    const int ab = s >> 1;
    unsigned id;
    if (s & 1) id = vb1[ab] + dir_base(dp1[ab], d - 1) + __popc(X[ab][d - 1] & below1);
    else id = vb[ab] + dir_base(dp[ab], d - 1) + __popc(X[ab][d - 1] & below);
    s_ids[threadIdx.x >> 5][e * 33 + (threadIdx.x & 31u)] = id;
  }
  // Triangles.  vox_tab[c8]: 12 triangles (3 edge slots x 5 bits each) of the voxel with ALL its mixed tets emitting,
  // then (that tet mask | triangle count << 8).  A lane that wrote its own voxel's triangles would run as long as the
  // warp's busiest voxel (2..12 triangles) and store 4 bytes at a time; instead the warp's triangles are dealt out one
  // per lane per round: each voxel marks its triangles with its lane in shared memory, then lane q of a round takes
  // triangle q -- its voxel from the mark, its row of the table, three ids from s_ids -- and writes it where the scan
  // put it (tbase[word] + offset in the word + index in the voxel): no assumption about the order of the list.
  const unsigned o = valid ? tb0 + ((unsigned)(cid >> 19) & 511u) : 0u;   // the entry's offset is relative to the word's first triangle
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const unsigned* ids = s_ids[warp];
  const uint32_t full = __ldg(vox_tab + c8 * 13 + 12);
  const bool table_path = emit == (full & 63u);
  const unsigned nt = (valid && table_path) ? full >> 8 : 0u;
  if (valid && !table_path) {
    // a voxel that lost tets to the allclose rule (rare): per-tet table, written by its own lane
    unsigned tri = o;
    for (int t = 0; t < 6; ++t) {
      if (!((emit >> t) & 1u)) continue;
      const uint32_t e = c_tri_packed[t * 16 + tet_mask_of(c8, t)];
      for (unsigned h = 0; h < (e & 3u); ++h, ++tri) {
        if (tri >= cap_t) break;
        int* dst = tris + (size_t)tri * 3;
        dst[0] = (int)ids[((e >> (2 + 15 * h)) & 31u) * 33 + lane];
        dst[1] = (int)ids[((e >> (7 + 15 * h)) & 31u) * 33 + lane];
        dst[2] = (int)ids[((e >> (12 + 15 * h)) & 31u) * 33 + lane];
      }
    }
  }
  const unsigned inc = warp_incl_scan_u32(nt);
  const unsigned first = inc - nt;
  const unsigned total = __shfl_sync(0xffffffffu, inc, 31);
  uint8_t* own = s_own[warp];
  for (unsigned t = 0; t < nt; ++t) own[first + t] = (uint8_t)lane;
  __syncwarp();
  for (unsigned q0 = 0; q0 < total; q0 += 32) {
    const unsigned q = q0 + lane;
    const bool act = q < total;
    const unsigned l = act ? own[q] : 0u;
    const unsigned l_first = __shfl_sync(0xffffffffu, first, l);
    const unsigned l_o = __shfl_sync(0xffffffffu, o, l);
    const unsigned l_c8 = __shfl_sync(0xffffffffu, c8, l);
    if (!act) continue;
    const unsigned t = q - l_first;
    const size_t tri = (size_t)l_o + t;
    if (tri >= (size_t)cap_t) continue;
    const uint32_t e = __ldg(vox_tab + l_c8 * 13 + t);
    int* dst = tris + tri * 3;
    dst[0] = (int)ids[(e & 31u) * 33 + l];
    dst[1] = (int)ids[((e >> 5) & 31u) * 33 + l];
    dst[2] = (int)ids[((e >> 10) & 31u) * 33 + l];
  }
}

// ------------------------------------------------------------------------------------------------
// Parity output: (voxel, case code) of emitting voxels, recomputed from the samples in fp64
// (independent of the bit logic above).  Same order as the voxel list.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_codes(Grid<T> g, const unsigned long long* __restrict__ cell_id, unsigned n_cells,
                                               long long* __restrict__ cells, uint32_t* __restrict__ codes) {
  unsigned a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_cells) return;
  const unsigned long long cid = cell_id[a];
  const int b = (int)((cid >> 14) & 31u);
  const unsigned gw = (unsigned)(cid >> 28);
  const unsigned row = gw / (unsigned)g.W;
  const int w = (int)(gw - row * (unsigned)g.W);
  const int i = (int)(row / (unsigned)g.n1), j = (int)(row - (unsigned)i * (unsigned)g.n1);
  const int k = w * 32 + b;
  unsigned code = 0;
  unsigned e = cell_emit_exact(g, i, j, k, &code);
  cells[a] = e ? (((long long)i + g.plane_offset) * (g.n1 - 1) + j) * (long long)(g.n2 - 1) + k : -1;
  codes[a] = code;
}

// ctr_mt3d_offset_ids: vertex ids of the run's triangles shifted by a base that became known after the run was queued
__global__ void k_offset_ids(int* __restrict__ tris, size_t n, int base) {
  const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < n) tris[q] += base;
}

static_assert(sizeof(Counters) <= 1024 && sizeof(Counters) % 4 == 0, "pinned counter mirror is 1 KiB");

// Last kernel of a run: the counter block goes to its page-locked mirror on the host (written through the mapping: a
// cudaMemcpyAsync here put a copy-engine hop between this run's last kernel and the next run's first) and, for
// ctr_mt3d_publish_counts, {n_verts, n_tris} to the device address a collective reads them from.
__global__ void __launch_bounds__(128) k_counts_out(const Counters* __restrict__ ctr, uint32_t* __restrict__ host_mirror, int sharded,
                                                    long long* __restrict__ pub) {
  ctr_pdl_enter();
  const uint32_t* src = reinterpret_cast<const uint32_t*>(ctr);
  for (unsigned q = threadIdx.x; q < sizeof(Counters) / 4; q += blockDim.x) host_mirror[q] = src[q];
  if (pub && threadIdx.x == 0) {
    pub[0] = (long long)(sharded ? ctr->v_emit : ctr->tot_v);
    pub[1] = (long long)ctr->tot_t;
  }
}

// one launch instead of four memsets / copies in front of every run
__global__ void k_reset3(Counters* ctr, uint4* rowflag16, size_t n16, uint4* wordflag16, uint4* exactflag16, size_t nw16,
                         unsigned long long* tile_state, size_t ntile) {
  ctr_pdl_enter();
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)gridDim.x * blockDim.x;
  if (t == 0) {
    Counters c;
    memset(&c, 0, sizeof c);
    c.min_key = ~0ull;
    *ctr = c;
  }
  for (size_t q = t; q < n16; q += n) rowflag16[q] = make_uint4(0u, 0u, 0u, 0u);
  for (size_t q = t; q < nw16; q += n) {
    wordflag16[q] = make_uint4(0u, 0u, 0u, 0u);
    exactflag16[q] = make_uint4(0u, 0u, 0u, 0u);
  }
  for (size_t q = t; q < ntile; q += n) tile_state[q] = 0ull;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool g_tables_loaded[64] = {};

int load_tables(ctr_ctx* ctx) {
  if (ctx->device < 64 && g_tables_loaded[ctx->device]) return 0;
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c_tetmask, CTR_TETMASK3_H, sizeof(CTR_TETMASK3_H)));
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c_tet, CTR_TET3_H, sizeof(CTR_TET3_H)));
  uint32_t packed[96];
  for (int t = 0; t < 6; ++t)
    for (int m = 0; m < 16; ++m) {
      uint32_t e = CTR_TRI3_N_H[t][m];
      for (int q = 0; q < 6; ++q) e |= (uint32_t)(CTR_TRI3_E_H[t][m][q] & 31u) << (2 + 5 * q);
      packed[t * 16 + m] = e;
    }
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c_tri_packed, packed, sizeof(packed)));
  unsigned short vox[256];
  {
    const int xs[6] = {1, 3, 2, 6, 4, 5}, ys[6] = {3, 2, 6, 4, 5, 1};
    for (unsigned c8 = 0; c8 < 256; ++c8) {
      unsigned emit = 0, nt = 0;
      for (int t = 0; t < 6; ++t) {
        const unsigned tm = (c8 & 1u) | (((c8 >> 7) & 1u) << 1) | (((c8 >> xs[t]) & 1u) << 2) | (((c8 >> ys[t]) & 1u) << 3);
        if (tm != 0 && tm != 15) {
          emit |= 1u << t;
          nt += CTR_TRI3_N_H[t][tm];
        }
      }
      vox[c8] = (unsigned short)(emit | (nt << 8));
    }
  }
  CTR_CUDA(ctx, cudaMemcpyToSymbol(c_vox, vox, sizeof(vox)));
  if (ctx->device < 64) g_tables_loaded[ctx->device] = true;
  return 0;
}

// CTR_DEBUG_SYNC=1: synchronise after every launch so that a device fault is reported with the kernel's name
#define CTR_DBG(ctx, name)                                                                       \
  do {                                                                                           \
    static const bool dbg__ = getenv("CTR_DEBUG_SYNC") != nullptr;                               \
    if (dbg__) {                                                                                 \
      cudaError_t e__ = cudaStreamSynchronize((ctx)->stream);                                    \
      if (e__ != cudaSuccess) return ctr_fail(ctx, CTR_ERR_CUDA, name, cudaGetErrorString(e__)); \
    }                                                                                            \
  } while (0)

// phase 0: enqueue and wait (ctr_mt3d_run); 1: enqueue only (ctr_mt3d_enqueue); 2: wait for what phase 1 enqueued,
// check the counts, redo synchronously only if a capacity was too small (ctr_mt3d_finish)
template <typename T>
int run_typed(ctr_ctx* ctx, const ctr_mt3d_params* p, ctr_mt3d_counts* out, int phase) {
  const int n0 = (int)p->n0, n1 = (int)p->n1, n2 = (int)p->n2;
  const int W = (n2 + 31) / 32;
  const long long nrows = (long long)n0 * n1;
  const long long nwords = nrows * W;
  const size_t nsamp = (size_t)nrows * n2;
  cudaStream_t st = ctx->stream;
  if (nwords >= (1ll << 31) - 64) return ctr_fail(ctx, CTR_ERR_UNSUPPORTED, "volume too large for 32-bit word indices");
  int rc;
  if ((rc = load_tables(ctx))) return rc;
  if (phase != 2) ctr_stage_mark(ctx, 0);
  const T* dfield;
  if (p->flags & CTR_FIELD_ON_DEVICE) {
    dfield = (const T*)p->field;
  } else {
    if ((rc = ctr_ensure(ctx, ctx->field, nsamp * sizeof(T)))) return rc;
    if (phase != 2) CTR_CUDA(ctx, cudaMemcpyAsync(ctx->field.p, p->field, nsamp * sizeof(T), cudaMemcpyHostToDevice, st));
    dfield = (const T*)ctx->field.p;
  }
  if (phase != 2) ctr_stage_mark(ctx, 1);

  Grid<T> g;
  g.f = dfield;
  g.n0 = n0; g.n1 = n1; g.n2 = n2; g.W = W;
  g.i_lo = (int)p->i_lo;
  g.i_hi = (int)p->i_hi;
  g.i_hiv = std::min(g.i_hi + 1, n0);
  g.plane_offset = p->plane_offset;
  g.id_base = (unsigned)p->vert_id_base;
  g.v = p->isovalue;
  g.tolv = 1e-8 + 1e-5 * fabs(p->isovalue);
  g.any_near = 0;
  g.divW.init((unsigned)W);
  g.divN1.init((unsigned)n1);
  const long long plane_words = (long long)n1 * W;
  const unsigned word0 = (unsigned)((long long)g.i_lo * plane_words);
  const unsigned nscan = (unsigned)((long long)(g.i_hiv - g.i_lo) * plane_words);
  const int ntiles = (int)((nscan + CS_TILE - 1) / CS_TILE);

  if ((rc = ctr_ensure(ctx, ctx->bits, (size_t)(nwords + 4) * 4))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->nbits, (size_t)(nwords + 4) * 4))) return rc;
  // per word (first vertex id, first triangle, dirpack lo, dirpack hi): one 16-byte record, written for interesting words only
  if ((rc = ctr_ensure(ctx, ctx->wdir, (size_t)(nwords + 4) * 16))) return rc;
  if (!ctx->vox_tab.p) {
    // corner bits -> triangle list of the whole voxel (tet order, then triangle order), then (tet mask | count << 8)
    static uint32_t tab[256 * 13];
    const int xs[6] = {1, 3, 2, 6, 4, 5}, ys[6] = {3, 2, 6, 4, 5, 1};
    for (unsigned c8 = 0; c8 < 256; ++c8) {
      uint32_t* e = tab + c8 * 13;
      for (int q = 0; q < 13; ++q) e[q] = 0;
      unsigned k = 0, mask = 0;
      for (int t = 0; t < 6; ++t) {
        const unsigned m = (c8 & 1u) | (((c8 >> 7) & 1u) << 1) | (((c8 >> xs[t]) & 1u) << 2) | (((c8 >> ys[t]) & 1u) << 3);
        if (m != 0 && m != 15) mask |= 1u << t;
        for (int tri = 0; tri < CTR_TRI3_N_H[t][m]; ++tri, ++k)
          e[k] = (uint32_t)(CTR_TRI3_E_H[t][m][tri * 3] & 31u) | ((uint32_t)(CTR_TRI3_E_H[t][m][tri * 3 + 1] & 31u) << 5) |
                 ((uint32_t)(CTR_TRI3_E_H[t][m][tri * 3 + 2] & 31u) << 10);
      }
      e[12] = mask | (k << 8);
    }
    if ((rc = ctr_ensure(ctx, ctx->vox_tab, sizeof tab, true))) return rc;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->vox_tab.p, tab, sizeof tab, cudaMemcpyHostToDevice, st));
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  if ((rc = ctr_ensure(ctx, ctx->counters, sizeof(Counters)))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->aux[4], (size_t)nrows + 32))) return rc;
  if ((rc = ctr_ensure(ctx, ctx->aux[32], (size_t)nrows * 4 + 64))) return rc;      // word-level near flags
  if ((rc = ctr_ensure(ctx, ctx->aux[35], (size_t)nrows * 4 + 64))) return rc;      // word-level "exact differs" flags
  if ((rc = ctr_ensure(ctx, ctx->tile_state, (size_t)ntiles * 16 + 16))) return rc;
  if (!ctx->counters_host) CTR_CUDA(ctx, cudaMallocHost(&ctx->counters_host, 1024));
  g.bits = (const uint32_t*)ctx->bits.p;
  g.nbits = (const uint32_t*)ctx->nbits.p;
  g.rowflag = (const uint8_t*)ctx->aux[4].p;
  g.wordflag = (const uint32_t*)ctx->aux[32].p;
  g.exactflag = (uint32_t*)ctx->aux[35].p;
  g.wshift = 0;
  while ((W >> g.wshift) > 32) ++g.wshift;
  Counters* dctr = (Counters*)ctx->counters.p;
  unsigned long long* st_vt = (unsigned long long*)ctx->tile_state.p;

  const bool geom = !(p->flags & CTR_NO_GEOMETRY);
  const bool f64 = (p->flags & CTR_GEOM_F64) != 0;
  const size_t gsz = f64 ? 8 : 4;
  const bool want_n = (p->flags & CTR_WANT_NORMALS) != 0, want_k = (p->flags & CTR_WANT_KEYS) != 0;
  Xform xf;
  for (int a = 0; a < 3; ++a) {
    xf.origin[a] = p->origin[a];
    xf.delta[a] = p->delta[a];
    xf.inv_delta[a] = 1.0 / p->delta[a];
  }
  // Work lists and output pools are grow-only.  Their capacities come from earlier runs (or a guess on the first one):
  // every stage is enqueued against them without waiting for the counts -- kernels read the list lengths from the
  // device counters and never write past a capacity -- and the counts are checked after the single synchronisation
  // at the end.  Only when a capacity turns out too small are the buffers grown and the affected stages redone.
  DevBuf& b_own = ctx->aux[0];
  DevBuf& b_cell_id = ctx->aux[2];
  if (!ctx->spec_w) ctx->spec_w = std::max<size_t>((size_t)nwords / 4, 1 << 14);
  if (!ctx->spec_own) ctx->spec_own = std::max<size_t>((size_t)nwords / 2, 1 << 14);
  if (!ctx->spec_cell) ctx->spec_cell = ctx->spec_own;
  if (!ctx->spec_v) ctx->spec_v = ctx->spec_own * 2;
  if (!ctx->spec_t) ctx->spec_t = ctx->spec_cell * 4;
  Counters h;
  unsigned long long totV = 0, totT = 0, nOwn = 0, nCell = 0, nV = 0;
  for (int attempt = 0;; ++attempt) {
    if ((rc = ctr_ensure(ctx, b_own, ctx->spec_own * 16, true))) return rc;
    if ((rc = ctr_ensure(ctx, b_cell_id, ctx->spec_cell * 8, true))) return rc;
    if ((rc = ctr_ensure(ctx, ctx->wlist, ctx->spec_w * 4, true))) return rc;
    if ((rc = ctr_ensure(ctx, ctx->aux[33], ctx->spec_w * 4, true))) return rc;                 // records of the listed words
    if ((rc = ctr_ensure(ctx, ctx->aux[41], ctx->spec_w * 8, true))) return rc;                 // their first slots in the work lists
    if ((rc = ctr_ensure(ctx, ctx->aux[34], (size_t)ntiles * 8 + 16))) return rc;               // (first entry, entries) per tile
    if (geom) {
      if ((rc = ctr_ensure(ctx, ctx->verts, ctx->spec_v * 3 * gsz, true))) return rc;
      if (want_n && (rc = ctr_ensure(ctx, ctx->normals, ctx->spec_v * 3 * gsz, true))) return rc;
      if (want_k && (rc = ctr_ensure(ctx, ctx->keys, ctx->spec_v * 8, true))) return rc;
      if (want_k && (rc = ctr_ensure(ctx, ctx->lowmin, ctx->spec_v, true))) return rc;
      if ((rc = ctr_ensure(ctx, ctx->tris, ctx->spec_t * 12, true))) return rc;
    }
    const unsigned cap_own = (unsigned)std::min<size_t>(ctx->spec_own, 0x7fffffffu);
    const unsigned cap_cell = (unsigned)std::min<size_t>(ctx->spec_cell, 0x7fffffffu);
    const unsigned cap_v = (unsigned)std::min<size_t>(ctx->spec_v, 0x7fffffffu);
    const unsigned cap_t = (unsigned)std::min<size_t>(ctx->spec_t, 0x7fffffffu);
    const unsigned cap_w = (unsigned)std::min<size_t>(ctx->spec_w, 0x7fffffffu);

    if (!(phase == 2 && attempt == 0)) {                 // phase 2: attempt 0 was enqueued by phase 1
    ctr_launch_dep(k_reset3, 64, 256, 0, st, dctr, (uint4*)ctx->aux[4].p, (size_t)(nrows + 15) / 16, (uint4*)ctx->aux[32].p,
                   (uint4*)ctx->aux[35].p, (size_t)(nrows + 3) / 4, st_vt, (size_t)ntiles);
    ctx->launches++;
    CTR_DBG(ctx, "k_reset3");
    rc = launch_bitplane<T>(ctx, dfield, (unsigned)nrows, n2, W, n0, n1, p->isovalue, (uint32_t*)ctx->bits.p, (uint32_t*)ctx->nbits.p,
                            (uint8_t*)ctx->aux[4].p, (MinMaxKeys*)dctr, (p->flags & CTR_WANT_MINMAX) != 0, false, (uint32_t*)ctx->aux[32].p);
    if (rc) return rc;
    CTR_DBG(ctx, "k_bitplane");
    ctr_stage_mark(ctx, 2);
    if (ntiles > 0) {
      ctr_launch_dep(k_count_a<T>, ntiles, CS_THREADS, 0, st, g, word0, nscan, (uint32_t*)ctx->wlist.p, (uint2*)ctx->aux[41].p,
                     (uint2*)ctx->aux[34].p, cap_w, dctr);
      CTR_DBG(ctx, "k_count_a");
      // the grid covers the expected list length (last run's, with head-room); blocks past the real length only take a ticket
      const unsigned wb = (unsigned)((std::min<size_t>(cap_w, ctx->last_w + ctx->last_w / 8 + 4096) + CB_THREADS - 1) / CB_THREADS);
      ctr_launch_dep(k_count_b<T>, wb, CB_THREADS, 0, st, g, word0, (const uint32_t*)ctx->wlist.p, (const uint2*)ctx->aux[41].p, cap_w,
                     (uint32_t*)ctx->aux[33].p,
                     (uint4*)ctx->wdir.p, (ulonglong2*)b_own.p, (unsigned long long*)b_cell_id.p, cap_own, cap_cell, st_vt, dctr, ntiles);
      const int fused = ntiles <= SCAN_FUSE_TILES ? 1 : 0;
      if (!fused) ctr_launch_dep(k_tile_scan3, 1, 1024, 0, st, st_vt, ntiles, dctr);
      ctx->launches += 3 - fused;
      ctx->cover_w = (size_t)wb * CB_THREADS;
      CTR_DBG(ctx, "k_count_b");
      ctr_launch_dep(k_scan<T>, (ntiles + SCAN_WARPS - 1) / SCAN_WARPS, SCAN_WARPS * 32, 0, st,
                     g, word0, ntiles, (const uint32_t*)ctx->wlist.p, (const uint32_t*)ctx->aux[33].p, (const uint2*)ctx->aux[34].p, cap_w,
                     (const unsigned long long*)st_vt, (uint4*)ctx->wdir.p, dctr, fused);
      ctx->launches++;
      CTR_DBG(ctx, "k_scan");
    }
    ctr_stage_mark(ctx, 3);
    if (geom && ntiles > 0) {
      unsigned long long* dkeys = want_k ? (unsigned long long*)ctx->keys.p : nullptr;
      uint8_t* dlow = want_k ? (uint8_t*)ctx->lowmin.p : nullptr;
      // grids cover the expected list lengths (last run's, with head-room); blocks past the real length return at once
      const unsigned vb = (unsigned)((std::min<size_t>(cap_own, ctx->last_own + ctx->last_own / 8 + 4096) + 255) / 256);
      // the kernels read list entries below min(list length, this bound): the grid's cover rounded up to whole blocks
      // may pass the list's capacity, and entries behind the capacity do not exist
      const unsigned bound_own = std::min(vb * 256u, cap_own);
      const unsigned w_bound = (unsigned)std::min<size_t>(cap_w, ctx->cover_w);
      const ulonglong2* oid = (const ulonglong2*)b_own.p;
      const uint4* dwr = (const uint4*)ctx->wdir.p;
      if (f64)
        ctr_launch_dep(k_emit_verts<T, double>, vb, 256, 0, st, g, oid, dwr, dctr, bound_own, cap_v, w_bound, xf, (double*)ctx->verts.p,
                       want_n ? (double*)ctx->normals.p : (double*)nullptr, dkeys, dlow);
      else
        ctr_launch_dep(k_emit_verts<T, float>, vb, 256, 0, st, g, oid, dwr, dctr, bound_own, cap_v, w_bound, xf, (float*)ctx->verts.p,
                       want_n ? (float*)ctx->normals.p : (float*)nullptr, dkeys, dlow);
      ctx->launches++;
      CTR_DBG(ctx, "k_emit_verts");
      ctr_stage_mark(ctx, 4);
      const unsigned tb = (unsigned)((std::min<size_t>(cap_cell, ctx->last_cell + ctx->last_cell / 8 + 4096) + ET_THREADS - 1) / ET_THREADS);
      ctr_launch_dep(k_emit_tris<T>, tb, ET_THREADS, 0, st, g, (const unsigned long long*)b_cell_id.p, (const Counters*)dctr,
                     std::min(tb * (unsigned)ET_THREADS, cap_cell), cap_t, w_bound, (const uint4*)ctx->wdir.p,
                     (const uint32_t*)ctx->vox_tab.p, (int*)ctx->tris.p);
      ctx->launches++;
      CTR_DBG(ctx, "k_emit_tris");
      ctr_stage_mark(ctx, 5);
      // what the launches above could cover
      ctx->cover_own = (size_t)vb * 256u;
      ctx->cover_cell = (size_t)tb * ET_THREADS;
    } else {
      ctr_stage_mark(ctx, 4);
      ctr_stage_mark(ctx, 5);
      ctx->cover_own = ctx->cover_cell = (size_t)-1;
    }
    // the counts travel behind the last kernel (nothing sits between the kernels of a run: each may start under the tail
    // of the one before, ctr_launch_dep); the host reads them after its single wait anyway
    {
      void* mirror = nullptr;
      CTR_CUDA(ctx, cudaHostGetDevicePointer(&mirror, ctx->counters_host, 0));
      ctr_launch_dep(k_counts_out, 1, 128, 0, st, (const Counters*)dctr, (uint32_t*)mirror, g.i_hiv > g.i_hi ? 1 : 0, ctx->publish3);
      ctx->launches++;
    }
    }
    if (phase == 1) {
      CTR_CUDA(ctx, cudaGetLastError());
      if (!ctx->ev_enqueued) CTR_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_enqueued, cudaEventDisableTiming));
      CTR_CUDA(ctx, cudaEventRecord(ctx->ev_enqueued, st));
      return 0;                                          // ctr_mt3d_finish picks up from here
    }
    CTR_CUDA(ctx, cudaGetLastError());
    if (phase == 2 && attempt == 0) CTR_CUDA(ctx, cudaEventSynchronize(ctx->ev_enqueued));   // only what the enqueue queued
    else CTR_CUDA(ctx, cudaStreamSynchronize(st));
    memcpy(&h, ctx->counters_host, sizeof h);
    totV = h.tot_v;
    totT = h.tot_t;
    nOwn = h.n_own;
    nCell = h.n_cell;
    nV = (g.i_hiv > g.i_hi) ? h.v_emit : totV;
    if (totV >= 0x7ffffff0ull || totT >= 0x7ffffff0ull)
      return ctr_fail(ctx, CTR_ERR_OVERFLOW, "more than 2^31 vertices or triangles in one call; shard the volume");
    ctx->last_own = (size_t)nOwn;
    ctx->last_cell = (size_t)nCell;
    const size_t nWord = (size_t)h.n_word;
    ctx->last_w = nWord;
    const bool ok = nWord <= cap_w && nWord <= ctx->cover_w && nOwn <= cap_own && nCell <= cap_cell && (!geom || (nV <= cap_v && totT <= cap_t && nOwn <= ctx->cover_own &&
                                                                       nCell <= ctx->cover_cell));
    if (ok) break;
    if (attempt == 3) return ctr_fail(ctx, CTR_ERR_STATE, "capacities did not converge");
    ctx->spec_w = std::max<size_t>(ctx->spec_w, nWord + nWord / 4 + 1024);
    ctx->spec_own = std::max<size_t>(ctx->spec_own, (size_t)nOwn + (size_t)nOwn / 4 + 1024);
    ctx->spec_cell = std::max<size_t>(ctx->spec_cell, (size_t)nCell + (size_t)nCell / 4 + 1024);
    ctx->spec_v = std::max<size_t>(ctx->spec_v, (size_t)nV + (size_t)nV / 4 + 1024);
    ctx->spec_t = std::max<size_t>(ctx->spec_t, (size_t)totT + (size_t)totT / 4 + 1024);
  }

  out->n_verts = (int64_t)nV;
  out->n_tris = (int64_t)totT;
  out->n_active_cells = (int64_t)h.n_cells;
  out->n_crossings = (int64_t)h.n_cross;
  out->n_codes = 0;
  const bool mm = (p->flags & CTR_WANT_MINMAX) && h.min_key != ~0ull;
  out->fmin = mm ? key_to_double(h.min_key) : NAN;
  out->fmax = mm ? key_to_double(h.max_key) : NAN;

  if (p->flags & CTR_WANT_CODES) {
    if ((rc = ctr_ensure(ctx, ctx->cells, (size_t)nCell * 8 + 8))) return rc;
    if ((rc = ctr_ensure(ctx, ctx->codes, (size_t)nCell * 4 + 4))) return rc;
    if (nCell) {
      k_codes<T><<<(unsigned)((nCell + 255) / 256), 256, 0, st>>>(g, (const unsigned long long*)b_cell_id.p, (unsigned)nCell,
                                                                   (long long*)ctx->cells.p, (uint32_t*)ctx->codes.p);
      ctx->launches++;
    }
    out->n_codes = (int64_t)nCell;
    CTR_CUDA(ctx, cudaGetLastError());
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
  }
  ctr_stage_mark(ctx, 6);
  if (ctx->timing) {
    CTR_CUDA(ctx, cudaStreamSynchronize(st));
    for (int s = 0; s < 6; ++s) {
      ctx->stage_ms[s] = 0.f;
      if (ctx->ev_set[s] && ctx->ev_set[s + 1]) cudaEventElapsedTime(&ctx->stage_ms[s], ctx->ev[s], ctx->ev[s + 1]);
    }
  }
  ctx->last_kind = 3;
  ctx->last3_edited = 0;
  ctx->last_flags = p->flags;
  ctx->last_counts[0] = (int64_t)nV;
  ctx->last_counts[1] = (int64_t)totT;
  ctx->last_counts[2] = out->n_codes;
  memcpy(ctx->last3_params, p, sizeof *p);            // ctr_mt3d_select_seeded works on this run
  return 0;
}

#include "mt3d_select.cuh"
#include "mt3d_keep.cuh"
#include "mt3d_clean.cuh"
#include "attr3d.cuh"

}  // namespace

static_assert(sizeof(ctr_mt3d_params) <= sizeof(((ctr_ctx*)nullptr)->pending3_params), "pending3_params too small");

static int mt3d_check(ctr_ctx* ctx, const ctr_mt3d_params* p) {
  if (!p || !p->field) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (p->n0 < 2 || p->n1 < 2 || p->n2 < 2) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "grid must have at least 2 samples per axis");
  if (p->n0 > 0x7ffffff0ll || p->n1 > 0x7ffffff0ll || p->n2 > 0x7ffffff0ll) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "axis too long");
  if (p->i_lo < 0 || p->i_hi > p->n0 || p->i_lo >= p->i_hi) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "bad slab range [i_lo, i_hi)");
  if (p->vert_id_base < 0 || p->vert_id_base > 0x7fffffffll) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "vert_id_base out of range");
  if (!(p->isovalue == p->isovalue)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "isovalue is NaN");
  for (int a = 0; a < 3; ++a)
    if (p->delta[a] == 0.0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "delta must be non-zero");
  if (p->dtype != CTR_F32 && p->dtype != CTR_F64 && p->dtype != CTR_U8 && p->dtype != CTR_I16 && p->dtype != CTR_U16)
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32, CTR_F64, CTR_U8, CTR_I16 or CTR_U16");
  return 0;
}

static int mt3d_dispatch(ctr_ctx* ctx, const ctr_mt3d_params* p, ctr_mt3d_counts* out, int phase) {
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (out) memset(out, 0, sizeof *out);
  ctx->last_kind = 0;
  ctx->mesh_gen++;
  ctx->attr_ncomp = 0;                                 // vertex values of the previous run are gone
  ctx->comp_count = -1;                                // ... and so are its components
  switch (p->dtype) {
    case CTR_F32: return run_typed<float>(ctx, p, out, phase);
    case CTR_F64: return run_typed<double>(ctx, p, out, phase);
    case CTR_U8: return run_typed<uint8_t>(ctx, p, out, phase);
    case CTR_I16: return run_typed<int16_t>(ctx, p, out, phase);
    case CTR_U16: return run_typed<uint16_t>(ctx, p, out, phase);
  }
  return ctr_fail(ctx, CTR_ERR_BAD_ARG, "unknown dtype");
}

extern "C" int ctr_mt3d_run(ctr_ctx* ctx, const ctr_mt3d_params* p, ctr_mt3d_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  ctx->pending3 = false;
  int rc = mt3d_check(ctx, p);
  if (rc) return rc;
  return mt3d_dispatch(ctx, p, out, 0);
}

extern "C" int ctr_mt3d_enqueue(ctr_ctx* ctx, const ctr_mt3d_params* p) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  ctx->pending3 = false;
  int rc = mt3d_check(ctx, p);
  if (rc) return rc;
  if (p->flags & CTR_WANT_CODES) return ctr_fail(ctx, CTR_ERR_UNSUPPORTED, "CTR_WANT_CODES needs the synchronous ctr_mt3d_run");
  memcpy(ctx->pending3_params, p, sizeof *p);
  rc = mt3d_dispatch(ctx, p, nullptr, 1);
  ctx->pending3 = rc == 0;
  return rc;
}

extern "C" int ctr_mt3d_finish(ctr_ctx* ctx, ctr_mt3d_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (!ctx->pending3) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_enqueue to finish");
  ctx->pending3 = false;
  return mt3d_dispatch(ctx, (const ctr_mt3d_params*)ctx->pending3_params, out, 2);
}

extern "C" int ctr_mt3d_offset_ids(ctr_ctx* ctx, int64_t base) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY)) return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry");
  if (base < 0 || base > 0x7fffffffll) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "id base out of range");
  const size_t n = (size_t)ctx->last_counts[1] * 3;
  if (!n || !base) return 0;
  ctx->mesh_gen++;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  k_offset_ids<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>((int*)ctx->tris.p, n, (int)base);
  ctx->launches++;
  CTR_CUDA(ctx, cudaGetLastError());
  return 0;                                            // stream-ordered: the fetch that follows sees the shifted ids
}

extern "C" int ctr_mt3d_publish_counts(ctr_ctx* ctx, void* device_counts) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (((uintptr_t)device_counts) & 7u) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "device_counts must be 8-byte aligned");
  ctx->publish3 = (long long*)device_counts;
  return 0;
}

extern "C" int ctr_mt3d_fetch(ctr_ctx* ctx, void* verts, void* normals, int32_t* tris, uint64_t* keys,
                              uint8_t* lowmin, int64_t* cells, uint32_t* codes) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3) return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run to fetch from");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  const uint32_t fl = ctx->last_flags;
  const size_t gsz = (fl & CTR_GEOM_F64) ? 8 : 4;
  const size_t nV = (size_t)ctx->last_counts[0], nT = (size_t)ctx->last_counts[1], nC = (size_t)ctx->last_counts[2];
  cudaStream_t st = ctx->stream;
  const bool geom = !(fl & CTR_NO_GEOMETRY);
  if (verts) {
    if (!geom) return ctr_fail(ctx, CTR_ERR_STATE, "run had CTR_NO_GEOMETRY");
    if (nV) CTR_CUDA(ctx, cudaMemcpyAsync(verts, ctx->verts.p, nV * 3 * gsz, cudaMemcpyDeviceToHost, st));
  }
  if (normals) {
    if (!geom || !(fl & CTR_WANT_NORMALS)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not compute normals");
    if (nV) CTR_CUDA(ctx, cudaMemcpyAsync(normals, ctx->normals.p, nV * 3 * gsz, cudaMemcpyDeviceToHost, st));
  }
  if (tris) {
    if (!geom) return ctr_fail(ctx, CTR_ERR_STATE, "run had CTR_NO_GEOMETRY");
    if (nT) CTR_CUDA(ctx, cudaMemcpyAsync(tris, ctx->tris.p, nT * 12, cudaMemcpyDeviceToHost, st));
  }
  if (keys || lowmin) {
    if (!geom || !(fl & CTR_WANT_KEYS)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not compute keys");
    if (keys && nV) CTR_CUDA(ctx, cudaMemcpyAsync(keys, ctx->keys.p, nV * 8, cudaMemcpyDeviceToHost, st));
    if (lowmin && nV) CTR_CUDA(ctx, cudaMemcpyAsync(lowmin, ctx->lowmin.p, nV, cudaMemcpyDeviceToHost, st));
  }
  if (cells || codes) {
    if (!(fl & CTR_WANT_CODES)) return ctr_fail(ctx, CTR_ERR_STATE, "run did not compute case codes");
    if (cells && nC) CTR_CUDA(ctx, cudaMemcpyAsync(cells, ctx->cells.p, nC * 8, cudaMemcpyDeviceToHost, st));
    if (codes && nC) CTR_CUDA(ctx, cudaMemcpyAsync(codes, ctx->codes.p, nC * 4, cudaMemcpyDeviceToHost, st));
  }
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  return 0;
}

extern "C" int ctr_mt3d_device_ptrs(ctr_ctx* ctx, void** verts, void** normals, int32_t** tris) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3) return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run");
  if (verts) *verts = ctx->verts.p;
  if (normals) *normals = (ctx->last_flags & CTR_WANT_NORMALS) ? ctx->normals.p : nullptr;
  if (tris) *tris = (int32_t*)ctx->tris.p;
  return 0;
}

extern "C" int ctr_mt3d_select_seeded(ctr_ctx* ctx, const int32_t* seed_voxels, int64_t n_seeds, int64_t* n_verts,
                                      int64_t* n_tris, int64_t* n_voxels) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (n_seeds < 0 || (n_seeds > 0 && !seed_voxels)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "bad seed list");
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to select from");
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  if (p->i_lo != 0 || p->i_hi != p->n0)
    return ctr_fail(ctx, CTR_ERR_UNSUPPORTED, "seeded selection needs a full-volume run (components cross slab faces)");
  // the selection compacts the run's mesh in place while the voxel work list keeps its per-voxel triangle offsets: it
  // can be applied once per run
  if (ctx->last3_edited)
    return ctr_fail(ctx, CTR_ERR_STATE, "the mesh of this run has already been selected from, cleaned, filtered or smoothed; run ctr_mt3d_run again");
  ctx->mesh_gen++;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  switch (p->dtype) {
    case CTR_F32: return select_typed<float>(ctx, p, seed_voxels, n_seeds, n_verts, n_tris, n_voxels);
    case CTR_F64: return select_typed<double>(ctx, p, seed_voxels, n_seeds, n_verts, n_tris, n_voxels);
    case CTR_U8: return select_typed<uint8_t>(ctx, p, seed_voxels, n_seeds, n_verts, n_tris, n_voxels);
    case CTR_I16: return select_typed<int16_t>(ctx, p, seed_voxels, n_seeds, n_verts, n_tris, n_voxels);
    case CTR_U16: return select_typed<uint16_t>(ctx, p, seed_voxels, n_seeds, n_verts, n_tris, n_voxels);
  }
  return ctr_fail(ctx, CTR_ERR_BAD_ARG, "unknown dtype");
}

extern "C" int ctr_mt3d_keep_components(ctr_ctx* ctx, const uint8_t* keep, int64_t n_keep, int64_t* n_verts, int64_t* n_tris) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (ctx->last_kind != 3 || ctx->comp_count < 0)
    return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_components since the last 3D run");
  if (ctx->comp_gen != ctx->mesh_gen)
    return ctr_fail(ctx, CTR_ERR_STATE, "the mesh was edited after ctr_mt3d_components (selection, clean-up, smoothing or offset_ids): "
                                        "call ctr_mt3d_components again");
  if (n_keep != ctx->comp_count || (!keep && n_keep > 0))
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "keep must hold one byte per component of the last ctr_mt3d_components call");
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  return keep_components_run(ctx, keep, n_verts, n_tris);
}

extern "C" int ctr_mt3d_clean(ctr_ctx* ctx, const ctr_clean_params* cp, ctr_clean_counts* out) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!cp || !out) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  memset(out, 0, sizeof *out);
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to clean");
  if (ctx->last3_edited & 2u) return ctr_fail(ctx, CTR_ERR_STATE, "the mesh of this run has already been cleaned");
  // the reference's clean-up (quantize, tiny simplices) is defined on the interpolated positions
  if (ctx->last3_edited & 8u) return ctr_fail(ctx, CTR_ERR_STATE, "the mesh of this run has been smoothed: clean it up before smoothing");
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  if (p->i_lo != 0 || p->i_hi != p->n0 || p->vert_id_base != 0)
    return ctr_fail(ctx, CTR_ERR_UNSUPPORTED, "mesh clean-up needs a full-volume run (merges cross slab faces)");
  for (int a = 0; a < 3; ++a) {
    if (p->origin[a] != 0.0 || p->delta[a] != 1.0)
      return ctr_fail(ctx, CTR_ERR_STATE, "mesh clean-up works in grid coordinates: run with origin 0, delta 1 and pass the transform here");
    if (cp->corner[a] < 1) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "corner must be >= 1 on every axis");
    if (cp->delta[a] == 0.0) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "delta must be non-zero");
  }
  if (cp->divisions < 1 || cp->divisions >= (1 << 21)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "divisions must be in [1, 2^21)");
  if (!(cp->epsilon == cp->epsilon)) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "epsilon is NaN");
  ctx->mesh_gen++;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->last_flags & CTR_GEOM_F64) return clean_typed<double>(ctx, cp, out);
  return clean_typed<float>(ctx, cp, out);
}

extern "C" int ctr_mt3d_interpolate(ctr_ctx* ctx, const ctr_attr_params* a, int64_t* n_verts) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!a || !a->field) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  if (a->ncomp < 1 || a->ncomp > 4) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "ncomp must be 1..4");
  if (a->dtype != CTR_F32 && a->dtype != CTR_F64 && a->dtype != CTR_U8 && a->dtype != CTR_I16 && a->dtype != CTR_U16)
    return ctr_fail(ctx, CTR_ERR_BAD_ARG, "dtype must be CTR_F32, CTR_F64, CTR_U8, CTR_I16 or CTR_U16");
  if (ctx->last_kind != 3 || (ctx->last_flags & CTR_NO_GEOMETRY))
    return ctr_fail(ctx, CTR_ERR_STATE, "no completed ctr_mt3d_run with geometry to interpolate on");
  if (!(ctx->last_flags & CTR_WANT_KEYS)) return ctr_fail(ctx, CTR_ERR_STATE, "the run did not keep its keys: run with CTR_WANT_KEYS");
  ctx->attr_ncomp = 0;                                 // the buffer is rewritten: earlier values are gone
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  switch (p->dtype) {
    case CTR_F32: return interp_typed<float>(ctx, a, n_verts);
    case CTR_F64: return interp_typed<double>(ctx, a, n_verts);
    case CTR_U8: return interp_typed<uint8_t>(ctx, a, n_verts);
    case CTR_I16: return interp_typed<int16_t>(ctx, a, n_verts);
    case CTR_U16: return interp_typed<uint16_t>(ctx, a, n_verts);
  }
  return ctr_fail(ctx, CTR_ERR_BAD_ARG, "unknown dtype");
}

static int interp_check(ctr_ctx* ctx) {
  if (ctx->last_kind != 3 || !ctx->attr_ncomp) return ctr_fail(ctx, CTR_ERR_STATE, "no ctr_mt3d_interpolate since the last 3D run");
  return 0;
}

extern "C" int ctr_mt3d_interpolate_fetch(ctr_ctx* ctx, void* values) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!values) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  int rc = interp_check(ctx);
  if (rc) return rc;
  CTR_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t bytes = ctx->attr_rows * (size_t)ctx->attr_ncomp * ((ctx->last_flags & CTR_GEOM_F64) ? 8 : 4);
  if (bytes) CTR_CUDA(ctx, cudaMemcpyAsync(values, ctx->aux[43].p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CTR_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int ctr_mt3d_interpolate_device_ptr(ctr_ctx* ctx, void** values) {
  if (!ctx) return CTR_ERR_BAD_ARG;
  if (!values) return ctr_fail(ctx, CTR_ERR_BAD_ARG, "null argument");
  int rc = interp_check(ctx);
  if (rc) return rc;
  *values = ctx->aux[43].p;
  return 0;
}
