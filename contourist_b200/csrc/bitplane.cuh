// Stage 1 shared by the 3D and 4D paths: scalar field -> low / near bitplanes (+ min / max, + dilated row flags).
// Rows are runs of the contiguous (last) axis; a row index decomposes as ((a*rb + b)*rc + c).
#pragma once
#include <math.h>
#include <string.h>

#include <algorithm>
#include <climits>
#include <limits>
#include <type_traits>

#include "common.cuh"

namespace {

struct MinMaxKeys {
  unsigned long long min_key, max_key;     // order-preserving encodings, combined with atomicMin / atomicMax
};

// exact n / d for 32-bit n, d via one 64-bit multiply-high (M = ceil(2^64 / d))
struct FastDiv {
  unsigned long long M;
  unsigned d;
  __host__ void init(unsigned dd) {
    d = dd;
    M = dd <= 1 ? 0ull : (~0ull / dd) + 1ull;
  }
  __device__ __forceinline__ unsigned div(unsigned n) const { return d <= 1 ? n : (unsigned)__umul64hi((unsigned long long)n, M); }
};

__device__ __forceinline__ unsigned long long order_key(double x) {
  unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// ------------------------------------------------------------------------------------------------
// Stage 1: field -> low bitplane (the only pass over the whole field; HBM-bound), plus the "any sample
// near the isovalue" flag and optional min/max.  Near words are written with the low words; a word
// that has a near sample also raises the (dilated) row flags that switch later stages to their exact paths.
//   k_bitplane_tma     : rows a multiple of 32 samples, field 16-byte aligned: the volume is one linear stream, staged
//                        through shared memory by TMA bulk copies (cp.async.bulk + mbarrier full/empty ring): one
//                        producer lane + 8 consumer warps per CTA.  float / double consumers read the staged samples
//                        bank-conflict-free and ballot straight into bit words; uint8 / int16 / uint16 consumers compare
//                        4 / 2 samples per register and assemble words from lane bit groups.
//   k_bitplane_generic : any shape (rows padded to whole words), one warp converts 32 samples per step.
// Both take float, double, uint8, int16 and uint16 samples.  Floats compare in T against thresholds<T>; integer samples
// compare in int against thresholds_int<T>, which give the fp64 predicates on the widened sample exactly.
// ------------------------------------------------------------------------------------------------
struct RowGeom {
  uint8_t* rowflag;
  uint32_t* wordflag;                      // optional (3D): per row, one bit per group of 2^wshift words, see flag_rows
  FastDiv divW, divRc, divRb;
  int rb, rc;                              // row = (a*rb + b)*rc + c   (3D: a = 0, b = i, c = j)
  int W, wshift;
};

// word `word` holds a near sample: flag every row whose 3x3(x3) row neighbourhood contains it.  The word flags say
// where in those rows: bit (w >> wshift) for the words w-1, w, w+1 (an edge or voxel of word w-1 reaches sample 0 of
// word w; the exact paths of word w+1 look back at sample 31 of word w), so that later stages take their exact path
// for 3 words of a flagged row, not for all of it.
__device__ __noinline__ void flag_rows(const RowGeom& rg, unsigned word) {
  const unsigned row = rg.divW.div(word);
  const unsigned ab = rg.divRc.div(row), c = row - ab * (unsigned)rg.rc;
  const unsigned a = rg.divRb.div(ab), b = ab - a * (unsigned)rg.rb;
  uint32_t m = 0;
  if (rg.wordflag) {
    const int w = (int)(word - row * (unsigned)rg.W);
    for (int q = max(w - 1, 0); q <= min(w + 1, rg.W - 1); ++q) m |= 1u << (q >> rg.wshift);
  }
  for (int da = 0; da < 3; ++da)
    for (int db = 0; db < 3; ++db)
      for (int dc = 0; dc < 3; ++dc)
        if ((int)a - da >= 0 && (int)b - db >= 0 && (int)c - dc >= 0) {
          const size_t r = ((size_t)(a - da) * rg.rb + (b - db)) * rg.rc + (c - dc);
          rg.rowflag[r] = 1;
          if (rg.wordflag) atomicOr(&rg.wordflag[r], m);
        }
}

// Float samples: f < thr is low, nlo <= f <= nhi is near (thresholds<T>).
template <typename T>
struct FloatThr {
  T thr, nlo, nhi;
};

// An integer sample f meets the fp64 predicates on its widened value exactly when it meets integer ones (IntThr, from
// thresholds_int on the host):   f < v  <=>  f < thr;   v - r <= f <= v + r  <=>  nlo <= f <= nhi.
struct IntThr {
  int thr;            // ceil(v) clamped to [min(T), max(T) + 1]
  int nlo, nhi;       // near samples, clipped to T's range; nlo > nhi: none
};

// What k_bitplane_generic compares a sample of type T in, and against: floats in T (fmin / fmax ignore NaN), integer
// samples in int.
template <typename T, bool FLOAT = std::is_floating_point<T>::value>
struct Stage1 {
  typedef T C;
  typedef FloatThr<T> Thr;
  static constexpr T TOP = INFINITY, BOTTOM = -INFINITY;      // identities of lo / hi
  __device__ static __forceinline__ T lo(T a, T b) { return fmin(a, b); }
  __device__ static __forceinline__ T hi(T a, T b) { return fmax(a, b); }
};
template <typename T>
struct Stage1<T, false> {
  typedef int C;
  typedef IntThr Thr;
  static constexpr int TOP = INT_MAX, BOTTOM = INT_MIN;
  __device__ static __forceinline__ int lo(int a, int b) { return min(a, b); }
  __device__ static __forceinline__ int hi(int a, int b) { return max(a, b); }
};

// One warp's min / max into the run's keys; lanes that saw no sample hold the identities (mn > mx).
template <typename T>
__device__ __forceinline__ void minmax_commit(T mn, T mx, MinMaxKeys* ctr) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane_id() == 0) {
    if (mn <= mx) {
      atomicMin(&ctr->min_key, order_key((double)mn));
      atomicMax(&ctr->max_key, order_key((double)mx));
    }
  }
}
__device__ __forceinline__ void minmax_commit(int mn, int mx, MinMaxKeys* ctr) {
  mn = __reduce_min_sync(0xffffffffu, mn);
  mx = __reduce_max_sync(0xffffffffu, mx);
  if (lane_id() == 0 && mn <= mx) {
    atomicMin(&ctr->min_key, order_key((double)mn));
    atomicMax(&ctr->max_key, order_key((double)mx));
  }
}

template <typename T, bool MINMAX>
__global__ void __launch_bounds__(256) k_bitplane_generic(const T* __restrict__ f, unsigned nrows, int n2, int W,
                                                          typename Stage1<T>::Thr th, uint32_t* __restrict__ bits,
                                                          uint32_t* __restrict__ nbits, RowGeom rg, MinMaxKeys* ctr) {
  typedef Stage1<T> S;
  typedef typename S::C C;
  constexpr int UNROLL = 4;
  ctr_pdl_enter();
  const unsigned lane = lane_id();
  const unsigned nwords = nrows * (unsigned)W;
  const unsigned warps = gridDim.x * (blockDim.x >> 5);
  unsigned g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  C mn = S::TOP, mx = S::BOTTOM;
  for (; g < nwords; g += warps * UNROLL) {
    C val[UNROLL];
    bool ok[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      unsigned gu = g + (unsigned)u * warps;
      ok[u] = false;
      val[u] = (C)0;
      if (gu < nwords) {
        unsigned row = gu / (unsigned)W;
        int k = (int)(gu - row * (unsigned)W) * 32 + (int)lane;
        if (k < n2) {
          ok[u] = true;
          val[u] = (C)__ldg(f + (size_t)row * n2 + k);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      unsigned gu = g + (unsigned)u * warps;
      if (gu < nwords) {                       // warp-uniform
        unsigned wl = __ballot_sync(0xffffffffu, ok[u] && (val[u] < th.thr));
        unsigned wn = __ballot_sync(0xffffffffu, ok[u] && (val[u] >= th.nlo) && (val[u] <= th.nhi));
        if (lane == 0) {
          bits[gu] = wl;
          nbits[gu] = wn;
          if (wn) flag_rows(rg, gu);
        }
        if (MINMAX && ok[u]) {
          mn = S::lo(mn, val[u]);
          mx = S::hi(mx, val[u]);
        }
      }
    }
  }
  minmax_commit(mn, mx, ctr);
}

// ---- TMA (bulk async copy) ring -------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LAB_DONE;\n"
      "bra LAB_WAIT;\n"
      "LAB_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// The field is read exactly once: its lines enter L2 marked evict-first, so that they do not push out the bitplanes this
// kernel writes (32 MiB that stage 2 reads right away) nor the dirty lines of the previous extraction's mesh.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}

constexpr int TMA_STAGES = 3;                      // x 16 KiB per CTA, 3 CTAs per SM: measured best of 1..6 x 2..6
constexpr int TMA_CTAS_PER_SM = 3;
constexpr int TMA_CHUNK = 16384;                   // bytes per stage
constexpr int TMA_CONSUMER_WARPS = 8;
constexpr int TMA_WARP_BYTES = TMA_CHUNK / TMA_CONSUMER_WARPS;   // a consumer warp's slice of a stage

// The consumer step of k_bitplane_tma, per sample type: load() copies the warp's slice of a stage into registers (the
// kernel releases the stage right after), step() turns them into the words word0 + [0, WPW) of the bitplanes, of
// which those below words_here (counted from the stage's first word) exist; commit() adds min / max to the run's.
template <typename T, bool MINMAX, bool FLOAT = std::is_floating_point<T>::value>
struct TmaConsumer {
  typedef FloatThr<T> Thr;
  static constexpr int NW = TMA_CHUNK / (32 * (int)sizeof(T));        // bit words per stage
  static constexpr int WPW = NW / TMA_CONSUMER_WARPS;                 // words per warp per stage (<= 32)
  static_assert(WPW >= 1 && WPW <= 32, "stage geometry");
  static constexpr int SCRATCH = TMA_CONSUMER_WARPS * 32 * 4;         // per-warp word staging, behind the barriers
  // registers for exactly TMA_CTAS_PER_SM CTAs per SM: with fewer, a fourth CTA fits, and CTAs that become resident
  // early (behind the previous kernel) crowd onto the SMs that free first (B200, 1000 W: 0.312 -> 0.356 ms per 512^3 step)
  static constexpr int MIN_CTAS = TMA_CTAS_PER_SM;
  uint32_t* swords;
  T vc, vr;
  T mn = INFINITY, mx = -INFINITY;
  T val[WPW];

  __device__ __forceinline__ TmaConsumer(const Thr& th, uint32_t* scratch) : swords(scratch) {
    // conservative centre / radius form of the hull test: |x - vc| <= vr  (superset of [nlo, nhi])
    vc = (T)0.5 * th.nlo + (T)0.5 * th.nhi;
    vr = (th.nhi - th.nlo) * (T)0.55 + fabs(vc) * (T)1e-6 + (T)1e-30;
  }
  __device__ __forceinline__ void load(const unsigned char* slice) {
    const T* sv = reinterpret_cast<const T*>(slice);
#pragma unroll
    for (int q = 0; q < WPW; ++q) val[q] = sv[q * 32 + lane_id()];   // conflict-free: lane <-> bank
  }
  __device__ __forceinline__ void step(const Thr& th, size_t word0, unsigned wbase, unsigned words_here, uint32_t* bits,
                                       uint32_t* nbits, const RowGeom& rg) {
    const unsigned lane = lane_id();
    if (words_here < (unsigned)NW) {
      // partial last chunk: samples past the end are stale shared memory.  NaN is neither low nor near, fmin / fmax
      // ignore it, and the words past the end are not stored.
#pragma unroll
      for (int q = 0; q < WPW; ++q)
        if (wbase + q >= words_here) val[q] = NAN;
    }
    T dist = INFINITY;
#pragma unroll
    for (int q = 0; q < WPW; ++q) {
      const unsigned wl = __ballot_sync(0xffffffffu, val[q] < th.thr);
      if (lane == 0) swords[q] = wl;
      dist = fmin(dist, fabs(val[q] - vc));                     // NaN never wins: not near
      if (MINMAX) {
        mn = fmin(mn, val[q]);
        mx = fmax(mx, val[q]);
      }
    }
    unsigned mine_n = 0;
    if (__any_sync(0xffffffffu, dist <= vr)) {                   // rare: materialise the near words of this warp
#pragma unroll
      for (int q = 0; q < WPW; ++q) {
        const unsigned wn = __ballot_sync(0xffffffffu, (val[q] >= th.nlo) && (val[q] <= th.nhi));
        if ((int)lane == q) {
          mine_n = wn;
          if (wn) flag_rows(rg, (unsigned)(word0 + q));
        }
      }
    }
    __syncwarp();
    if ((int)lane < WPW && wbase + lane < words_here) {
      bits[word0 + lane] = swords[lane];
      nbits[word0 + lane] = mine_n;
    }
    __syncwarp();
  }
  __device__ __forceinline__ void commit(MinMaxKeys* ctr) { minmax_commit(mn, mx, ctr); }
};

// SIMD view of one 32-bit register holding N = 4 (uint8) or 2 (int16 / uint16) samples.  Compares give 0 / all-ones
// per sample; pack() turns that into N bits, sample q at bit q; zeros() is non-zero iff some sample of t is 0 (the
// borrow can mark more samples than the zero ones, never a register without one).
template <typename T>
struct Simd;
template <>
struct Simd<uint8_t> {
  static constexpr int N = 4, MIN = 0, MAX = 255;
  __host__ __device__ static unsigned rep(int x) { return ((unsigned)x & 0xffu) * 0x01010101u; }
  __device__ static __forceinline__ unsigned lt(unsigned a, unsigned b) { return __vcmpltu4(a, b); }
  __device__ static __forceinline__ unsigned eq(unsigned a, unsigned b) { return __vcmpeq4(a, b); }
  __device__ static __forceinline__ unsigned mn(unsigned a, unsigned b) { return __vminu4(a, b); }
  __device__ static __forceinline__ unsigned mx(unsigned a, unsigned b) { return __vmaxu4(a, b); }
  __device__ static __forceinline__ unsigned pack(unsigned m) { return ((m & 0x08040201u) * 0x01010101u) >> 24; }
  __device__ static __forceinline__ unsigned zeros(unsigned t) { return (t - 0x01010101u) & ~t & 0x80808080u; }
  __device__ static __forceinline__ int hmin(unsigned m) {
    return (int)min(min(m & 0xffu, (m >> 8) & 0xffu), min((m >> 16) & 0xffu, m >> 24));
  }
  __device__ static __forceinline__ int hmax(unsigned m) {
    return (int)max(max(m & 0xffu, (m >> 8) & 0xffu), max((m >> 16) & 0xffu, m >> 24));
  }
};
template <>
struct Simd<uint16_t> {
  static constexpr int N = 2, MIN = 0, MAX = 65535;
  __host__ __device__ static unsigned rep(int x) { return ((unsigned)x & 0xffffu) * 0x00010001u; }
  // unsigned order = signed order with the sign bits flipped: one LOP3 in front of __vcmplts2 is shorter than __vcmpltu2
  __device__ static __forceinline__ unsigned lt(unsigned a, unsigned b) { return __vcmplts2(a ^ 0x80008000u, b ^ 0x80008000u); }
  __device__ static __forceinline__ unsigned eq(unsigned a, unsigned b) { return __vcmpeq2(a, b); }
  __device__ static __forceinline__ unsigned mn(unsigned a, unsigned b) { return __vminu2(a, b); }
  __device__ static __forceinline__ unsigned mx(unsigned a, unsigned b) { return __vmaxu2(a, b); }
  __device__ static __forceinline__ unsigned pack(unsigned m) { return ((m & 0x00020001u) * 0x00010001u) >> 16; }
  __device__ static __forceinline__ unsigned zeros(unsigned t) { return (t - 0x00010001u) & ~t & 0x80008000u; }
  __device__ static __forceinline__ int hmin(unsigned m) { return (int)min(m & 0xffffu, m >> 16); }
  __device__ static __forceinline__ int hmax(unsigned m) { return (int)max(m & 0xffffu, m >> 16); }
};
template <>
struct Simd<int16_t> : Simd<uint16_t> {
  static constexpr int MIN = -32768, MAX = 32767;
  __device__ static __forceinline__ unsigned lt(unsigned a, unsigned b) { return __vcmplts2(a, b); }
  __device__ static __forceinline__ unsigned mn(unsigned a, unsigned b) { return __vmins2(a, b); }
  __device__ static __forceinline__ unsigned mx(unsigned a, unsigned b) { return __vmaxs2(a, b); }
  __device__ static __forceinline__ int hmin(unsigned m) { return min((int)(short)(m & 0xffffu), (int)(short)(m >> 16)); }
  __device__ static __forceinline__ int hmax(unsigned m) { return max((int)(short)(m & 0xffffu), (int)(short)(m >> 16)); }
};

// Stage-1 thresholds of the TMA kernel for 1- and 2-byte samples, replicated into every sample slot of a register.
struct IntThrRep {
  unsigned thr;       // f < thr per sample (thr clamped to max(T)) ...
  unsigned lowall;    // ... or every sample is low (ceil(v) > max(T)): all ones
  unsigned near0, near1;  // the (at most two) near values
  int nnear;          // 0, 1 or 2
};

// uint8 / int16 / uint16: the consumers read 16 bytes (16 / 8 samples) per lane and load, compare 4 / 2 samples per
// instruction sequence (Simd<T>) and assemble each 32-bit word from the bit groups of 2 / 4 neighbouring lanes.  A
// warp's 2 KiB of a stage is 4 passes of 512 bytes: pass q, lane l has the samples of word q * WPP + l / GROUP, bits
// (l % GROUP) * S ...
template <typename T, bool MINMAX>
struct TmaConsumer<T, MINMAX, false> {
  typedef IntThrRep Thr;
  typedef Simd<T> V;
  static constexpr int S = 16 / (int)sizeof(T);                 // samples per lane and pass
  static constexpr int GROUP = 32 / S;                          // lanes per bit word
  static constexpr int WPP = 32 / GROUP;                        // words per warp and pass
  static constexpr int PASSES = TMA_WARP_BYTES / 512;
  static constexpr int WPW = PASSES * WPP;                      // words per warp per stage
  static_assert(PASSES * 512 == TMA_WARP_BYTES && WPW * 32 * (int)sizeof(T) == TMA_WARP_BYTES, "stage geometry");
  static constexpr int SCRATCH = 0;
  static constexpr int MIN_CTAS = 0;                             // no bound: ptxas picks the register count
  unsigned vmn = V::rep(V::MAX), vmx = V::rep(V::MIN);        // identities of V::mn / V::mx
  uint4 v[PASSES];

  __device__ __forceinline__ TmaConsumer(const Thr&, uint32_t*) {}
  __device__ __forceinline__ void load(const unsigned char* slice) {
    const uint4* sv = reinterpret_cast<const uint4*>(slice);
#pragma unroll
    for (int q = 0; q < PASSES; ++q) v[q] = sv[q * 32 + lane_id()];   // 16 bytes per lane: conflict-free
  }
  __device__ __forceinline__ void step(const Thr& th, size_t word0, unsigned wbase, unsigned words_here, uint32_t* bits,
                                       uint32_t* nbits, const RowGeom& rg) {
    const unsigned lane = lane_id(), sub = lane % GROUP;
    unsigned lo[PASSES], zacc = 0;
    bool ok[PASSES];
#pragma unroll
    for (int q = 0; q < PASSES; ++q) {
      // a partial last chunk: the words past its end are stale shared memory; their lanes contribute nothing
      ok[q] = wbase + q * WPP + lane / GROUP < words_here;
      const unsigned x[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
      unsigned b = 0, z = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        b |= V::pack(V::lt(x[e], th.thr) | th.lowall) << (e * V::N);
        if (th.nnear > 0) z |= V::zeros(x[e] ^ th.near0);
        if (th.nnear > 1) z |= V::zeros(x[e] ^ th.near1);
        if (MINMAX && ok[q]) {
          vmn = V::mn(vmn, x[e]);
          vmx = V::mx(vmx, x[e]);
        }
      }
      lo[q] = ok[q] ? b : 0u;
      if (ok[q]) zacc |= z;
    }
#pragma unroll
    for (int q = 0; q < PASSES; ++q) {
      unsigned wl = lo[q] << (S * sub);
#pragma unroll
      for (int o = 1; o < GROUP; o <<= 1) wl |= __shfl_xor_sync(0xffffffffu, wl, o);
      if (sub == 0 && ok[q]) bits[word0 + q * WPP + lane / GROUP] = wl;
    }
    unsigned nr[PASSES];
#pragma unroll
    for (int q = 0; q < PASSES; ++q) nr[q] = 0;
    if (__any_sync(0xffffffffu, zacc != 0)) {                   // some sample of this warp is near: materialise the words
#pragma unroll
      for (int q = 0; q < PASSES; ++q) {
        const unsigned x[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
        unsigned b = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          unsigned m = V::eq(x[e], th.near0);
          if (th.nnear > 1) m |= V::eq(x[e], th.near1);
          b |= V::pack(m) << (e * V::N);
        }
        unsigned wn = ok[q] ? b << (S * sub) : 0u;
#pragma unroll
        for (int o = 1; o < GROUP; o <<= 1) wn |= __shfl_xor_sync(0xffffffffu, wn, o);
        nr[q] = wn;
        if (sub == 0 && ok[q] && wn) flag_rows(rg, (unsigned)(word0 + q * WPP + lane / GROUP));
      }
    }
#pragma unroll
    for (int q = 0; q < PASSES; ++q)
      if (sub == 0 && ok[q]) nbits[word0 + q * WPP + lane / GROUP] = nr[q];
  }
  __device__ __forceinline__ void commit(MinMaxKeys* ctr) {
    int mn = INT_MAX, mx = INT_MIN;
    if (MINMAX) {
      mn = V::hmin(vmn);
      mx = V::hmax(vmx);
    }
    minmax_commit(mn, mx, ctr);
  }
};

// dynamic shared memory of k_bitplane_tma<T>: the ring, its full / empty barriers, the consumers' scratch
template <typename T>
constexpr int tma_smem_bytes() {
  return TMA_STAGES * TMA_CHUNK + 2 * TMA_STAGES * 8 + TmaConsumer<T, false>::SCRATCH;
}

template <typename T, bool MINMAX>
__global__ void __launch_bounds__((TMA_CONSUMER_WARPS + 1) * 32, TmaConsumer<T, MINMAX>::MIN_CTAS)
    k_bitplane_tma(const T* __restrict__ f, size_t nbytes, typename TmaConsumer<T, MINMAX>::Thr th, uint32_t* __restrict__ bits,
                   uint32_t* __restrict__ nbits, RowGeom rg, MinMaxKeys* ctr) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + TMA_STAGES * TMA_CHUNK);
  uint64_t* empty = full + TMA_STAGES;
  const unsigned warp = threadIdx.x >> 5, lane = lane_id();
  if (threadIdx.x == 0) {
    for (int s = 0; s < TMA_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], TMA_CONSUMER_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const unsigned nchunks = (unsigned)((nbytes + TMA_CHUNK - 1) / TMA_CHUNK);   // fewer than the (32-bit) word indices
  if (warp == TMA_CONSUMER_WARPS) {
    if (lane == 0) {
      unsigned it = 0;
      const uint64_t pol = l2_evict_first_policy();
      for (unsigned c = blockIdx.x; c < nchunks; c += gridDim.x, ++it) {
        const int s = it % TMA_STAGES;
        const unsigned ph = (it / TMA_STAGES) & 1u;
        mbar_wait(&empty[s], ph ^ 1u);                           // first round passes immediately
        const size_t off = c * (size_t)TMA_CHUNK;
        const unsigned bytes = (unsigned)((nbytes - off) < (size_t)TMA_CHUNK ? (nbytes - off) : (size_t)TMA_CHUNK);
        mbar_expect_tx(&full[s], bytes);
        tma_bulk_g2s(smem + s * TMA_CHUNK, reinterpret_cast<const unsigned char*>(f) + off, bytes, &full[s], pol);
      }
    }
    return;
  }
  TmaConsumer<T, MINMAX> cons(th, reinterpret_cast<uint32_t*>(empty + TMA_STAGES) + warp * 32);
  const unsigned wbase = warp * cons.WPW;
  unsigned it = 0;
  // The producer above starts fetching at once: the field is complete before the kernel in front of this one passed its
  // own wait (common.cuh, rule 2).  The consumers wait here, in front of their first write: the flags they set are
  // zeroed by that kernel, and the bit planes may still be read by the previous run's last kernel.
  ctr_pdl_enter();
  for (unsigned c = blockIdx.x; c < nchunks; c += gridDim.x, ++it) {
    const int s = it % TMA_STAGES;
    const unsigned ph = (it / TMA_STAGES) & 1u;
    const size_t off = c * (size_t)TMA_CHUNK;
    const unsigned bytes = (unsigned)((nbytes - off) < (size_t)TMA_CHUNK ? (nbytes - off) : (size_t)TMA_CHUNK);
    mbar_wait(&full[s], ph);
    cons.load(smem + s * TMA_CHUNK + warp * TMA_WARP_BYTES);
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);                       // stage is in registers: release it early
    cons.step(th, off / (32 * sizeof(T)) + wbase, wbase, bytes / (32u * (unsigned)sizeof(T)), bits, nbits, rg);
  }
  cons.commit(ctr);
}


double key_to_double(unsigned long long k) {
  unsigned long long u = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  double d;
  memcpy(&d, &u, 8);
  return d;
}

template <typename T>
void thresholds(double v, T& thr, T& nlo, T& nhi);

template <>
void thresholds<double>(double v, double& thr, double& nlo, double& nhi) {
  thr = v;
  double r = (1e-8 + 1e-5 * fabs(v)) * 1.0001;
  nlo = v - r;
  nhi = v + r;
}
template <>
void thresholds<float>(double v, float& thr, float& nlo, float& nhi) {
  thr = (float)v;                               // f < v  <=>  f < thr, thr = smallest float >= v
  if ((double)thr < v) thr = nextafterf(thr, INFINITY);
  double r = (1e-8 + 1e-5 * fabs(v)) * 1.0001;
  nlo = (float)(v - r);
  if ((double)nlo > v - r) nlo = nextafterf(nlo, -INFINITY);
  nhi = (float)(v + r);
  if ((double)nhi < v + r) nhi = nextafterf(nhi, INFINITY);
}

// Integer samples: the same predicates as thresholds<double> on the widened sample, as integer bounds (IntThr).
template <typename T>
IntThr thresholds_int(double v) {
  const double tmin = (double)std::numeric_limits<T>::min(), tmax = (double)std::numeric_limits<T>::max();
  IntThr t;
  const double c = ceil(v);                     // f < v  <=>  f < ceil(v) for integer f (v = +-inf included)
  t.thr = c > tmax ? (int)tmax + 1 : c < tmin ? (int)tmin : (int)c;
  const double r = (1e-8 + 1e-5 * fabs(v)) * 1.0001;
  const double a = ceil(std::max(v - r, tmin)), b = floor(std::min(v + r, tmax));
  // v - r or v + r is NaN for v = +-inf (inf - inf): no sample is near, as in the fp64 compare
  if (a <= b) {
    t.nlo = (int)a;
    t.nhi = (int)b;
  } else {
    t.nlo = 1;
    t.nhi = 0;
  }
  return t;
}

RowGeom row_geom(uint8_t* rowflag, uint32_t* wordflag, int W, int rb, int rc) {
  RowGeom rg;
  rg.rowflag = rowflag;
  rg.wordflag = wordflag;
  rg.W = W;
  rg.wshift = 0;
  while ((W >> rg.wshift) > 32) ++rg.wshift;
  rg.divW.init((unsigned)W);
  rg.divRc.init((unsigned)rc);
  rg.divRb.init((unsigned)rb);
  rg.rb = rb;
  rg.rc = rc;
  return rg;
}

// Stage 1 over float, double, uint8, int16 or uint16 samples.  The TMA kernel takes the field when it is one linear
// stream of whole words (rows a multiple of 32 samples, 16-byte aligned) and, for integer samples, at most two sample
// values are near; the generic kernel takes any other field.
template <typename T>
int launch_bitplane(ctr_ctx* ctx, const T* dfield, unsigned nrows, int n2, int W, int rb, int rc, double iso,
                    uint32_t* bits, uint32_t* nbits, uint8_t* rowflag, MinMaxKeys* dctr, bool minmax,
                    bool clear_rowflag = true, uint32_t* wordflag = nullptr) {
  static_assert(std::is_floating_point<T>::value || std::is_same<T, uint8_t>::value || std::is_same<T, int16_t>::value ||
                    std::is_same<T, uint16_t>::value,
                "samples: float, double, uint8, int16, uint16");
  cudaStream_t st = ctx->stream;
  bool tma = (n2 % 32 == 0) && (((uintptr_t)dfield) % 16 == 0);
  typename Stage1<T>::Thr th;
  typename TmaConsumer<T, false>::Thr tth;
  if constexpr (std::is_floating_point<T>::value) {
    thresholds<T>(iso, th.thr, th.nlo, th.nhi);
    tth = th;
  } else {
    th = thresholds_int<T>(iso);
    // the TMA consumers compare against at most two near values: always so for these types (r < 0.66 inside their range)
    tma = tma && (th.nlo > th.nhi || th.nhi - th.nlo <= 1);
    typedef Simd<T> V;
    const int tmax = (int)std::numeric_limits<T>::max();
    tth.thr = V::rep(std::min(th.thr, tmax));
    tth.lowall = th.thr > tmax ? 0xffffffffu : 0u;
    tth.nnear = th.nlo > th.nhi ? 0 : th.nhi - th.nlo + 1;
    tth.near0 = V::rep(th.nlo);
    tth.near1 = V::rep(th.nhi);
  }
  const RowGeom rg = row_geom(rowflag, wordflag, W, rb, rc);
  if (clear_rowflag) CTR_CUDA(ctx, cudaMemsetAsync(rg.rowflag, 0, (size_t)nrows, st));
  if (tma) {
    const auto kern = minmax ? k_bitplane_tma<T, true> : k_bitplane_tma<T, false>;
    constexpr int smem = tma_smem_bytes<T>();
    CTR_CUDA(ctx, ctr_smem_optin(ctx, kern, smem));
    const size_t nbytes = (size_t)nrows * n2 * sizeof(T);
    const size_t nchunks = (nbytes + TMA_CHUNK - 1) / TMA_CHUNK;
    const int blocks = (int)std::min<size_t>(nchunks, (size_t)ctx->sm_count * TMA_CTAS_PER_SM);
    ctr_launch_dep(kern, blocks, (TMA_CONSUMER_WARPS + 1) * 32, smem, st, dfield, nbytes, tth, bits, nbits, rg, dctr);
  } else {
    // 256 threads, 4 words per warp and round, at most 8 blocks per SM
    const size_t need = ((size_t)nrows * W + 8 * 4 - 1) / (8 * 4);
    const int blocks = (int)std::min<size_t>(std::max<size_t>(need, 1), (size_t)ctx->sm_count * 8);
    const auto kern = minmax ? k_bitplane_generic<T, true> : k_bitplane_generic<T, false>;
    ctr_launch_dep(kern, blocks, 256, 0, st, dfield, nrows, n2, W, th, bits, nbits, rg, dctr);
  }
  ctx->launches++;
  CTR_CUDA(ctx, cudaGetLastError());
  return 0;
}

}  // namespace
