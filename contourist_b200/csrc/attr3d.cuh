// Per-vertex values of another field on the 3D mesh (ctr_mt3d_interpolate; included by mt3d.cu inside its namespace).
//
//   k_interp_attr : thread per vertex of the last run's mesh (device keys, in vertex order = owner-word order, so
//                   neighbouring lanes gather from neighbouring rows): the edge's two run samples give the ratio exactly
//                   as k_emit_verts computes it, the two attribute rows (ncomp samples each, vector loads where the
//                   rows are aligned) give value = a_low + ratio * (a_high - a_low) per component.
// Templated on the run's sample type and the geometry type only (10 kernels); the attribute's sample type and load
// width are uniform kernel parameters read through switches.

struct AttrSrc {
  const char* p;        // attribute samples, component-last [n0][n1][n2][ncomp]
  int dtype;            // ctr_dtype
  int ncomp;            // 1..4
  unsigned row_bytes;   // ncomp * sample size (<= 32)
  unsigned vw;          // bytes per load: the largest power of two <= 16 that divides row_bytes and the address of p
};

static inline size_t attr_sample_bytes(int dtype) {
  switch (dtype) {
    case CTR_F32: return 4;
    case CTR_F64: return 8;
    case CTR_U8: return 1;
    case CTR_I16:
    case CTR_U16: return 2;
  }
  return 0;
}

// the row at p (row_bytes bytes, p aligned to VW) as little-endian 32-bit words; w must start zeroed
template <int VW>
__device__ __forceinline__ void attr_load_row(const char* __restrict__ p, unsigned rb, uint32_t w[8]) {
#pragma unroll
  for (int s = 0; s < 32 / VW; ++s) {
    if ((unsigned)(s * VW) >= rb) break;
    if (VW == 16) {
      const uint4 q = __ldg((const uint4*)(p + s * 16));
      w[4 * s] = q.x; w[4 * s + 1] = q.y; w[4 * s + 2] = q.z; w[4 * s + 3] = q.w;
    } else if (VW == 8) {
      const uint2 q = __ldg((const uint2*)(p + s * 8));
      w[2 * s] = q.x; w[2 * s + 1] = q.y;
    } else if (VW == 4) {
      w[s] = __ldg((const unsigned int*)(p + s * 4));
    } else if (VW == 2) {
      w[s >> 1] |= (uint32_t)__ldg((const unsigned short*)(p + s * 2)) << (16 * (s & 1));
    } else {
      w[s >> 2] |= (uint32_t)__ldg((const unsigned char*)(p + s)) << (8 * (s & 3));
    }
  }
}

__device__ __forceinline__ void attr_load(const AttrSrc& a, long long pt, uint32_t w[8]) {
  const char* p = a.p + pt * (long long)a.row_bytes;
  switch (a.vw) {
    case 16: attr_load_row<16>(p, a.row_bytes, w); break;
    case 8: attr_load_row<8>(p, a.row_bytes, w); break;
    case 4: attr_load_row<4>(p, a.row_bytes, w); break;
    case 2: attr_load_row<2>(p, a.row_bytes, w); break;
    default: attr_load_row<1>(p, a.row_bytes, w); break;
  }
}

// component c of a loaded row, widened (or, for fp64 samples in fp32 mode, rounded) to the geometry type
template <typename G>
__device__ __forceinline__ G attr_comp(int dtype, const uint32_t w[8], int c) {
  switch (dtype) {
    case CTR_F32: return (G)__uint_as_float(w[c]);
    case CTR_F64: return (G)__hiloint2double((int)w[2 * c + 1], (int)w[2 * c]);
    case CTR_U8: return (G)((w[c >> 2] >> (8 * (c & 3))) & 255u);
    case CTR_I16: return (G)(int)(short)(w[c >> 1] >> (16 * (c & 1)));
    default: return (G)((w[c >> 1] >> (16 * (c & 1))) & 0xffffu);
  }
}

template <typename T, typename G>
__global__ void __launch_bounds__(256) k_interp_attr(const T* __restrict__ f, int n1, int n2, long long off, double value,
                                                     const unsigned long long* __restrict__ keys,
                                                     const uint8_t* __restrict__ lowmin, unsigned nV, AttrSrc a,
                                                     G* __restrict__ out) {
  const unsigned id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nV) return;
  const unsigned long long key = keys[id];
  const bool p_low = lowmin[id] != 0;
  const unsigned d = (unsigned)key & 7u;
  // key = global lin * 8 + d; off = plane_offset * n1 * n2 makes lin local to the run's array
  const long long p = (long long)(key >> 3) - off;
  const long long q = p + ((long long)((d >> 2) & 1u) * n1 + ((d >> 1) & 1u)) * n2 + (d & 1u);
  // the ratio of k_emit_verts (tetrahedral.py:476-487), orientation from lowmin
  const G fp = (G)f[p], fq = (G)f[q];
  const G flow = p_low ? fp : fq, fhigh = p_low ? fq : fp;
  const G den = fhigh - flow;
  const G ratio = (fabs((double)den) <= 1e-8) ? (G)0.5 : quot((G)value - flow, den);
  uint32_t wl[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u}, wh[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  attr_load(a, p_low ? p : q, wl);
  attr_load(a, p_low ? q : p, wh);
  G* o = out + (size_t)id * (unsigned)a.ncomp;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (c >= a.ncomp) break;
    const G al = attr_comp<G>(a.dtype, wl, c), ah = attr_comp<G>(a.dtype, wh, c);
    o[c] = add_rn(al, mul_rn(ratio, ah - al));
  }
}

template <typename T>
int interp_typed(ctr_ctx* ctx, const ctr_attr_params* ap, int64_t* n_verts) {
  const ctr_mt3d_params* p = (const ctr_mt3d_params*)ctx->last3_params;
  const size_t nV = (size_t)ctx->last_counts[0];
  const bool f64 = (ctx->last_flags & CTR_GEOM_F64) != 0;
  const size_t gsz = f64 ? 8 : 4;
  const size_t rb = attr_sample_bytes(ap->dtype) * (size_t)ap->ncomp;
  const size_t npts = (size_t)p->n0 * (size_t)p->n1 * (size_t)p->n2;
  cudaStream_t st = ctx->stream;
  int rc;
  const char* src;
  if (ap->flags & CTR_FIELD_ON_DEVICE) {
    src = (const char*)ap->field;
  } else {
    // a buffer of its own: ctx->field still holds the run's staged samples, which the ratio needs
    if ((rc = ctr_ensure(ctx, ctx->aux[42], npts * rb))) return rc;
    CTR_CUDA(ctx, cudaMemcpyAsync(ctx->aux[42].p, ap->field, npts * rb, cudaMemcpyHostToDevice, st));
    src = (const char*)ctx->aux[42].p;
  }
  if ((rc = ctr_ensure(ctx, ctx->aux[43], nV * (size_t)ap->ncomp * gsz))) return rc;
  AttrSrc a;
  a.p = src;
  a.dtype = ap->dtype;
  a.ncomp = ap->ncomp;
  a.row_bytes = (unsigned)rb;
  a.vw = 16;
  while (a.vw > 1 && ((rb % a.vw) != 0 || ((uintptr_t)src % a.vw) != 0)) a.vw >>= 1;
  const T* f = (p->flags & CTR_FIELD_ON_DEVICE) ? (const T*)p->field : (const T*)ctx->field.p;
  const long long off = p->plane_offset * p->n1 * p->n2;
  if (nV) {
    const unsigned nb = (unsigned)((nV + 255) / 256);
    if (f64)
      k_interp_attr<T, double><<<nb, 256, 0, st>>>(f, (int)p->n1, (int)p->n2, off, p->isovalue,
                                                    (const unsigned long long*)ctx->keys.p, (const uint8_t*)ctx->lowmin.p,
                                                    (unsigned)nV, a, (double*)ctx->aux[43].p);
    else
      k_interp_attr<T, float><<<nb, 256, 0, st>>>(f, (int)p->n1, (int)p->n2, off, p->isovalue,
                                                   (const unsigned long long*)ctx->keys.p, (const uint8_t*)ctx->lowmin.p,
                                                   (unsigned)nV, a, (float*)ctx->aux[43].p);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->attr_rows = nV;
  ctx->attr_ncomp = ap->ncomp;
  if (n_verts) *n_verts = (int64_t)nV;
  return 0;
}
