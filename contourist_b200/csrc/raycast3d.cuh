// First hits of rays on the 3D device mesh (ctr_mt3d_raycast): the linear BVH of closest3d.cuh (cq_build, rebuilt on
// every call) and one nearest-hit descent per ray.
//
// Included into mesh3d.cu inside its anonymous namespace, after closest3d.cuh.  The definition is
// oracle/mt3d_raycast.py:raycast: Woop, Benthin and Wald's watertight ray/triangle test (JCGT 2013) in fp64, one
// fixed-order formula with __dadd_rn / __dmul_rn / __ddiv_rn (nothing contracts), a hit only when its point lies in the
// triangle's padded box, and the winner the smallest (t, triangle index), so the device result equals it bit for bit.
//   k_ray_check : thread per ray (device rays): a non-finite coordinate or an all-zero direction raises the query flag
//                 of the counters, read at cq_build's host wait, so every error is reported before anything is written;
//   k_ray_query : thread per ray: near child first (by the entry t of the child boxes, the left child on a tie), the
//                 stack in shared memory; `best` starts at t_max with triangle INT32_MAX, so a hit at t_max is found.
// Pruning is conservative (DESIGN.md, "Ray casting", has the proof).  A hit's computed point p lies in its padded box
// (step 7 of the definition), so in its fp32 leaf box and every ancestor's.  For a box [L, H] on axis k the exact
// o_k + t d_k of such a hit is within E = 2^-52 (2M + |o_k|) + 2^-1073 of p_k (M: the largest |coordinate| of the root's
// boxes), so t lies in the exact slab of [L - E, H + E].  The computed slab ends fl(fl(L inv_k) - oi_k), with
// inv_k = fl(1/d_k) and oi_k = fl(o_k inv_k), are within 2^-51 (M + |o_k|) |1/d_k| of the exact ones; each end moves out
// by sg_k = (2^-49 (M + |o_k|) + 2^-1020) |inv_k| + 2^-1000, twice the sum of both bounds, which also covers the
// rounding of sg_k and of the subtraction.  An axis with d_k == 0 has p_k == o_k exactly and tests o_k against [L, H];
// an axis whose products could overflow ((M + |o_k|) |inv_k| > 2^1000) is not used for pruning.  A child is skipped
// only when max(entries, t_min) > min(exits, best), so no box holding a hit with t <= best (a tie too) is skipped.
// Results: AUX_RAY_RESULT (t, weights, point, triangle, side).  Staged host rays: AUX_RAY_INPUT (origins, directions).

struct RaySlab {                                       // per ray, the slab test's constants of one axis
  double inv, oi, sg;                                  // d_k == 0: inv = oi = 0, sg = NaN (o_k is tested against the box)
};

template <typename R>
__global__ void __launch_bounds__(256) k_ray_check(const R* __restrict__ org, const R* __restrict__ dir, unsigned n,
                                                   CqCounters* ctr) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool ok = true, moves = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const R o = org[(size_t)i * 3 + k], d = dir[(size_t)i * 3 + k];
    ok = ok && isfinite(o) && isfinite(d);
    moves = moves || d != (R)0;
  }
  if (!(ok && moves)) ctr->bad_points = 1u;
}

__device__ __forceinline__ double rc_pick(int k, D3 v) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }

struct RayShear {                                      // step 1 of the definition
  int kx, ky, kz;
  double sx, sy, sz;
};

__device__ __forceinline__ RayShear rc_shear(D3 d) {
  const double ax = fabs(d.x), ay = fabs(d.y), az = fabs(d.z);
  RayShear s;
  s.kz = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);   // the largest |d_k|, the first on a tie
  s.kx = s.kz == 2 ? 0 : s.kz + 1;
  s.ky = s.kx == 2 ? 0 : s.kx + 1;
  const double dz = rc_pick(s.kz, d);
  if (dz < 0.0) {
    const int k = s.kx;
    s.kx = s.ky;
    s.ky = k;
  }
  s.sx = __ddiv_rn(rc_pick(s.kx, d), dz);
  s.sy = __ddiv_rn(rc_pick(s.ky, d), dz);
  s.sz = __ddiv_rn(1.0, dz);
  return s;
}

struct RayHit {
  double t, u, v, w, det;
  D3 p;
};

// steps 2-7 of the definition for ray (o, d) and triangle (a, b, c): true on a hit with t_min <= t <= t_max
__device__ __forceinline__ bool rc_triangle(D3 o, D3 d, const RayShear& s, D3 a, D3 b, D3 c, double t_min, double t_max,
                                            RayHit& h) {
  const D3 A = d3_sub(a, o), B = d3_sub(b, o), C = d3_sub(c, o);
  const double az = rc_pick(s.kz, A), bz = rc_pick(s.kz, B), cz = rc_pick(s.kz, C);
  const double ax = __dsub_rn(rc_pick(s.kx, A), __dmul_rn(s.sx, az)), ay = __dsub_rn(rc_pick(s.ky, A), __dmul_rn(s.sy, az));
  const double bx = __dsub_rn(rc_pick(s.kx, B), __dmul_rn(s.sx, bz)), by = __dsub_rn(rc_pick(s.ky, B), __dmul_rn(s.sy, bz));
  const double cx = __dsub_rn(rc_pick(s.kx, C), __dmul_rn(s.sx, cz)), cy = __dsub_rn(rc_pick(s.ky, C), __dmul_rn(s.sy, cz));
  const double U = __dsub_rn(__dmul_rn(cx, by), __dmul_rn(cy, bx));
  const double V = __dsub_rn(__dmul_rn(ax, cy), __dmul_rn(ay, cx));
  const double W = __dsub_rn(__dmul_rn(bx, ay), __dmul_rn(by, ax));
  if ((U < 0.0 || V < 0.0 || W < 0.0) && (U > 0.0 || V > 0.0 || W > 0.0)) return false;
  const double det = __dadd_rn(__dadd_rn(U, V), W);
  if (det == 0.0) return false;
  const double T = __dadd_rn(__dadd_rn(__dmul_rn(U, __dmul_rn(s.sz, az)), __dmul_rn(V, __dmul_rn(s.sz, bz))),
                             __dmul_rn(W, __dmul_rn(s.sz, cz)));
  const double t = __ddiv_rn(T, det);
  if (!(t_min <= t && t <= t_max)) return false;
  const D3 p = d3_axpy(o, t, d);
  const double lo[3] = {fmin(fmin(a.x, b.x), c.x), fmin(fmin(a.y, b.y), c.y), fmin(fmin(a.z, b.z), c.z)};
  const double hi[3] = {fmax(fmax(a.x, b.x), c.x), fmax(fmax(a.y, b.y), c.y), fmax(fmax(a.z, b.z), c.z)};
  double m = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) m = fmax(m, fmax(fabs(lo[k]), fabs(hi[k])));
  const double pad = __dmul_rn(m, 0x1p-40);
  const double pk[3] = {p.x, p.y, p.z};
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (!(__dsub_rn(lo[k], pad) <= pk[k] && pk[k] <= __dadd_rn(hi[k], pad))) return false;
  h.t = t;
  h.u = U;
  h.v = V;
  h.w = W;
  h.det = det;
  h.p = p;
  return true;
}

// one axis of the slab test: the entry and exit t of [L, H], widened by sg; d_k == 0 (sg NaN): o_k against [L, H]
__device__ __forceinline__ void rc_slab(const RaySlab& s, double o, float L, float H, double& tn, double& tf) {
  const double l = (double)L, h = (double)H;
  const double tl = __dsub_rn(__dmul_rn(l, s.inv), s.oi), th = __dsub_rn(__dmul_rn(h, s.inv), s.oi);
  const double sg = s.sg == s.sg ? s.sg : (l <= o && o <= h ? INFINITY : -INFINITY);
  tn = fmax(tn, __dsub_rn(fmin(tl, th), sg));
  tf = fmin(tf, __dadd_rn(fmax(tl, th), sg));
}

// the entry t of box (lo, hi) when some hit with t in [t_min, best] may lie in it, else NaN
__device__ __forceinline__ double rc_box(const RaySlab* sl, D3 o, double t_min, double best, float lx, float ly, float lz,
                                         float hx, float hy, float hz) {
  double tn = t_min, tf = best;
  rc_slab(sl[0], o.x, lx, hx, tn, tf);
  rc_slab(sl[1], o.y, ly, hy, tn, tf);
  rc_slab(sl[2], o.z, lz, hz, tn, tf);
  return tn <= tf ? tn : NAN;
}

__device__ __forceinline__ RaySlab rc_axis(double o, double d, double M) {
  RaySlab s;
  if (d == 0.0) {
    s.inv = s.oi = 0.0;
    s.sg = NAN;
    return s;
  }
  s.inv = __ddiv_rn(1.0, d);
  const double w = __dmul_rn(__dadd_rn(M, fabs(o)), fabs(s.inv));
  if (!(w <= 0x1p1000)) {                              // the products could overflow: no pruning on this axis
    s.inv = s.oi = 0.0;
    s.sg = INFINITY;
    return s;
  }
  s.oi = __dmul_rn(o, s.inv);
  s.sg = __dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(M, fabs(o)), 0x1p-49), 0x1p-1020), fabs(s.inv)), 0x1p-1000);
  return s;
}

template <typename R>
__device__ __forceinline__ D3 rc_load(const R* __restrict__ x, unsigned i) {
  return {(double)x[(size_t)i * 3], (double)x[(size_t)i * 3 + 1], (double)x[(size_t)i * 3 + 2]};
}

template <typename G>
__device__ __forceinline__ bool rc_tri_at(const G* __restrict__ verts, const int* __restrict__ tris, int t, D3 o, D3 d,
                                          const RayShear& s, double t_min, double t_max, RayHit& h) {
  const int* tv = tris + (size_t)t * 3;
  return rc_triangle(o, d, s, cq_vertex(verts, __ldg(tv)), cq_vertex(verts, __ldg(tv + 1)), cq_vertex(verts, __ldg(tv + 2)),
                     t_min, t_max, h);
}

template <typename G, typename R>
__global__ void __launch_bounds__(CQ_THREADS) k_ray_query(const R* __restrict__ org, const R* __restrict__ dir, unsigned nr,
                                                          const CqNode* __restrict__ node, int root,
                                                          const G* __restrict__ verts, const int* __restrict__ tris,
                                                          double t_min, double t_max, double* __restrict__ t_out,
                                                          double* __restrict__ wt_out, double* __restrict__ pt_out,
                                                          int* __restrict__ tri_out, signed char* __restrict__ side_out,
                                                          CqCounters* ctr) {
  __shared__ int s_stack[CQ_STACK * CQ_THREADS];       // entry e of thread x at e * CQ_THREADS + x: no bank conflicts
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  bool found = false;
  if (i < nr) {
    const D3 o = rc_load(org, i), d = rc_load(dir, i);
    const RayShear sh = rc_shear(d);
    double best = t_max;
    int bt = 0x7fffffff;
    if (root >= 0) {
      // M: the largest |coordinate| of the root's two child boxes, which hold every box of the tree
      const float4* nd = reinterpret_cast<const float4*>(node + root);
      const float4 a = __ldg(nd), b = __ldg(nd + 1), c = __ldg(nd + 2);
      const float m = fmaxf(fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))),
                                  fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w)))),
                            fmaxf(fmaxf(fabsf(c.x), fabsf(c.y)), fmaxf(fabsf(c.z), fabsf(c.w))));
      const RaySlab sl[3] = {rc_axis(o.x, d.x, (double)m), rc_axis(o.y, d.y, (double)m), rc_axis(o.z, d.z, (double)m)};
      int* stk = s_stack + threadIdx.x;
      int sp = 0, cur = root;
      while (true) {
        if (cur >= 0) {
          const float4* q = reinterpret_cast<const float4*>(node + cur);
          const float4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
          const int4 e = __ldg(reinterpret_cast<const int4*>(q + 3));
          const double tl = rc_box(sl, o, t_min, best, a.x, a.y, a.z, a.w, b.x, b.y);
          const double tr = rc_box(sl, o, t_min, best, b.z, b.w, c.x, c.y, c.z, c.w);
          const bool vl = tl == tl, vr = tr == tr;
          if (vl && vr) {
            const bool rfirst = tr < tl;
            stk[sp * CQ_THREADS] = rfirst ? e.x : e.y;
            ++sp;
            cur = rfirst ? e.y : e.x;
            continue;
          }
          if (vl || vr) {
            cur = vl ? e.x : e.y;
            continue;
          }
        } else {
          const int t = ~cur;
          RayHit h;
          if (rc_tri_at(verts, tris, t, o, d, sh, t_min, best, h) && (h.t < best || t < bt)) {
            best = h.t;
            bt = t;
          }
        }
        if (sp == 0) break;
        --sp;
        cur = stk[sp * CQ_THREADS];
      }
    } else if (root != CQ_EMPTY) {                     // one triangle: the root is its leaf
      RayHit h;
      if (rc_tri_at(verts, tris, 0, o, d, sh, t_min, best, h)) {
        best = h.t;
        bt = 0;
      }
    }
    found = bt != 0x7fffffff;
    RayHit h;                                          // the winner again, for its weights, point and side
    if (found) rc_tri_at(verts, tris, bt, o, d, sh, t_min, best, h);
    t_out[i] = found ? best : INFINITY;
    tri_out[i] = found ? bt : -1;
    wt_out[(size_t)i * 3] = found ? __ddiv_rn(h.u, h.det) : NAN;
    wt_out[(size_t)i * 3 + 1] = found ? __ddiv_rn(h.v, h.det) : NAN;
    wt_out[(size_t)i * 3 + 2] = found ? __ddiv_rn(h.w, h.det) : NAN;
    pt_out[(size_t)i * 3] = found ? h.p.x : NAN;
    pt_out[(size_t)i * 3 + 1] = found ? h.p.y : NAN;
    pt_out[(size_t)i * 3 + 2] = found ? h.p.z : NAN;
    side_out[i] = found ? (h.det > 0.0 ? 1 : -1) : 0;
  }
  const unsigned f = __ballot_sync(0xffffffffu, found);
  if (lane_id() == 0 && f) atomicAdd(&ctr->n_found, (unsigned)__popc(f));
}

template <typename G, typename R>
int raycast_run(ctr_ctx* ctx, const ctr_ray_params* rp, const R* org, const R* dir, ctr_ray_counts* out) {
  cudaStream_t st = ctx->stream;
  const size_t nT = (size_t)ctx->last_counts[1], nR = (size_t)rp->n_rays;
  const int* tris = (const int*)ctx->tris.p;
  const G* verts = (const G*)ctx->verts.p;
  const bool on_device = rp->flags & CTR_FIELD_ON_DEVICE;
  CqTree tr;
  int rc;
  if ((rc = cq_build<G>(ctx, [&](CqCounters* ctr) -> int64_t {
         if (!on_device || !nR) return 0;
         k_ray_check<R><<<(unsigned)((nR + 255) / 256), 256, 0, st>>>(org, dir, (unsigned)nR, ctr);
         return 1;
       }, "rays must be finite with a non-zero direction", &tr)))
    return rc;
  double *t_out, *wt_out, *pt_out;
  int* tri_out;
  signed char* side_out;
  if ((rc = ctr_carve_buf(ctx, ctx->aux[AUX_RAY_RESULT], [&](ctr_carve& c) {
         c(t_out, nR * 8);
         c(wt_out, nR * 24);
         c(pt_out, nR * 24);
         c(tri_out, nR * 4);
         c(side_out, nR);
       })))
    return rc;
  if (nR) {
    k_ray_query<G, R><<<(unsigned)((nR + CQ_THREADS - 1) / CQ_THREADS), CQ_THREADS, 0, st>>>(
        org, dir, (unsigned)nR, tr.node, tr.root, verts, tris, rp->t_min, rp->t_max, t_out, wt_out, pt_out, tri_out,
        side_out, tr.ctr);
    ctx->launches++;
  }
  CTR_CUDA(ctx, cudaGetLastError());
  CqCounters& h = tr.h;
  CTR_CUDA(ctx, cudaMemcpyAsync(&h, tr.ctr, sizeof h, cudaMemcpyDeviceToHost, st));
  CTR_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->ray_n = (int64_t)nR;
  out->n_hit = h.n_found;
  out->height = nT > 1 ? (int64_t)h.height : 0;
  return 0;
}

template <typename G>
int raycast_typed(ctr_ctx* ctx, const ctr_ray_params* rp, ctr_ray_counts* out) {
  const size_t nR = (size_t)rp->n_rays, rsz = rp->dtype == CTR_F64 ? 8 : 4, bytes = nR * 3 * rsz;
  const void *org = rp->origins, *dir = rp->directions;
  if (!(rp->flags & CTR_FIELD_ON_DEVICE) && nR) {      // host rays: staged in their own type, origins then directions
    if (int rc = ctr_ensure(ctx, ctx->aux[AUX_RAY_INPUT], 2 * bytes)) return rc;
    char* buf = (char*)ctx->aux[AUX_RAY_INPUT].p;
    CTR_CUDA(ctx, cudaMemcpyAsync(buf, org, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CTR_CUDA(ctx, cudaMemcpyAsync(buf + bytes, dir, bytes, cudaMemcpyHostToDevice, ctx->stream));
    org = buf;
    dir = buf + bytes;
  }
  if (rp->dtype == CTR_F64) return raycast_run<G, double>(ctx, rp, (const double*)org, (const double*)dir, out);
  return raycast_run<G, float>(ctx, rp, (const float*)org, (const float*)dir, out);
}
