// Face-normal sums and per-vertex normals of a 3D device mesh, shared by the passes that move vertices: smoothing
// (smooth3d.cuh) and decimation (decimate3d.cuh).  Included by mesh3d.cu inside its anonymous namespace.  The definition is oracle/mt3d_smooth.py:normals (within rounding: the face normals are summed
// with atomics).
//   k_s_nsum : per triangle, cross(b - a, c - a) in fp64 added to its three corners (fp64 atomicAdd);
//   k_s_nfin : per vertex, the sum normalised, its sign chosen so that it does not point against the old normal; a zero
//              sum keeps the old normal.

template <typename G>
__device__ __forceinline__ void tri_corners(const G* __restrict__ verts, const int v[3], double p[3][3]) {
#pragma unroll
  for (int q = 0; q < 3; ++q)
#pragma unroll
    for (int a = 0; a < 3; ++a) p[q][a] = (double)verts[(size_t)v[q] * 3 + a];
}

constexpr int N_THREADS = 256;

template <typename G>
__global__ void __launch_bounds__(N_THREADS) k_s_nsum(const G* __restrict__ verts, const int* __restrict__ tris, unsigned nt,
                                                      double* __restrict__ sum) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  const int v[3] = {tris[(size_t)t * 3], tris[(size_t)t * 3 + 1], tris[(size_t)t * 3 + 2]};
  double p[3][3];
  tri_corners(verts, v, p);
  const double ux = __dsub_rn(p[1][0], p[0][0]), uy = __dsub_rn(p[1][1], p[0][1]), uz = __dsub_rn(p[1][2], p[0][2]);
  const double wx = __dsub_rn(p[2][0], p[0][0]), wy = __dsub_rn(p[2][1], p[0][1]), wz = __dsub_rn(p[2][2], p[0][2]);
  const double cx = __dsub_rn(__dmul_rn(uy, wz), __dmul_rn(uz, wy));
  const double cy = __dsub_rn(__dmul_rn(uz, wx), __dmul_rn(ux, wz));
  const double cz = __dsub_rn(__dmul_rn(ux, wy), __dmul_rn(uy, wx));
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    double* s = sum + (size_t)v[q] * 3;
    atomicAdd(s, cx);
    atomicAdd(s + 1, cy);
    atomicAdd(s + 2, cz);
  }
}

template <typename G>
__global__ void k_s_nfin(const double* __restrict__ sum, unsigned nv, G* __restrict__ normals) {
  const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const double sx = sum[(size_t)v * 3], sy = sum[(size_t)v * 3 + 1], sz = sum[(size_t)v * 3 + 2];
  if (sx == 0.0 && sy == 0.0 && sz == 0.0) return;    // no face normal here: the old normal stays
  const double len = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(sx, sx), __dmul_rn(sy, sy)), __dmul_rn(sz, sz)));
  double nx = __ddiv_rn(sx, len), ny = __ddiv_rn(sy, len), nz = __ddiv_rn(sz, len);
  G* o = normals + (size_t)v * 3;
  const double dot = __dadd_rn(__dadd_rn(__dmul_rn(nx, (double)o[0]), __dmul_rn(ny, (double)o[1])), __dmul_rn(nz, (double)o[2]));
  if (dot < 0.0) {                                    // keep pointing up the field, whatever the winding
    nx = -nx;
    ny = -ny;
    nz = -nz;
  }
  o[0] = (G)nx;
  o[1] = (G)ny;
  o[2] = (G)nz;
}
