"""Cost of ray casts (ctr_mt3d_raycast) on the headline 512^3 surface, in one run.

    python tools/bench_raycast.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry.  The cases, each one call (the tree is built by every call):
  one_ray     1 random ray from inside the box: mostly the build of the tree;
  camera_1k   the 1024 x 1024 primary rays of a pinhole camera outside the box, aimed at its centre (host fp64 rays):
              coherent rays, a depth image and a triangle-id image of the surface;
  random_1m   1 M rays with uniform random origins in the box [0, n-1]^3 and random directions (host fp64): incoherent;
  thickness   every vertex along its normal, origins and directions the engine's own device arrays (mt3d_device_ptrs)
              in the geometry type, t_min = 1e-3 voxels: the wall thickness of the bright object (the normals point up
              the field, into it).
Reported per geometry and case:
  n_rays, n_hit, height
  call_ms     median of --calls calls (one untimed call first; CUDA events on the engine's stream around the call, which
              ends in a host wait and the fetch of every result to host memory, so launches, host copies and waits are
              included)
  kernel_us   device time per launch of the pass's kernels (the tree's, the sort's CUB kernels included) and copies
              (torch.profiler, one call of its own)
  equal       t, triangle, weights, point, side equal oracle/mt3d_raycast.py:raycast (pruned) on 200 sampled rays of
              the case (checked before the timed calls)
  thickness   for thickness: the hit share and the median thickness (t of the rays that hit, in voxels; the normals are
              unit length)
Prints one JSON line (also written to --out).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, per_call  # noqa: E402


def camera_rays(n, res):
    "a res x res pinhole camera outside the box [0, n-1]^3, aimed at its centre (about a 48 degree field of view)"
    c = np.full(3, (n - 1) / 2)
    eye = c + np.array([1.3, 0.9, 0.7]) * n
    fwd = (c - eye) / np.linalg.norm(c - eye)
    right = np.cross(fwd, [0.0, 0.0, 1.0])
    right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    s = (np.arange(res) + 0.5) / res * 2 - 1
    U, V = np.meshgrid(s, s, indexing="xy")
    D = fwd + 0.45 * (U.reshape(-1, 1) * right + V.reshape(-1, 1) * up)
    return np.ascontiguousarray(np.broadcast_to(eye, D.shape)), np.ascontiguousarray(D)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_raycast
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    eng, stream = cuda_engine()
    rng = np.random.default_rng(0)
    Oc, Dc = camera_rays(n, 1024)
    host_cases = {"one_ray": (rng.uniform(0, n - 1, (1, 3)), rng.normal(size=(1, 3))), "camera_1k": (Oc, Dc),
                  "random_1m": (rng.uniform(0, n - 1, (1 << 20, 3)), rng.normal(size=(1 << 20, 3)))}
    t_thick = 1e-3

    res = dict(tool="bench_raycast", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag
        gd = np.float64 if gflag else np.float32
        c0 = eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)
        mesh = eng.mt3d_fetch()
        nv = len(mesh["verts"])

        def thickness():
            v, nrm, _ = eng.mt3d_device_ptrs()
            return eng.mt3d_raycast(v, nrm, t_thick, n=nv, dtype=gd)

        cases = {k: (lambda o=o, d=d: eng.mt3d_raycast(o, d)) for k, (o, d) in host_cases.items()}
        cases["thickness"] = thickness
        for cname, call in cases.items():
            got, c = call()                                     # the check: the definition on sampled rays of the case
            if cname == "thickness":
                O, D, t_min = mesh["verts"], mesh["normals"], t_thick
            else:
                (O, D), t_min = host_cases[cname], 0.0
            idx = rng.integers(0, len(O), min(200, len(O)))
            want, _ = mt3d_raycast.raycast(mesh["verts"], mesh["tris"], O[idx], D[idx], t_min, prune=True)
            equal = all(np.array_equal(got[k][idx], want[k], equal_nan=True) for k in want)
            extra = dict(n_rays=len(O), n_hit=int(c.n_hit), height=int(c.height))
            if cname == "thickness":
                hit = got["triangle"] >= 0
                extra["thickness"] = dict(hit_share=round(float(hit.mean()), 4), median=float(np.median(got["t"][hit])),
                                          side_plus_share=round(float((got["side"][hit] == 1).mean()), 4))
            del got
            ms = per_call(stream, call, args.calls, 1)
            kernel_us = kernel_table(call, ("k_cq_", "k_ray_", "DeviceRadixSort", "Memcpy", "Memset"))
            res["%s_%s" % (gname, cname)] = dict(n_verts=int(c0.n_verts), n_tris=int(c0.n_tris),
                                                 call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms],
                                                 kernel_us=kernel_us, equal=bool(equal), **extra)
    emit(res, args.out)


if __name__ == "__main__":
    main()
