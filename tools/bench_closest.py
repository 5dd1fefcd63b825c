"""Cost of closest-point queries (ctr_mt3d_closest) on the headline 512^3 surface, in one run.

    python tools/bench_closest.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry.  The cases, each one call (the tree is built by every call):
  one_point       1 random point in the box: mostly the build of the tree;
  random_1m       1 M uniform random points in the box [0, n-1]^3 (host fp64 points, copied in the call);
  lattice_128     the 128^3 = 2.1 M points of a lattice over the box (host fp64);
  surface_to_dec  the symmetric surface distance between the mesh and its decimate(cell=4) version, held by a second
                  context: the mesh's vertices against the decimated mesh and the decimated vertices against the mesh,
                  device points in the geometry type, both directions in the timed window.
Reported per geometry and case:
  n_points, n_found, height
  call_ms     median of --calls calls (one untimed call first; CUDA events on the engine's stream around the call, which
              ends in a host wait, so launches, host copies and waits are included)
  kernel_us   device time per launch of the pass's kernels (the sort's CUB kernels included) and copies (torch.profiler,
              one call of its own)
  equal       distance, triangle, point and n_found equal oracle/mt3d_closest.py:closest (pruned) on 400 sampled
              points of the case (checked before the timed calls)
  ssd         for surface_to_dec: the average symmetric surface distance and the 95th-percentile Hausdorff distance
Prints one JSON line (also written to --out).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, per_call  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_closest
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    eng, stream = cuda_engine()
    dec, _ = cuda_engine()
    rng = np.random.default_rng(0)
    g = np.linspace(0.0, n - 1.0, 128)
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    host_cases = {"one_point": rng.uniform(0, n - 1, (1, 3)), "random_1m": rng.uniform(0, n - 1, (1 << 20, 3)),
                  "lattice_128": lattice}

    res = dict(tool="bench_closest", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag
        gd = np.float64 if gflag else np.float32
        c0 = eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)
        dec.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)
        dec.mt3d_decimate(4.0)
        mesh, dmesh = eng.mt3d_fetch(), dec.mt3d_fetch()
        nv, ndv = len(mesh["verts"]), len(dmesh["verts"])

        def symmetric():
            a, ca = dec.mt3d_closest(eng.mt3d_device_ptrs()[0], n=nv, dtype=gd)
            b, cb = eng.mt3d_closest(dec.mt3d_device_ptrs()[0], n=ndv, dtype=gd)
            return a, b, ca, cb

        cases = {k: (lambda p=p: eng.mt3d_closest(p)) for k, p in host_cases.items()}
        cases["surface_to_dec"] = symmetric
        for cname, call in cases.items():
            # the check: the definition on sampled points of the case
            out = call()
            if cname == "surface_to_dec":
                a, b, ca, cb = out
                ia, ib = rng.integers(0, nv, 200), rng.integers(0, ndv, 200)
                wa, _ = mt3d_closest.closest(dmesh["verts"], dmesh["tris"], mesh["verts"][ia], prune=True)
                wb, _ = mt3d_closest.closest(mesh["verts"], mesh["tris"], dmesh["verts"][ib], prune=True)
                equal = all(np.array_equal(a[k][ia], wa[k], equal_nan=True) and np.array_equal(b[k][ib], wb[k], equal_nan=True)
                            for k in wa) and ca.n_found == nv and cb.n_found == ndv
                d = np.concatenate([a["distance"], b["distance"]])
                extra = dict(ssd=dict(assd=float(d.mean()), hd95=float(np.percentile(d, 95)),
                                      max=float(d.max())), n_points=nv + ndv, n_found=int(ca.n_found + cb.n_found),
                             height=[int(ca.height), int(cb.height)], n_tris_dec=len(dmesh["tris"]))
            else:
                got, c = out
                pts = host_cases[cname]
                idx = rng.integers(0, len(pts), min(400, len(pts)))
                want, _ = mt3d_closest.closest(mesh["verts"], mesh["tris"], pts[idx], prune=True)
                equal = all(np.array_equal(got[k][idx], want[k], equal_nan=True) for k in want) and c.n_found == len(pts)
                extra = dict(n_points=len(pts), n_found=int(c.n_found), height=int(c.height))
            del out
            ms = per_call(stream, call, args.calls, 1)
            kernel_us = kernel_table(call, ("k_cq_", "DeviceRadixSort", "Memcpy", "Memset"))
            res["%s_%s" % (gname, cname)] = dict(n_verts=int(c0.n_verts), n_tris=int(c0.n_tris),
                                                 call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms],
                                                 kernel_us=kernel_us, equal=bool(equal), **extra)
    emit(res, args.out)


if __name__ == "__main__":
    main()
