"""Cost of Taubin smoothing (ctr_mt3d_smooth) on the headline 512^3 surface, in one run.

    python tools/bench_smooth.py [--n 512] [--calls 10] [--out FILE]

The meshes: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in
fp64 geometry; and the mask (ct_like(n) > 0.5) as uint8 at isovalue 0.5 (the staircase surface smoothing is for), fp32
geometry, WANT_NORMALS.  Smoothing moves vertices and leaves the topology alone, so every timed call runs on the same
mesh, one call after the other (the positions keep being smoothed; the work per call does not depend on them).  CUDA
events on the engine's stream bracket one ctr_mt3d_smooth call (synchronous: the time includes its launches and its two
waits for the counters).  Reported per mesh:
  setup_ms     median call time at iterations=0 (edge table, fixed vertices, degrees and their scan; nothing written)
  call10_ms    median call time at 10 iterations (lambda 0.5, mu -0.53: 20 steps, then the store and the normals)
  step_us      (t(20) - t(0)) / 40 with the medians of 20 and 0 iterations (this also spreads the CSR build, the store
               and the normals over the steps: an upper bound on one step)
  step_bytes   what one step reads and writes by the shapes if the neighbour rows hit in L2: its CSR offsets, neighbour
               ids, own fp64 row and written row; step_gbs = step_bytes / step_us
  kernel_us    device time per launch of the pass's kernels and copies (torch.profiler, a pass of its own, 10 iterations)
  equal        positions and counts equal oracle/mt3d_smooth.py:smooth at 2 iterations on the fetched mesh (checked once,
               before the timed calls), normals within 2e-6 (fp32) / 1e-9 rad (fp64) of oracle/mt3d_smooth.py:normals
Prints one JSON line (also written to --out).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, normals_close, per_call  # noqa: E402


def step_bytes(nv, n_free, total_deg):
    "one Jacobi step, neighbour rows assumed in L2: offsets of every vertex, ids and rows of the free vertices"
    return (nv + 1) * 4 + total_deg * 4 + n_free * 24 * 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_smooth
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    mask = (field > 0.5).to(torch.uint8)
    eng, stream = cuda_engine()

    res = dict(tool="bench_smooth", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0),
               lam=0.5, mu=-0.53)
    meshes = [("ct_like_fp32", field, np.float32, E.WANT_NORMALS | E.WANT_KEYS),
              ("ct_like_fp64", field, np.float32, E.WANT_NORMALS | E.WANT_KEYS | E.GEOM_F64),
              ("mask_uint8_fp32", mask, np.uint8, E.WANT_NORMALS)]
    for name, f, dt, flags in meshes:
        eng.mt3d_run(f.data_ptr(), 0.5, shape=shape, dtype=dt, flags=flags)
        pre = eng.mt3d_fetch()
        c = eng.mt3d_smooth(2)
        out = eng.mt3d_fetch()
        want, cnt = mt3d_smooth.smooth(pre["verts"], pre["tris"], 2, 0.5, -0.53)
        geom64 = bool(flags & E.GEOM_F64)
        equal = bool(out["verts"].tobytes() == want.tobytes() and (c.n_edges, c.n_fixed_verts) ==
                     (cnt["n_edges"], cnt["n_fixed_verts"]) and np.array_equal(out["tris"], pre["tris"]) and
                     normals_close(out["normals"], mt3d_smooth.normals(want, pre["tris"], pre["normals"]), want,
                                   pre["tris"], geom64))
        off, nbr, fixed, _ = mt3d_smooth.neighbours(len(pre["verts"]), pre["tris"])
        nv, nt, n_free = len(pre["verts"]), len(pre["tris"]), int((~fixed).sum())
        del pre, out, want, off, fixed
        t0, t10, t20 = (per_call(stream, lambda: eng.mt3d_smooth(it), args.calls, 2) for it in (0, 10, 20))
        kernel_us = kernel_table(lambda: eng.mt3d_smooth(10), ("k_s_", "k_m_", "Memcpy", "Memset"))
        step_us = (float(np.median(t20)) - float(np.median(t0))) / 40 * 1000
        sb = step_bytes(nv, n_free, len(nbr))
        res[name] = dict(n_verts=nv, n_tris=nt,
                         n_edges=int(c.n_edges), n_fixed_verts=int(c.n_fixed_verts),
                         setup_ms=round(float(np.median(t0)), 4), call10_ms=round(float(np.median(t10)), 4),
                         call20_ms=round(float(np.median(t20)), 4), step_us=round(step_us, 2),
                         calls_ms=dict(it0=[round(x, 4) for x in t0], it10=[round(x, 4) for x in t10],
                                       it20=[round(x, 4) for x in t20]),
                         step_bytes=sb, step_gbs=round(sb / step_us / 1e3, 1), kernel_us=kernel_us, equal=equal)
        del nbr
    emit(res, args.out)


if __name__ == "__main__":
    main()
