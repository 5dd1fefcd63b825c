"""Cost of quadric vertex-clustering decimation (ctr_mt3d_decimate) on the headline 512^3 surface, in one run.

    python tools/bench_decimate.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry; cells of 2, 4 and 8 voxels with origin 0.  Decimation edits the mesh, so every timed call runs on a fresh
extraction: the run is outside the timed window, which holds one ctr_mt3d_decimate call (CUDA events on the engine's
stream; synchronous: the time includes its launches and its three waits for counters).  Reported per geometry and cell:
  counts      n_verts / n_tris before, and DecimateCounts after
  call_ms     median of --calls calls (each on a fresh run; two untimed calls first); calls_ms every call
  kernel_us   device time per launch of the pass's kernels and copies (torch.profiler, a call of its own)
  equal       counts, triangles, keys and lowmin equal oracle/mt3d_decimate.py:decimate on the fetched mesh, positions
              within 1e-9 * cell (+ one fp32 spacing with fp32 geometry), normals within 2e-6 (fp32) / 1e-9 rad (fp64)
              of oracle/mt3d_smooth.py:normals (checked once, before the timed calls)
Prints one JSON line (also written to --out).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, normals_close, per_call  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_decimate, mt3d_smooth
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    eng, stream = cuda_engine()

    res = dict(tool="bench_decimate", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag
        geom64 = bool(gflag)

        def run():
            return eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)

        for cell in (2.0, 4.0, 8.0):
            c0 = run()
            pre = eng.mt3d_fetch()
            c = eng.mt3d_decimate(cell)
            out = eng.mt3d_fetch()
            want, tris, member, cnt = mt3d_decimate.decimate(pre["verts"], pre["tris"], cell)
            tol = 1e-9 * cell + (0 if geom64 else np.spacing(np.abs(want)).astype(np.float64))
            equal = bool(dict(n_verts=c.n_verts, n_tris=c.n_tris, n_clusters=c.n_clusters, n_collapsed=c.n_collapsed,
                              n_duplicate=c.n_duplicate) == cnt and np.array_equal(out["tris"], tris) and
                         np.array_equal(out["keys"], pre["keys"][member]) and
                         np.array_equal(out["lowmin"], pre["lowmin"][member]) and
                         out["verts"].shape == want.shape and
                         bool((np.abs(out["verts"].astype(np.float64) - want.astype(np.float64)) <= tol).all()) and
                         normals_close(out["normals"], mt3d_smooth.normals(out["verts"], tris, pre["normals"][member]),
                                       out["verts"], tris, geom64))
            del pre, out, want, tris, member
            ms = per_call(stream, lambda: eng.mt3d_decimate(cell), args.calls, 2, setup=run)
            kernel_us = kernel_table(lambda: eng.mt3d_decimate(cell),
                                     ("k_d_", "k_c_", "k_flag_scan", "k_sel_", "k_s_", "Memcpy", "Memset"), setup=run)
            res["%s_cell%d" % (gname, int(cell))] = dict(
                n_verts_in=int(c0.n_verts), n_tris_in=int(c0.n_tris), n_verts=int(c.n_verts), n_tris=int(c.n_tris),
                n_clusters=int(c.n_clusters), n_collapsed=int(c.n_collapsed), n_duplicate=int(c.n_duplicate),
                call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms], kernel_us=kernel_us,
                equal=equal)
    emit(res, args.out)


if __name__ == "__main__":
    main()
