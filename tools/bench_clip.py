"""Cost of clipping (ctr_mt3d_clip) the headline 512^3 surface, in one run.

    python tools/bench_clip.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry.  The cases: a plane along axis 0 through the middle (x = n/2 + 0.25), keep high and keep low; an oblique plane
(normal (1, 2, 3)) through the centre of the volume; a value clip on a second field (synthetic.turbulence, interpolated
on the mesh first) at the median of its vertex values; a box of six planes (x, y, z within [n/4, 3n/4]) clipped one
plane after the other, timed as a whole.  A clip edits the mesh, so every timed call runs on a fresh extraction (and,
for the value clip, a fresh interpolation); the window holds the clip calls only (CUDA events on the engine's stream;
synchronous: the time includes the launches and the two host waits).  Reported per geometry and case:
  counts      n_verts / n_tris of the mesh before, ClipCounts after (the last clip for the box)
  call_ms     median of --calls calls (one untimed call first); calls_ms every call
  kernel_us   device time per launch of the pass's kernels and copies (torch.profiler, a call of its own)
  equal       counts, triangles, positions, normals, keys, lowmin (and vertex values) equal oracle/mt3d_clip.py:clip on
              the fetched mesh (checked once, before the timed calls)
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
    from oracle import mt3d_clip
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    second = synthetic.turbulence(n, device=dev).to(torch.float32).contiguous()
    eng, stream = cuda_engine()
    lo, hi = n / 4.0 + 0.25, 3.0 * n / 4.0 + 0.25
    box = [((1.0, 0, 0), lo, "high"), ((1.0, 0, 0), hi, "low"), ((0, 1.0, 0), lo, "high"), ((0, 1.0, 0), hi, "low"),
           ((0, 0, 1.0), lo, "high"), ((0, 0, 1.0), hi, "low")]

    res = dict(tool="bench_clip", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag

        def fresh(value_field):
            c0 = eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)
            if value_field:
                eng.mt3d_interpolate(second.data_ptr(), shape=shape, dtype=np.float32)
            return c0

        c0 = fresh(True)
        vals = eng.mt3d_interpolate(second.data_ptr(), shape=shape, dtype=np.float32)
        med = float(np.median(vals.astype(np.float64)))
        del vals
        cases = {"axis0_high": [dict(normal=(1.0, 0.0, 0.0), offset=n / 2.0 + 0.25, keep="high")],
                 "axis0_low": [dict(normal=(1.0, 0.0, 0.0), offset=n / 2.0 + 0.25, keep="low")],
                 "oblique": [dict(normal=(1.0, 2.0, 3.0), offset=3.0 * (n - 1) + 0.25, keep="high")],
                 "value_median": [dict(component=0, offset=med, keep="high")],
                 "box6": [dict(normal=a, offset=d, keep=k) for a, d, k in box]}
        for cname, calls in cases.items():
            value = cname.startswith("value")
            # the check: the oracle applied call by call to the fetched mesh
            fresh(value)
            equal = True
            for kw in calls:
                pre = eng.mt3d_fetch()
                v = eng.mt3d_interpolate(second.data_ptr(), shape=shape, dtype=np.float32) if value else None
                want, wc = mt3d_clip.clip(pre["verts"], pre["tris"], normals=pre["normals"], keys=pre["keys"],
                                          lowmin=pre["lowmin"], values=v, geom_dtype=pre["verts"].dtype, side=kw["keep"],
                                          normal=kw.get("normal"), component=kw.get("component"), offset=kw["offset"])
                c = eng.mt3d_clip(**kw)
                post = eng.mt3d_fetch()
                equal = equal and (c.n_verts, c.n_tris, c.n_new_verts, c.n_cut_tris, c.n_dropped_tris) == (
                    wc["n_verts"], wc["n_tris"], wc["n_new_verts"], wc["n_cut_tris"], wc["n_dropped_tris"])
                for k in ("tris", "verts", "normals", "keys", "lowmin"):
                    equal = equal and bool(np.array_equal(post[k], np.asarray(want[k]).reshape(post[k].shape)))
                del pre, post, want

            def clip_all():
                for kw in calls:
                    eng.mt3d_clip(**kw)

            ms = per_call(stream, clip_all, args.calls, 1, setup=lambda: fresh(value))
            kernel_us = kernel_table(clip_all, ("k_clip_", "k_flag_scan", "k_sel_rows", "k_o_init", "Memcpy", "Memset"),
                                     setup=lambda: fresh(value))
            res["%s_%s" % (gname, cname)] = dict(
                n_verts_in=int(c0.n_verts), n_tris_in=int(c0.n_tris), n_verts=int(c.n_verts), n_tris=int(c.n_tris),
                n_new_verts=int(c.n_new_verts), n_cut_tris=int(c.n_cut_tris), n_dropped_tris=int(c.n_dropped_tris),
                call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms], kernel_us=kernel_us,
                equal=equal)
    emit(res, args.out)


if __name__ == "__main__":
    main()
