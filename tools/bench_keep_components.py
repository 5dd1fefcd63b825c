"""Cost of the component filter (ctr_mt3d_keep_components) on the headline 512^3 surface, in one run.

    python tools/bench_keep_components.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device), isovalue 0.5, WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry; two masks: keep the component with the most triangles ("largest") and keep every component ("all").  A
filtered mesh is a different input, so every timed call has a fresh ctr_mt3d_run and ctr_mt3d_components before it;
CUDA events on the engine's stream bracket the ctr_mt3d_keep_components call alone (it is synchronous: the time
includes its launches, its one wait for the three scan totals, and the upload of the C-byte mask).
Reported per geometry type and mask:
  keep_ms      median (and every value) over --calls timed calls
  kernel_us    device time per launch of the pass's kernels and of its device-to-device copies (torch.profiler, a pass
               of its own)
  bytes_moved  what the pass reads and writes by the shapes (flags, scans, compaction reads, scratch writes and the
               copies back), for comparison with the measured time
  equal        the filtered mesh and component results equal oracle/mt3d_filter.py:keep_components on the pre-filter
               fetch (checked once per configuration, outside the timed calls)
Prints one JSON line (also written to --out).
"""
import argparse
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, per_call  # noqa: E402


def bytes_moved(nv, nt, nc, nv2, nt2, nc2, gsz):
    "bytes the pass reads and writes, from the shapes (before: nv / nt / nc, after: nv2 / nt2 / nc2)"
    vrow = 3 * gsz * 2 + 8 + 1                                  # positions, normals, key, lowmin
    flags = nt * (4 + 1) + nt * (12 + 1) + nv                   # k_keep_tris (label -> keep_t), k_sel_used (ids -> used_v)
    scans = (nt + nv + nc) * (1 + 4)                            # flag in, index out
    rows = nv * (1 + 4) * 4 + nv2 * vrow * 2                    # per array: flags + indices read; scratch written, copied back
    tris = nt * (1 + 4 + 12) + nt2 * 4 * 3 * 2 + nt2 * 12 * 2   # k_sel_tris (ids through idx_v) and its copy back
    labels = nt * (1 + 4 + 4) + nt2 * (4 + 4) * 2               # k_keep_labels and its copy back
    table = nc * 113 + nc2 * 112 * 3
    return flags + scans + rows + tris + labels + table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_filter
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    value = 0.5
    field = synthetic.ct_like(n, device=dev)
    eng, stream = cuda_engine()
    nv_, nt_, nc_ = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()

    res = dict(tool="bench_keep_components", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0),
               isovalue=value, run_flags="WANT_NORMALS|WANT_KEYS")
    for geom, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag

        def prepare():
            eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
            eng._check(eng.lib.ctr_mt3d_components(eng.h, ctypes.byref(nc_)), "ctr_mt3d_components")

        eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
        pre = eng.mt3d_fetch()
        lab, tab = eng.mt3d_components()
        masks = dict(largest=(np.arange(len(tab)) == int(np.argsort(-tab["n_tris"], kind="stable")[0])).astype(np.uint8),
                     all=np.ones(len(tab), np.uint8))
        for name, mask in masks.items():
            # parity once, outside the timed calls, against the labels and table of the same components call (area and
            # volume sums of another call may differ in their last bits)
            eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
            pre = eng.mt3d_fetch()
            lab, tab = eng.mt3d_components()
            eng.mt3d_keep_components(mask.astype(bool))
            out = eng.mt3d_fetch()
            t, used, lab2, tab2 = mt3d_filter.keep_components(pre["tris"], lab, tab, mask)
            lab_f, tab_f = eng.mt3d_components_fetch()
            equal = bool(np.array_equal(out["tris"], t) and all(np.array_equal(out[k], pre[k][used])
                                                                 for k in ("verts", "normals", "keys", "lowmin")) and
                         np.array_equal(lab_f, lab2) and tab_f.tobytes() == tab2.tobytes())
            mp = mask.ctypes.data_as(ctypes.c_void_p)

            def keep():
                eng._check(eng.lib.ctr_mt3d_keep_components(eng.h, mp, len(mask), ctypes.byref(nv_), ctypes.byref(nt_)),
                           "ctr_mt3d_keep_components")

            ms = per_call(stream, keep, args.calls, 2, setup=prepare)
            kernel_us = kernel_table(keep, ("k_keep_", "k_sel_", "k_flag_scan", "Memcpy", "Memset"), setup=prepare)
            gsz = 8 if gflag else 4
            res.setdefault(geom, {})[name] = dict(
                n_verts=len(pre["verts"]), n_tris=len(pre["tris"]), n_components=len(tab), kept_verts=int(nv_.value),
                kept_tris=int(nt_.value), kept_components=int(mask.sum()),
                keep_ms=round(float(np.median(ms)), 4), keep_ms_calls=[round(x, 4) for x in ms], kernel_us=kernel_us,
                bytes_moved=bytes_moved(len(pre["verts"]), len(pre["tris"]), len(tab), int(nv_.value), int(nt_.value),
                                        int(mask.sum()), gsz),
                equal=equal)
    emit(res, args.out)


if __name__ == "__main__":
    main()
