"""Cost of the plane sections (ctr_mt3d_section) of the headline 512^3 surface, in one run.

    python tools/bench_section.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry.  The planes: 1, 64 and 512 planes along axis 0 (x = i + 0.5 for k evenly spaced grid rows i), and 512 oblique
planes (normal (1, 2, 3), spread over the mesh's extent).  A section does not edit the mesh, so every timed call runs on
the same extraction; the window holds one ctr_mt3d_section call (CUDA events on the engine's stream; synchronous: the
time includes its launches and host waits).  Reported per geometry and plane set:
  counts      n_verts / n_tris of the mesh, SectionCounts
  call_ms     median of --calls calls (two untimed calls first); calls_ms every call
  kernel_us   device time per launch of the pass's kernels and copies (torch.profiler, a call of its own)
  equal       segments, polylines, flags, points and junction planes equal oracle/mt3d_section.py:section on the fetched
              mesh, lengths and areas within rtol 1e-12 (checked once, before the timed calls)
Prints one JSON line (also written to --out).
"""
import argparse
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, kernel_table, per_call  # noqa: E402


def same(polys, want):
    for got, ref in zip(polys, want):
        if (got is None) != (ref is None):
            return False
        if ref is None:
            continue
        if len(got) != len(ref):
            return False
        for (c, k, p, ln, ar), (rc, rk, rp, rln, rar) in zip(got, ref):
            if (c, k) != (rc, rk) or not np.array_equal(p, rp) or not np.isclose(ln, rln, rtol=1e-12, atol=0) or \
                    not np.isclose(ar, rar, rtol=1e-12, atol=1e-12 * rln * rln):
                return False
    return len(polys) == len(want)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_section
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    eng, stream = cuda_engine()

    res = dict(tool="bench_section", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        c0 = eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=E.WANT_NORMALS | E.WANT_KEYS | gflag)
        mesh = eng.mt3d_fetch()
        s = mesh["verts"].astype(np.float64) @ np.array([1.0, 2.0, 3.0])
        cases = {"axis0_%d" % k: ((1.0, 0.0, 0.0), (np.arange(2 * k, step=2) + 1) * n // (2 * k) + 0.5) for k in (1, 64, 512)}
        cases["oblique_512"] = ((1.0, 2.0, 3.0), np.linspace(s.min(), s.max(), 514)[1:-1])
        for cname, (normal, offs) in cases.items():
            seg, polys = eng.mt3d_section(normal, offs)
            want = mt3d_section.section(mesh["verts"], mesh["tris"], normal, offs, mesh["verts"].dtype)
            equal = bool(np.array_equal(seg["plane"], want["plane"]) and np.array_equal(seg["edges"], want["edges"]) and
                         np.array_equal(seg["points"], want["points"]) and same(polys, want["polylines"]))
            del seg, want
            c, p = E.SectionCounts(), E.SectionParams()
            for a in range(3):
                p.normal[a] = normal[a]
            off = np.ascontiguousarray(offs, np.float64)
            p.offsets = off.ctypes.data
            p.nplanes = len(off)

            def section():
                eng._check(eng.lib.ctr_mt3d_section(eng.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_section")

            ms = per_call(stream, section, args.calls, 2)
            kernel_us = kernel_table(lambda: eng.mt3d_section(normal, offs),
                                     ("k_sec_", "k_p_", "k_ps_", "k_m_", "k_o_", "k_s_", "Memcpy", "Memset"))
            res["%s_%s" % (gname, cname)] = dict(
                n_verts=int(c0.n_verts), n_tris=int(c0.n_tris), n_segments=int(c.n_segments),
                n_polylines=int(c.n_polylines), n_points=int(c.n_points), n_junction_planes=int(c.n_junction_planes),
                call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms], kernel_us=kernel_us,
                equal=equal)
        del mesh
    emit(res, args.out)


if __name__ == "__main__":
    main()
