"""Cost of the connected-components pass (ctr_mt3d_components) on the headline 512^3 surface, in one run.

    python tools/bench_components.py [--n 512] [--calls 20] [--rounds 5] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device), isovalue 0.5, WANT_NORMALS, in fp32 and in fp64 geometry.
Reported per geometry type:
  pass_ms        ctr_mt3d_components per call (CUDA events around --calls back-to-back calls, median of --rounds
                 rounds); the call is synchronous (it waits twice inside, for the id check and for the component count),
                 so this includes launches and waits
  orient_ms      ctr_mt3d_orient_reference on the same mesh, timed the same way, for comparison (it rewinds the mesh;
                 every call after the first finds nothing to flip, the work is the same)
  kernel_us      device time per launch of every kernel of both passes (torch.profiler, a pass of its own)
  host_oracle_ms oracle/mt3d_components.py:components on the fetched mesh (numpy + scipy, one host core, median of 3)
  oracle_equal   labels and integer fields equal to the oracle, box bit for bit, max relative area / volume differences
The field is 512 MB, larger than L2; the pass touches the mesh (7.9 M triangles: 94 MB of ids, 47 or 94 MB of positions)
and two 512 MB hash tables.  Prints one JSON line (also written to --out).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = (x.strip() for x in out[0].split(","))
        return dict(name=name, power_limit=power)
    except Exception as e:                                      # the line still carries torch's device name
        return dict(name=None, power_limit=None, error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_components
    assert torch.cuda.is_available(), "bench_components measures on a CUDA device"
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    value = 0.5
    field = synthetic.ct_like(n, device=dev)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    eng = E.Engine(0)
    eng.set_stream(stream.cuda_stream)
    nret, nc, nf = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()

    def comp():
        eng._check(eng.lib.ctr_mt3d_components(eng.h, ctypes.byref(nret)), "ctr_mt3d_components")

    def orient():
        eng._check(eng.lib.ctr_mt3d_orient_reference(eng.h, ctypes.byref(nc), ctypes.byref(nf)), "ctr_mt3d_orient_reference")

    def timed(fn):
        for _ in range(3):
            fn()
        ms = []
        for _ in range(args.rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.calls):
                fn()
            e1.record(stream)
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1) / args.calls)
        return ms

    res = dict(tool="bench_components", n=n, calls=args.calls, rounds=args.rounds, gpu=gpu_info(),
               device=torch.cuda.get_device_name(0), isovalue=value, run_flags="WANT_NORMALS")
    from torch.profiler import ProfilerActivity, profile
    for geom, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        c = eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=E.WANT_NORMALS | gflag)
        out = eng.mt3d_fetch()
        lab, tab = eng.mt3d_components()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            want_lab, want = mt3d_components.components(out["verts"], out["tris"])
            ts.append((time.perf_counter() - t0) * 1e3)
        equal = bool(np.array_equal(lab, want_lab) and len(tab) == len(want) and
                     all(np.array_equal(tab[f], want[f]) for f in ("n_tris", "n_verts", "n_edges", "n_boundary_edges",
                                                                   "n_nonmanifold_edges", "first_tri", "lo", "hi")))
        rel_area = float(np.max(np.abs(tab["area"] - want["area"]) / want["area"])) if equal else None
        vscale = want["area"] * (want["hi"] - want["lo"]).max(axis=1)
        rel_vol = float(np.max(np.abs(tab["volume"] - want["volume"]) / vscale)) if equal else None
        pass_ms = timed(comp)
        orient_ms = timed(orient)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                comp()
                orient()
            torch.cuda.synchronize()
        kernel_us = {}
        for ev in prof.key_averages():
            name = ev.key
            for tag in ("k_m_", "k_o_"):
                if tag in name:
                    short = name[name.index(tag):].split("(")[0].split("<")[0]
                    tot = getattr(ev, "device_time_total", None)
                    tot = ev.cuda_time_total if tot is None else tot
                    kernel_us[short] = dict(launches=ev.count, us_per_launch=round(tot / max(ev.count, 1), 2))
        closed = tab["n_boundary_edges"] == 0
        res[geom] = dict(n_verts=int(c.n_verts), n_tris=int(c.n_tris), n_components=len(tab), closed=int(closed.sum()),
                         largest_component_tris=int(tab["n_tris"].max()) if len(tab) else 0,
                         pass_ms=round(float(np.median(pass_ms)), 4), pass_ms_rounds=[round(x, 4) for x in pass_ms],
                         orient_ms=round(float(np.median(orient_ms)), 4), orient_ms_rounds=[round(x, 4) for x in orient_ms],
                         orient_n_components=int(nc.value), kernel_us=kernel_us,
                         host_oracle_ms=round(float(np.median(ts)), 1), oracle_equal=equal,
                         max_rel_area_diff=rel_area, max_rel_volume_diff=rel_vol)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
