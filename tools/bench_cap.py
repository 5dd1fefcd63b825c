"""Cost of the caps at the box faces (ctr_mt3d_cap) on the headline 512^3 surface, in one run.

    python tools/bench_cap.py [--n 512] [--calls 10] [--out FILE]

The mesh: synthetic.ct_like(n) (fp32, on the device) at isovalue 0.5 with WANT_NORMALS | WANT_KEYS, in fp32 and in fp64
geometry; both sides.  A cap edits the mesh and refuses a capped one, so every timed call runs on a fresh extraction:
the run is outside the timed window, which holds one ctr_mt3d_cap call (CUDA events on the engine's stream; synchronous:
the time includes its launches, its one wait for the totals and any growth of the output buffers).  Reported per
geometry and side:
  counts      n_verts / n_tris before, and CapCounts after
  call_ms     median of --calls calls (each on a fresh run; two untimed calls first); calls_ms every call
  kernel_us   device time per launch of the pass's kernels and copies (torch.profiler, a call of its own)
  equal       counts, triangles, keys, lowmin, new positions and the old rows equal oracle/mt3d_cap.py:cap on the fetched
              mesh, new normals within one ulp (checked once, before the timed calls)
Prints one JSON line (also written to --out).
"""
import argparse
import json
import os
import subprocess
import sys

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
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_cap
    assert torch.cuda.is_available(), "bench_cap measures on a CUDA device"
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    field = synthetic.ct_like(n, device=dev)
    host = field.cpu().numpy()
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    eng = E.Engine(0)
    eng.set_stream(stream.cuda_stream)

    res = dict(tool="bench_cap", n=n, calls=args.calls, gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    for gname, gflag in (("fp32", 0), ("fp64", E.GEOM_F64)):
        flags = E.WANT_NORMALS | E.WANT_KEYS | gflag
        gd = np.float64 if gflag else np.float32

        def run():
            return eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=flags)

        for side in ("high", "low"):
            c0 = run()
            pre = eng.mt3d_fetch()
            c = eng.mt3d_cap(side)
            out = eng.mt3d_fetch()
            want, cnt = mt3d_cap.cap(pre, host, 0.5, side, geom_dtype=gd)
            nV = int(c0.n_verts)
            equal = bool(dict(n_verts=c.n_verts, n_tris=c.n_tris, n_cap_verts=c.n_cap_verts, n_cap_tris=c.n_cap_tris,
                              n_missing=c.n_missing) == cnt and
                         all(np.array_equal(out[k], want[k]) for k in ("tris", "keys", "lowmin", "verts")) and
                         np.array_equal(out["normals"][:nV], pre["normals"]) and
                         bool((np.abs(out["normals"][nV:] - want["normals"][nV:]) <=
                               np.spacing(np.abs(want["normals"][nV:]))).all()))
            del pre, out, want
            ms = []
            for q in range(args.calls + 2):                       # two untimed calls first
                run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                eng.mt3d_cap(side)
                e1.record(stream)
                torch.cuda.synchronize()
                if q >= 2:
                    ms.append(e0.elapsed_time(e1))
            run()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eng.mt3d_cap(side)
                torch.cuda.synchronize()
            kernel_us = {}
            for ev in prof.key_averages():
                key = ev.key
                tag = next((t_ for t_ in ("k_cap_", "k_d_", "k_flag_scan", "Memcpy", "Memset") if t_ in key), None)
                if tag is None:
                    continue
                short = key[key.index(tag):].split("(")[0].split("<")[0] if tag.startswith("k_") else key
                tot = getattr(ev, "device_time_total", None)
                tot = ev.cuda_time_total if tot is None else tot
                kernel_us[short] = dict(launches=ev.count, us_per_launch=round(tot / max(ev.count, 1), 2))
            res["%s_%s" % (gname, side)] = dict(
                n_verts_in=nV, n_tris_in=int(c0.n_tris), n_verts=int(c.n_verts), n_tris=int(c.n_tris),
                n_cap_verts=int(c.n_cap_verts), n_cap_tris=int(c.n_cap_tris), n_missing=int(c.n_missing),
                call_ms=round(float(np.median(ms)), 4), calls_ms=[round(x, 4) for x in ms], kernel_us=kernel_us,
                equal=equal)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
