#!/usr/bin/env python
"""Mean device time per launch of every k_* kernel of the bench extraction, from a torch.profiler trace.

    python tools/stage2_kernels.py --out DIR [--n 512] [--iters 50] [--warmup 10]

Runs --iters extractions of bench.py's field (synthetic.ct_like(n), isovalue 0.5, fp32 geometry with normals, one
context, synchronous steps) under torch.profiler with CUDA activities, after --warmup untimed ones, writes the trace to
DIR/trace.json and prints one line per kernel (launches, mean device microseconds per launch) under a header line with
the GPU's name and power limit.  The stage timer of the engine (stage_times) lumps k_count_a, k_count_b and k_scan
into one number; this gives each kernel its own.  The kernels are chained with programmatic dependent launch, so a
kernel's span includes the time it waits for the one in front and the spans add up to more than a step.  Tracing
slows the host: take step times from bench.py, not from here.
"""
import argparse
import json
import os
import re
import sys
from collections import OrderedDict

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import gpu_info  # noqa: E402


def kernel_times(trace_path):
    """{kernel: [device microseconds of each launch]} of the k_* kernels of a chrome trace, in first-launch order."""
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    per = OrderedDict()
    for e in events:
        if e.get("cat") != "kernel":
            continue
        m = re.search(r"\b(k_\w+)", e.get("name", ""))
        if m:
            per.setdefault(m.group(1), []).append(float(e["dur"]))
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the trace")
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--label", default="", help="printed on the header line")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    from contourist_b200 import engine as E
    from contourist_b200 import synthetic

    if not torch.cuda.is_available():
        raise SystemExit("stage2_kernels.py: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    n = args.n
    field = synthetic.ct_like(n, device=dev)
    shape = (n, n, n)
    eng = E.Engine(0)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)

    def step():
        return eng.mt3d_run(field.data_ptr(), 0.5, shape=shape, dtype=np.float32, flags=E.WANT_NORMALS)

    for _ in range(args.warmup):
        c = step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            step()
        torch.cuda.synchronize()
    trace = os.path.join(args.out, "trace.json")
    prof.export_chrome_trace(trace)
    gpu = gpu_info()
    print("%s%s, power limit %s: %d extractions of %d^3 (%d vertices, %d triangles), mean device time per launch"
          % (args.label + ": " if args.label else "", gpu["name"], gpu["power_limit"], args.iters, n, c.n_verts, c.n_tris))
    per = kernel_times(trace)
    for k, v in per.items():
        print("  %-24s %6d launches %9.2f us" % (k, len(v), sum(v) / len(v)))


if __name__ == "__main__":
    main()
