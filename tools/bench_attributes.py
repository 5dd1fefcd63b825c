"""Cost of per-vertex values of other fields (ctr_mt3d_interpolate) on the headline 512^3 surface, in one run.

    python tools/bench_attributes.py [--n 512] [--calls 200] [--rounds 5] [--steps 100] [--out FILE]

The run: synthetic.ct_like(n) (fp32, on the device), isovalue 0.5, fp32 geometry, WANT_NORMALS | WANT_KEYS (bench.py's
step plus keys).  Reported:
  pass_ms     ctr_mt3d_interpolate per call (CUDA events around --calls back-to-back calls, median of --rounds rounds)
              for a scalar fp32 field (ct_like(n, seed=1)), a 3-component fp32 field (seeds 1, 2, 3) and a scalar
              uint8 field (the seed-1 field * 255); each call is synchronous, so this includes the launch and the wait
  kernel_us   device time per launch of k_interp_attr and of k_emit_verts (torch.profiler, a pass of its own)
  emit_verts_stage_ms  k_emit_verts' stage time from an instrumented run (ctr_stage_times)
  keys        the device-resident step time with and without WANT_KEYS (what the façade's vertex_fields adds to the
              run), two contexts taking the steps in turn as bench.py does, the two arms alternating --rounds times
  host_oracle_ms  oracle/mt3d_values.py:vertex_values for the scalar fp32 field on the fetched keys (numpy, median of 3)
  identity    the int16 field of grid coordinates gives the vertex positions bit for bit
The fields are 0.5-1.6 GB, larger than L2, but each call touches only the rows around the surface.
Prints one JSON line (also written to --out).
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
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    from oracle import mt3d_values
    assert torch.cuda.is_available(), "bench_attributes measures on a CUDA device"
    dev = torch.device("cuda", 0)
    n = args.n
    shape = (n, n, n)
    value = 0.5
    field = synthetic.ct_like(n, device=dev)
    s1 = synthetic.ct_like(n, device=dev, seed=1)
    vec3 = torch.stack([s1, synthetic.ct_like(n, device=dev, seed=2), synthetic.ct_like(n, device=dev, seed=3)], -1).contiguous()
    u8 = torch.clamp(torch.round(s1 * 255), 0, 255).to(torch.uint8).contiguous()
    arms = [("scalar_f32", s1, np.float32, 1), ("vec3_f32", vec3, np.float32, 3), ("scalar_u8", u8, np.uint8, 1)]
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    eng = E.Engine(0)
    eng.set_stream(stream.cuda_stream)
    flags = E.WANT_NORMALS | E.WANT_KEYS
    c = eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
    out = eng.mt3d_fetch()
    nv = int(c.n_verts)

    params = {}
    for name, t, dt, nc in arms:
        p = E.AttrParams()
        p.field, p.dtype, p.flags, p.ncomp = t.data_ptr(), E.dtype_code(dt), E.FIELD_ON_DEVICE, nc
        params[name] = p
    nret = ctypes.c_int64()

    def call(name):
        eng._check(eng.lib.ctr_mt3d_interpolate(eng.h, ctypes.byref(params[name]), ctypes.byref(nret)), "ctr_mt3d_interpolate")

    # identity: grid coordinates -> positions, bit for bit
    ax = torch.arange(n, device=dev, dtype=torch.int16)
    grid = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).contiguous()
    torch.cuda.synchronize()
    identity = bool(np.array_equal(eng.mt3d_interpolate(grid.data_ptr(), shape=shape + (3,), dtype=np.int16), out["verts"]))
    del grid

    # pass time per call
    for name, *_ in arms:
        for _ in range(20):
            call(name)
    pass_ms = {name: [] for name, *_ in arms}
    for _ in range(args.rounds):
        for name, *_ in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.calls):
                call(name)
            e1.record(stream)
            torch.cuda.synchronize()
            pass_ms[name].append(e0.elapsed_time(e1) / args.calls)

    # reference: k_emit_verts' stage time in the same call
    eng.set_timing(True)
    acc = np.zeros(8)
    for _ in range(10):
        eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
        acc += np.array(eng.stage_times(8)) / 10
    eng.set_timing(False)

    # kernel times (a profiled pass of its own)
    from torch.profiler import ProfilerActivity, profile
    eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
            for name, *_ in arms:
                call(name)
        torch.cuda.synchronize()
    kernel_us = {}
    for ev in prof.key_averages():
        if "k_interp_attr" in ev.key or "k_emit_verts" in ev.key:
            tot = getattr(ev, "device_time_total", None)
            tot = ev.cuda_time_total if tot is None else tot
            kernel_us[ev.key[:96]] = dict(launches=ev.count, us_per_launch=round(tot / max(ev.count, 1), 2))
    # the two fp32 arms launch the same instantiation: one profiled pass per arm keeps them apart
    prof_arms = {}
    for name, *_ in arms:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                call(name)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if "k_interp_attr" in ev.key:
                tot = getattr(ev, "device_time_total", None)
                tot = ev.cuda_time_total if tot is None else tot
                prof_arms[name] = round(tot / max(ev.count, 1), 2)

    # what the façade option costs the run: WANT_KEYS on and off, alternated
    engines = (eng, E.Engine(0))
    engines[1].set_stream(stream.cuda_stream)

    def run_steps(fl, k):
        pending = None
        for s in range(k):
            e = engines[s & 1]
            e.mt3d_enqueue(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=fl)
            if pending is not None:
                pending.mt3d_finish()
            pending = e
        return pending.mt3d_finish()

    key_arms = [("with_keys", flags), ("without_keys", E.WANT_NORMALS)]
    for _, fl in key_arms:
        run_steps(fl, 20)
    step_ms = {name: [] for name, _ in key_arms}
    for _ in range(args.rounds):
        for name, fl in key_arms:
            run_steps(fl, 4)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run_steps(fl, args.steps)
            e1.record(stream)
            torch.cuda.synchronize()
            step_ms[name].append(e0.elapsed_time(e1) / args.steps)

    # host baseline: the numpy definition on the fetched keys
    hf, ha = field.cpu().numpy(), s1.cpu().numpy()
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        ref = mt3d_values.vertex_values(hf, value, out["keys"], out["lowmin"], ha, np.float32)
        ts.append((time.perf_counter() - t0) * 1e3)
    eng.mt3d_run(field.data_ptr(), value, shape=shape, dtype=np.float32, flags=flags)
    got = eng.mt3d_interpolate(s1.data_ptr(), shape=shape, dtype=np.float32)
    scale = float(ha.max() - ha.min())
    oracle_max_abs_diff = float(np.max(np.abs(got.astype(np.float64) - ref.astype(np.float64)))) if nv else 0.0

    res = dict(tool="bench_attributes", n=n, calls=args.calls, rounds=args.rounds, steps=args.steps, gpu=gpu_info(),
               device=torch.cuda.get_device_name(0), geometry="fp32", run_flags="WANT_NORMALS|WANT_KEYS", isovalue=value,
               n_verts=nv, identity_int16_coordinates=identity,
               pass_ms={k: round(float(np.median(v)), 4) for k, v in pass_ms.items()},
               pass_ms_rounds={k: [round(x, 4) for x in v] for k, v in pass_ms.items()},
               kernel_us_interp_attr=prof_arms, kernel_us=kernel_us,
               emit_verts_stage_ms=round(float(acc[3]), 4),
               keys=dict(step_ms={k: round(float(np.median(v)), 4) for k, v in step_ms.items()},
                         step_ms_rounds={k: [round(x, 4) for x in v] for k, v in step_ms.items()}),
               host_oracle_ms=round(float(np.median(ts)), 1),
               oracle_max_abs_diff_scalar_f32=oracle_max_abs_diff, attr_range=scale)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
