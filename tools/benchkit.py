"""What the pass benchmarks in tools/ share: the card they ran on, the engine on torch's stream, the two shapes of timed
window, the per-kernel table from torch.profiler and the JSON line.

Every timing here is CUDA events on the stream the engine runs on.  There is no fallback: a measurement that finds no
CUDA device fails.
"""
import json
import subprocess

import numpy as np


def gpu_info():
    "the card's name and power limit from nvidia-smi, which the line must carry beside its times"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = (x.strip() for x in out[0].split(","))
        return dict(name=name, power_limit=power)
    except Exception as e:                                      # the line still carries torch's device name
        return dict(name=None, power_limit=None, error=str(e))


def cuda_engine():
    "Engine(0) on torch's current stream, behind everything queued on it so far.  Returns (engine, stream)."
    import torch
    from contourist_b200 import engine as E
    assert torch.cuda.is_available(), "the benchmarks measure on a CUDA device"
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    eng = E.Engine(0)
    eng.set_stream(stream.cuda_stream)
    return eng, stream


def window(stream, body):
    "ms between two events recorded on `stream` around body(); returns once the second has happened"
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    body()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def per_call(stream, call, calls, untimed, setup=None):
    """ms of each of `calls` calls, each in a window of its own, after `untimed` calls not kept.  setup() (a fresh mesh
    for a pass that edits it) and a synchronise come before every window, outside it."""
    import torch
    ms = []
    for q in range(untimed + calls):
        if setup is not None:
            setup()
        torch.cuda.synchronize()
        t = window(stream, call)
        if q >= untimed:
            ms.append(t)
    return ms


def back_to_back(stream, arms, calls, rounds, warm):
    """{arm: [ms per call of each round]} for a dict of arms {name: call}: `warm` untimed calls of every arm, then per
    round one window of `calls` calls of each arm in turn."""
    for call in arms.values():
        for _ in range(warm):
            call()
    ms = {name: [] for name in arms}
    for _ in range(rounds):
        for name, call in arms.items():
            def body():
                for _ in range(calls):
                    call()
            ms[name].append(window(stream, body) / calls)
    return ms


def short_name(key, tag):
    "a kernel's name without its namespace, template arguments and parameters; copies and sets keep the profiler's key"
    return key if tag in ("Memcpy", "Memset") else key[key.index(tag):].split("(")[0].split("<")[0]


def kernel_table(call, tags, setup=None, reps=1, key=short_name):
    """{key(name, tag): {launches, us_per_launch}} of the profiler events whose name holds one of `tags` (the first that
    matches), from `reps` calls under torch.profiler with CUDA activities; setup() runs before, outside the profile."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    if setup is not None:
        setup()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    table = {}
    for ev in prof.key_averages():
        tag = next((t for t in tags if t in ev.key), None)
        if tag is None:
            continue
        tot = getattr(ev, "device_time_total", None)
        tot = ev.cuda_time_total if tot is None else tot
        table[key(ev.key, tag)] = dict(launches=ev.count, us_per_launch=round(tot / max(ev.count, 1), 2))
    return table


def emit(res, out):
    "print the result as one JSON line, and write it to `out` when given"
    line = json.dumps(res)
    print(line)
    if out:
        with open(out, "w") as fh:
            fh.write(line + "\n")


def normals_close(got, want, verts, tris, geom64):
    """normals within 1e-9 rad (fp64 geometry) or 2e-6 per component (fp32) of the definition's, at the vertices whose
    face-normal sum is not cancellation noise"""
    from oracle import mt3d_smooth
    mag, parts = mt3d_smooth.face_normal_sums(verts, tris)
    ok = (parts > 0) & (mag >= 1e-6 * parts)
    g, w = got[ok].astype(np.float64), want[ok].astype(np.float64)
    if geom64:
        return bool(np.arctan2(np.linalg.norm(np.cross(g, w), axis=1), (g * w).sum(axis=1)).max(initial=0) < 1e-9)
    return bool(np.abs(g - w).max(initial=0) <= 2e-6)
