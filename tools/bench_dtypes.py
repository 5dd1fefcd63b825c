"""float32 against uint16 / int16 / uint8 samples of the same quantized 512^3 surface, in one run.

    python tools/bench_dtypes.py [--n 512] [--steps 200] [--warmup 20] [--rounds 5] [--out FILE]

q = synthetic.ct_like(n) (fp32, on the device), quantized:
    uint16  clip(round(q * 4096), 0, 65535)   isovalues 2048.5 (half-integer: no sample on the isovalue) and 2048
    int16   the uint16 field - 2048            isovalues 0.5 and 0
    uint8   clip(round(q * 128), 0, 255)       isovalues 64.5 and 64
Each integer arm is paired with the float32 copy of its own field at the same isovalue (the same surface), with fp32
geometry and normals as bench.py.  Per arm: the device-resident step time (CUDA events over --steps steps after
--warmup, two contexts taking the steps in turn as bench.py steps; the arms alternate, --rounds times, median of the
rounds), the per-stage times of an instrumented pass (ctr_stage_times), the end-to-end mt3d_extract_host time from a
page-locked host array (median of 7 calls after 3 untimed ones) and the bytes stage 1 reads.  One step of every arm is
checked: the integer mesh equals the float32 mesh bit for bit.  Prints one JSON line (also written to --out).
"""
import argparse
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, window  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    dev = torch.device("cuda", 0)
    n = args.n
    q = synthetic.ct_like(n, device=dev)
    u16 = torch.clamp(torch.round(q * 4096), 0, 65535).to(torch.int32)
    fields = {
        "uint16": (u16.to(torch.uint16), np.uint16, (2048.5, 2048.0)),
        "int16": ((u16 - 2048).to(torch.int16), np.int16, (0.5, 0.0)),
        "uint8": (torch.clamp(torch.round(q * 128), 0, 255).to(torch.uint8), np.uint8, (64.5, 64.0)),
    }
    del q
    arms = []                                                   # (name, tensor, numpy dtype, isovalue, pair name)
    for key, (t, dt, values) in fields.items():
        t = t.contiguous()
        f32 = t.to(torch.float32).contiguous()
        for v in values:
            arms.append(("%s@%g" % (key, v), t, dt, v, "float32(%s)@%g" % (key, v)))
            arms.append(("float32(%s)@%g" % (key, v), f32, np.float32, v, None))
    shape = (n, n, n)
    flags = E.WANT_NORMALS
    eng, stream = cuda_engine()
    engines = (eng, cuda_engine()[0])

    def run_steps(t, dt, v, k):
        pending = None
        for s in range(k):
            e = engines[s & 1]
            e.mt3d_enqueue(t.data_ptr(), v, shape=shape, dtype=dt, flags=flags)
            if pending is not None:
                pending.mt3d_finish()
            pending = e
        return pending.mt3d_finish()

    # equality: one step of every integer arm against its float32 pair
    meshes = {}
    for name, t, dt, v, _ in arms:
        c = engines[0].mt3d_run(t.data_ptr(), v, shape=shape, dtype=dt, flags=flags | E.WANT_KEYS)
        o = engines[0].mt3d_fetch()
        meshes[name] = (int(c.n_verts), int(c.n_tris), int(c.n_active_cells), int(c.n_crossings), o)
    checked = []
    for name, _, _, _, pair in arms:
        if pair is None:
            continue
        a, b = meshes[name], meshes[pair]
        assert a[:4] == b[:4], (name, a[:4], b[:4])
        for k in ("verts", "normals", "tris", "keys", "lowmin"):
            assert np.array_equal(a[4][k], b[4][k]), (name, k)
        checked.append(name)
    counts = {name: dict(n_verts=m[0], n_tris=m[1], n_active_cells=m[2], n_crossings=m[3]) for name, m in meshes.items()}
    meshes = None

    # per-stage times: an instrumented pass of its own
    stages = {}
    for name, t, dt, v, _ in arms:
        e = engines[0]
        e.set_timing(True)
        acc = np.zeros(8)
        for _ in range(10):
            e.mt3d_run(t.data_ptr(), v, shape=shape, dtype=dt, flags=flags)
            acc += np.array(e.stage_times(8)) / 10
        e.set_timing(False)
        stages[name] = dict(bitplane_ms=round(acc[1], 4), count_scan_ms=round(acc[2], 4), emit_verts_ms=round(acc[3], 4),
                            emit_tris_ms=round(acc[4], 4))

    # device-resident step time: arms alternate, rounds x steps each
    for name, t, dt, v, _ in arms:
        run_steps(t, dt, v, max(args.warmup, 2))
    torch.cuda.synchronize()
    per_round = {name: [] for name, *_ in arms}
    for _ in range(args.rounds):
        for name, t, dt, v, _ in arms:
            run_steps(t, dt, v, 4)
            per_round[name].append(window(stream, lambda: run_steps(t, dt, v, args.steps)) / args.steps)

    # end to end from page-locked host memory (mt3d_extract_host: pipelined upload, extraction, download)
    host = E.Engine(0)
    e2e = {}
    for name, t, dt, v, _ in arms:
        pinned = host.pinned_empty("bench_in", shape, dt)
        pinned[...] = (t if dt == np.float32 else t.to(torch.int32)).cpu().numpy()
        for _ in range(3):
            host.mt3d_extract_host(pinned, v, flags=flags)
        ts = []
        for _ in range(7):
            t0 = time.perf_counter()
            host.mt3d_extract_host(pinned, v, flags=flags)
            ts.append((time.perf_counter() - t0) * 1e3)
        e2e[name] = dict(median_ms=round(float(np.median(ts)), 3), calls_ms=[round(x, 3) for x in ts])

    res = dict(tool="bench_dtypes", n=n, steps=args.steps, warmup=args.warmup, rounds=args.rounds,
               gpu=gpu_info(), device=torch.cuda.get_device_name(0), geometry="fp32", flags="WANT_NORMALS",
               equal_to_float32=checked, arms={})
    for name, t, dt, v, pair in arms:
        ms = per_round[name]
        res["arms"][name] = dict(dtype=np.dtype(dt).name, isovalue=v, step_ms=round(float(np.median(ms)), 4),
                                 step_ms_rounds=[round(x, 4) for x in ms], stage1_bytes=n ** 3 * np.dtype(dt).itemsize,
                                 stages=stages[name], e2e=e2e[name], counts=counts[name])
    emit(res, args.out)


if __name__ == "__main__":
    main()
