"""Step times of the extractions whose stage 1 is not the bench.py headline's: the generic stage-1 kernel and the 4D run.

    python tools/bench_stage1_paths.py [--n 512] [--n4d 128 --nt 64] [--steps 50] [--warmup 5] [--out FILE]

generic: the float32 ct_like(n) field from a device pointer one sample past a 16-byte boundary, which the TMA kernel
         cannot read, so stage 1 runs k_bitplane_generic (fp32 geometry and normals, as bench.py).
4d:      the float32 morph4d(n4d, nt) field from the device, with morph triangles (tools/bench_paths.py's 4D row).
Per path: the step time (CUDA events over --steps runs after --warmup), stage 1 of an instrumented pass
(ctr_stage_times), the counts and a SHA-256 of every fetched output array, so that two builds of the library
(CTR_LIB) can be checked for equal outputs at the timed sizes.  Prints one JSON line (also written to --out).
"""
import argparse
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.benchkit import cuda_engine, emit, gpu_info, window  # noqa: E402


def digest(out):
    h = hashlib.sha256()
    for k in sorted(out):
        v = out[k]
        if isinstance(v, np.ndarray):
            h.update(k.encode())
            h.update(np.ascontiguousarray(v).tobytes())
    return h.hexdigest()


def stage1_ms(eng, run, k=10):
    eng.set_timing(True)
    acc = 0.0
    for _ in range(k):
        run()
        acc += eng.stage_times(8)[1] / k
    eng.set_timing(False)
    return acc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--n4d", type=int, default=128)
    ap.add_argument("--nt", type=int, default=64)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic
    dev = torch.device("cuda", 0)
    eng, stream = cuda_engine()

    def timed(run):
        "ms per step: --steps runs in one window, after --warmup untimed ones"
        for _ in range(args.warmup):
            run()
        torch.cuda.synchronize()

        def steps():
            for _ in range(args.steps):
                run()
        return window(stream, steps) / args.steps

    res = dict(tool="bench_stage1_paths", lib=E.LIB_PATH, gpu=gpu_info(), device=torch.cuda.get_device_name(0),
               steps=args.steps, warmup=args.warmup, paths={})

    n = args.n
    q = synthetic.ct_like(n, device=dev).to(torch.float32).reshape(-1)
    buf = torch.empty(q.numel() + 4, dtype=torch.float32, device=dev)
    buf[1:1 + q.numel()] = q
    del q
    ptr, shape3 = buf.data_ptr() + 4, (n, n, n)
    assert ptr % 16 != 0

    def run3(flags=E.WANT_NORMALS):
        return eng.mt3d_run(ptr, 0.5, shape=shape3, dtype=np.float32, flags=flags | E.FIELD_ON_DEVICE)
    ms = timed(run3)
    s1 = stage1_ms(eng, run3)
    c = run3(E.WANT_NORMALS | E.WANT_MINMAX)
    res["paths"]["generic"] = dict(shape=list(shape3), ms_per_step=round(ms, 4), stage1_ms=round(s1, 4),
                                   counts=dict(n_verts=int(c.n_verts), n_tris=int(c.n_tris), fmin=c.fmin, fmax=c.fmax),
                                   sha256=digest(eng.mt3d_fetch()))
    del buf
    torch.cuda.empty_cache()

    f = synthetic.morph4d(args.n4d, args.nt, device=dev).to(torch.float32).contiguous()
    shape4 = tuple(f.shape)

    def run4(flags=E.MORPH):
        return eng.mp4d_run(f.data_ptr(), 1.2, shape=shape4, dtype=np.float32, flags=flags | E.FIELD_ON_DEVICE)
    ms = timed(run4)
    s1 = stage1_ms(eng, run4)
    c = run4(E.MORPH | E.WANT_MINMAX)
    res["paths"]["4d"] = dict(shape=list(shape4), ms_per_step=round(ms, 4), stage1_ms=round(s1, 4),
                              counts=dict(n_verts=int(c.n_verts), n_tets=int(c.n_tets), n_morph_tris=int(c.n_morph_tris),
                                          fmin=c.fmin, fmax=c.fmax),
                              sha256=digest(eng.mp4d_fetch()))
    eng.close()
    emit(res, args.out)


if __name__ == "__main__":
    main()
