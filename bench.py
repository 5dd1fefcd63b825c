#!/usr/bin/env python
"""bench.py -- headline benchmark: marching-tetrahedra extraction of a 512^3 fp32 volume on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n 512] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic 512^3 volume per GPU (BASELINE.json configs[2]:
CT-like fp32 volume, single isovalue, indexed mesh with normals).  N > 1 (torchrun, one rank per GPU):
weak scaling, each rank owns a 512-plane z-slab (+halo) of a (512*N) x 512 x 512 volume, extracts it
independently and joins an NCCL all-gather of (n_verts, n_tris) -> global vertex offsets.

Prints ONE JSON line (rank 0).  See DESIGN.md section 6 for what each key means.

--dump-outputs DIR (rank 0): after the timed steps, the mesh of the last timed step as DIR/<name>.npy (see
dump_outputs), so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ISOVALUE = 0.5
METRIC = "Gvoxels/s, 512^3 fp32 marching-tetrahedra extraction (indexed mesh + normals)"


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the kernels of one extraction, from the ncu --set full capture
    that tools/ncu_summary.py --json summarised into profiles/traffic.json (None when there is no such file)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    return float(d["total_bytes"]), d.get("source")


def workload_config(n, world):
    """The `config` of both arms (ours and --impl reference): the same workload, described once."""
    n_total = n * world
    return {"workload": "BASELINE configs[2]: %d^3 fp32 CT-like volume per GPU (48 Gaussian blobs + smoothed noise), "
                        "isovalue 0.5, indexed mesh + gradient normals, fp32 geometry" % n,
            "volume": [n_total, n, n],
            "generator": "contourist_b200.synthetic.ct_like(%d, n_total=%d), seed 0" % (n, n_total),
            "stacking": "one CT-like block (own 48 blobs) per GPU along the first axis, the neighbours' Gaussian tails "
                        "summed in: one continuous volume, the same amount of surface in every slab",
            "sharding": "z-slabs, 1 plane halo below / 2 above, NCCL all-gather of counts",
            "l2": "inputs (%.0f MB field) larger than the 126 MB L2; no explicit flush" % (float(n) ** 3 * 4 / 1e6)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(object):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.n_loaded = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        "end of the loaded window: rows that arrive later were sampled on an idle GPU and are not used"
        self.n_loaded = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = self.rows[:self.n_loaded] if self.n_loaded else self.rows
        for r in rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ reference arm
def _oracle_slab(args):
    """Worker: numpy oracle (restatement of the reference's algorithm) on one z-slab."""
    sub, value = args
    from oracle import mt3d
    r = mt3d.extract(sub, value, np.float32)
    mt3d.normals(sub, value, r["keys"], np.float32)
    return len(r["keys"]), len(r["tris"])


def bench_field(n):
    """The bench's own field on the host: synthetic.ct_like(n) (generated with torch on the GPU when there is one --
    plumbing, like in the timed arm -- else on the CPU), as a numpy array."""
    import torch
    from contourist_b200 import synthetic
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    return synthetic.ct_like(n, device=dev).cpu().numpy()


def time_oracle(field, value, cores):
    """Oracle port over `cores` processes (independent z-slabs with a one-plane overlap)."""
    import multiprocessing as mp
    n0 = field.shape[0]
    bounds = [round(r * (n0 - 1) / cores) for r in range(cores + 1)]
    jobs = [(np.ascontiguousarray(field[bounds[r]:bounds[r + 1] + 1]), value) for r in range(cores)
            if bounds[r + 1] > bounds[r]]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_oracle_slab(j) for j in jobs]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_oracle_slab, jobs)
    dt = time.perf_counter() - t0
    return dt, sum(r[1] for r in res)


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the Python reference itself cannot travel to the
    GPU box and would need hours at this size, BASELINE.md section 2) on all host cores, on the SAME 512^3 field as
    the timed arm.  A step is a bounded sample of that workload: a z-slab of the field, sized from a calibration run
    so that warmup + steps end within about two minutes, the slabs cycling through the volume (a step covers the whole
    volume when that fits)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = max(1, min(os.cpu_count() or 1, 64))
    n = args.n
    field = bench_field(n)
    # calibration (untimed): rate of the port on a slab of the middle of the volume
    cal = max(cores * 2 + 1, 33)
    c0 = (n - cal) // 2
    dt, _ = time_oracle(field[c0:c0 + cal], ISOVALUE, cores)
    rate = (cal - 1) * n * n / dt                                   # voxels per second
    budget = 100.0 / max(args.steps + args.warmup, 1)               # seconds per step
    planes = int(min(n, max(cores * 2 + 1, rate * budget / (n * n))))
    nslab = -(-n // planes)                                          # slabs that together cover the volume (they may overlap)
    starts = [int(round(q * (n - planes) / max(nslab - 1, 1))) for q in range(nslab)]
    times, vox, tris = [], 0, 0
    for s_i in range(args.warmup + args.steps):
        a = starts[s_i % len(starts)]
        sub = field[a:a + planes]
        dt, nt = time_oracle(sub, ISOVALUE, cores)
        if s_i >= args.warmup:
            times.append(dt)
            vox += (planes - 1) * (n - 1) * (n - 1)
            tris += nt
    tot = sum(times)
    val = vox / tot / 1e9
    sample = ("%d-plane z-slabs of the same %d^3 field per step (%d slabs, cycling), numpy oracle port "
              "(extract + normals), %d processes" % (planes, n, len(starts), cores))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Gvoxels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot / len(times) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, max(args.gpus, 1)),
            "mtris_per_s": tris / tot / 1e6,
            "cpu_baseline": {"value": val, "unit": "Gvoxels/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Gvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ our arm
DUMP_ROWS = 1 << 20     # vertex and triangle rows kept by --dump-outputs: 12.6 + 12.6 + 25.2 MB at most


def dump_outputs(out_dir, counts, mesh):
    """--dump-outputs: what a caller of the timed path receives -- the counts and the mesh mt3d_fetch() returns -- as
    DIR/{counts,verts,normals,tris}.npy (float32 geometry, float64 counts and triangle vertex ids).  Above DUMP_ROWS
    rows, verts / normals keep the same fixed sample of vertex rows and tris a fixed sample of triangle rows (seed 0,
    in row order): two builds with the same counts are compared on the same rows."""
    rng = np.random.default_rng(0)

    def rows(n):
        return np.arange(n) if n <= DUMP_ROWS else np.sort(rng.choice(n, DUMP_ROWS, replace=False))
    vi, ti = rows(len(mesh["verts"])), rows(len(mesh["tris"]))
    arrays = {"counts": np.array([counts.n_verts, counts.n_tris], dtype=np.float64),
              "verts": mesh["verts"][vi], "tris": mesh["tris"][ti].astype(np.float64)}
    if mesh["normals"] is not None:
        arrays["normals"] = mesh["normals"][vi]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def c5_strong(eng, world, rank, dev, stream, n=2048, chunk=256, steps=2, warmup=1):
    """BASELINE configs[4]: the 2048^3 fp32 turbulence field (isovalue 0), STRONG scaling: the volume is fixed and rank r
    takes 1/N of the owner planes, walking them in chunks of `chunk` planes (the 32 GiB field is generated chunk by
    chunk on the device and never resident at once; generation is not timed).  Job time = slowest rank's sum over its
    chunks + the all-gather of the per-rank counts (tools/bench_c5.py is the stand-alone form of this leg)."""
    import torch
    import torch.distributed as dist
    from contourist_b200 import engine as E
    from contourist_b200 import sharding, synthetic
    a_r, b_r = sharding.slab_bounds(n, world)[rank]
    tot_ms, nv, nt = 0.0, 0, 0
    for a in range(a_r, b_r, chunk):
        b = min(a + chunk, b_r)
        lo, hi, kw = sharding.slab_with_halo(a, b, n)
        f = synthetic.turbulence(n, lo, hi, device=dev, n_total=n)
        shape = (hi - lo, n, n)
        run = lambda: eng.mt3d_run(f.data_ptr(), 0.0, shape=shape, dtype=np.float32, flags=E.WANT_NORMALS, **kw)
        for _ in range(warmup):
            c = run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            c = run()
        e1.record(stream)
        torch.cuda.synchronize()
        tot_ms += e0.elapsed_time(e1) / steps
        nv += int(c.n_verts)
        nt += int(c.n_tris)
        del f
    mine = torch.tensor([nv, nt], dtype=torch.int64, device=dev)
    t = torch.tensor([tot_ms, 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        out = torch.zeros(2 * world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(out, mine)
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            dist.all_gather_into_tensor(out, mine)
        e1.record()
        torch.cuda.synchronize()
        t[1] = e0.elapsed_time(e1) / 10
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot = out.view(world, 2).sum(0)
    else:
        tot = mine
    ms = float(t[0]) + float(t[1])
    V, T = int(tot[0]), int(tot[1])
    alg = float(n) ** 3 * 4 + V * 24.0 + T * 12.0
    peak, _ = peaks()
    torch.cuda.empty_cache()
    return {"workload": "BASELINE configs[4]: %d^3 fp32 turbulence (64 sines), isovalue 0, z-slabs over %d GPU(s), chunks of %d planes"
                        % (n, world, chunk), "scaling": "strong", "n_gpus": world, "ms_total": ms, "allgather_ms": float(t[1]),
            "value": float(n) ** 3 / ms / 1e6, "unit": "Gvoxels/s", "mtris_per_s": T / ms / 1e3, "n_verts": V, "n_tris": T,
            "steps": steps, "warmup": warmup,
            "roofline_frac_per_gpu": alg / ms / 1e6 / world / peak}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from contourist_b200 import engine as E
    from contourist_b200 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL_DEBUG=VERSION makes NCCL print its version on rank 0's stdout, in front of the one JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # whatever NCCL logs: not on the JSON line's stream
        dist.init_process_group("nccl", device_id=dev)
    n = args.n
    # this rank's slab of the (n*world) x n x n volume, with halo planes (1 below, 2 above)
    n_total = n * world
    a, b = rank * n, (rank + 1) * n
    lo, hi = max(a - 1, 0), min(b + 2, n_total)
    field = synthetic.ct_like(n, lo, hi, device=dev, n_total=n_total)
    shape = (hi - lo, n, n)
    eng = E.Engine(local)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_timing(True)
    flags = E.WANT_NORMALS if not os.environ.get("CTR_BENCH_NO_NORMALS") else 0   # (diagnostic switch; the metric needs normals)
    # The collective of the path: all-gather of (n_verts, n_tris) -> exclusive scan = global vertex / triangle offsets.
    # The counts never visit the host: the engine stores them on the device behind the extraction's last kernel
    # (ctr_mt3d_publish_counts) and the all-gather is queued on the same stream right behind it, before the host has
    # even seen the counts; ctr_mt3d_finish waits for the extraction only (an event behind its last kernel), so the host
    # is already enqueueing step k+1 while the collective of step k runs.  Measured on 8 B200 (profiles/): 0.417 ms per
    # step against 0.407 on one GPU; the same collective on a side stream (CTR_BENCH_AG=side) costs more (0.458 ms:
    # the NCCL kernel then competes with the extraction kernels), the round-1 form with a host round trip 0.553 ms.
    counts_dev = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(2)]
    gathered = [torch.zeros(2 * world, dtype=torch.int64, device=dev) for _ in range(2)]
    # CTR_BENCH_AG (diagnostic): "main" (default), "side" = the same all-gather on a side stream, "none" = no collective
    ag_mode = os.environ.get("CTR_BENCH_AG", "main")
    side = torch.cuda.Stream(device=dev) if (world > 1 and ag_mode == "side") else None
    ev_done = [torch.cuda.Event() for _ in range(2)]        # extraction of the slot finished (main stream)
    ev_sent = [None, None]                                  # all-gather of the slot finished (side stream)
    n_step = [0]

    # Two contexts on the same stream take the steps in turn and step k+1 is queued (ctr_mt3d_enqueue, and behind it the
    # all-gather of its counts) before the host waits for step k (ctr_mt3d_finish), so the device never waits for the
    # host's wake-up and first launch between two extractions (~10 us per 0.35 ms step with a synchronous step); every
    # step still is one complete extraction with its counts read back by the host (and, on several GPUs, all-gathered).
    eng_b = E.Engine(local)
    eng_b.set_stream(stream.cuda_stream)
    engines = (eng, eng_b)
    pending = [None]

    def step_sync():
        return eng.mt3d_run(field.data_ptr(), ISOVALUE, shape=shape, dtype=np.float32, flags=flags,
                            i_lo=a - lo, i_hi=b - lo, plane_offset=lo)

    def step():
        slot = n_step[0] & 1
        n_step[0] += 1
        e = engines[slot]
        if world > 1:
            if ev_sent[slot] is not None:
                stream.wait_event(ev_sent[slot])            # the slot's previous counts have been sent (two steps ago)
            e.mt3d_publish_counts(counts_dev[slot].data_ptr())
        e.mt3d_enqueue(field.data_ptr(), ISOVALUE, shape=shape, dtype=np.float32, flags=flags,
                       i_lo=a - lo, i_hi=b - lo, plane_offset=lo)
        if world > 1 and side is not None:
            ev_done[slot].record(stream)
            with torch.cuda.stream(side):
                side.wait_event(ev_done[slot])
                dist.all_gather_into_tensor(gathered[slot], counts_dev[slot])
                if ev_sent[slot] is None:
                    ev_sent[slot] = torch.cuda.Event()
                ev_sent[slot].record(side)
        elif world > 1 and ag_mode == "main":
            dist.all_gather_into_tensor(gathered[slot], counts_dev[slot])
        prev, pending[0] = pending[0], e
        return prev.mt3d_finish() if prev is not None else None

    def flush():
        if side is not None:
            stream.wait_stream(side)
        if pending[0] is not None:
            prev, pending[0] = pending[0], None
            return prev.mt3d_finish()
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 2)):              # (both contexts size their pools)
        step()
    flush()
    barrier()
    # per-stage CUDA-event times come from a separate instrumented pass (the event records and their read-back sit
    # between the kernels and after every run); the timed region below runs with the instrumentation off
    stage_acc = np.zeros(8)
    n_inst = max(3, min(args.steps, 10))
    for _ in range(n_inst):
        c = step_sync()                               # (no collective: the same on every rank)
        stage_acc += np.array(eng.stage_times(8)) / n_inst
    eng.set_timing(False)
    step()
    c = flush() or c
    barrier()
    # nvidia-smi samples every 100 ms and K steps may last a few ms: the same steps run untimed for ~0.4 s right before
    # the timed region (same count on every rank: each step holds a collective), so that the clock samples are taken
    # under this load and the timed steps start on a GPU already at its sustained state
    PRELOAD = 800
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(PRELOAD):
        step()
    c = flush() or c
    l0 = eng.kernel_launches() + eng_b.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cs = step()
        c = cs if cs is not None else c
    c = flush() or c                                  # one all-gather per step inside the timed region
    ev1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    sampler.mark()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.kernel_launches() + eng_b.kernel_launches() - l0
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "%d untimed steps of the same loop directly before the timed region, and the timed region" % PRELOAD
    if args.dump_outputs and rank == 0:                  # the context of the last timed step still holds its mesh
        dump_outputs(args.dump_outputs, c, engines[(n_step[0] - 1) & 1].mt3d_fetch())
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([c.n_tris, c.n_verts], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_step = float(tmax.item()) / args.steps
    vox_all = float(n) ** 3 * world
    value = vox_all / (ms_step * 1e-3) / 1e9
    n_tris_all, n_verts_all = int(tot[0].item()), int(tot[1].item())
    if world > 1:                                     # the offsets the last timed step gathered are the real ones
        g = gathered[(n_step[0] - 1) & 1].view(world, 2).sum(0)
        assert ag_mode == "none" or (int(g[0]) == n_verts_all and int(g[1]) == n_tris_all), (g, n_verts_all, n_tris_all)

    # ---- the same K steps with fp64 geometry (the reference's arithmetic; north_star's 1e-6 mode): secondary number
    f64 = None
    if world == 1 and not args.no_e2e:
        fl64 = flags | E.GEOM_F64
        run64 = lambda: eng.mt3d_run(field.data_ptr(), ISOVALUE, shape=shape, dtype=np.float32, flags=fl64)
        for _ in range(3):
            run64()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            run64()
        e1.record(stream)
        torch.cuda.synchronize()
        ms64 = e0.elapsed_time(e1) / args.steps
        f64 = {"ms_per_step": ms64, "value": float(n) ** 3 / (ms64 * 1e-3) / 1e9, "unit": "Gvoxels/s",
               "note": "positions and normals computed and stored in fp64 (CTR_GEOM_F64: 0 ulp vs the oracle), same field"}
        eng.mt3d_run(field.data_ptr(), ISOVALUE, shape=shape, dtype=np.float32, flags=flags)   # pools back to fp32 sizes

    # ---- end-to-end through the C ABI with HOST buffers (H2D of the field + D2H of the mesh in the timed region)
    host_field = torch.empty(field.shape, dtype=torch.float32, pin_memory=True)
    host_field.copy_(field)
    hf = host_field.numpy()
    e2e_times = []
    outs = None
    # the call a user makes: an engine of its own (own stream), not the context the loops above bound to torch's stream
    # -- on the legacy default stream the same calls showed sporadic 40-110 ms stalls in this process, none on a
    # stream of the engine's own
    eng_host = None if args.no_e2e else E.Engine(local)
    E2E_WARM = 6          # untimed calls: pools sized on the first, page-locked output buffers touched, lazy module loads
    E2E_CALLS = 15        # timed calls; the value is their MEDIAN: on the shared boxes of the pool single calls of this
                          # PCIe- and host-bound leg stall for 40-240 ms now and then (the same loop in a process of
                          # its own on a quiet box: 10.54-10.58 ms for 40 calls in a row); every call is listed in the line
    for s in range(0 if args.no_e2e else E2E_WARM + E2E_CALLS):
        barrier()
        t1 = time.perf_counter()
        # the host-array call of the engine: slabs uploaded / extracted / downloaded in a pipeline (every rank its own slab)
        tot_e, outs = eng_host.mt3d_extract_host(hf, ISOVALUE, flags=flags, nslabs=args.e2e_slabs, own=(a - lo, b - lo), plane_offset=lo)
        if world > 1:
            counts_dev[0].copy_(torch.tensor([tot_e["n_verts"], tot_e["n_tris"]], dtype=torch.int64))
            dist.all_gather_into_tensor(gathered[0], counts_dev[0])
        barrier()
        if s >= E2E_WARM:
            e2e_times.append(time.perf_counter() - t1)
    # what the platform gives: this rank's H2D rate while every rank copies its field at the same time
    h2d_gbs = None
    if not args.no_e2e:
        barrier()
        t1 = time.perf_counter()
        for _ in range(3):
            field.copy_(host_field, non_blocking=True)
        torch.cuda.synchronize()
        h2d_gbs = 3 * hf.nbytes / (time.perf_counter() - t1) / 1e9
        barrier()
    e2e_t = torch.tensor([float(np.median(e2e_times)) if e2e_times else float('nan'),
                          float(np.mean(e2e_times)) if e2e_times else float('nan')], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = vox_all / float(e2e_t[0].item()) / 1e9
    e2e_mean_val = vox_all / float(e2e_t[1].item()) / 1e9
    h2d = hf.nbytes
    d2h = (outs["verts"].nbytes + outs["normals"].nbytes + outs["tris"].nbytes) if outs else 0

    # ---- the mesh passes that follow an extraction (not part of the metric): reference orientation, seeded selection
    post = None
    if world == 1 and not args.no_e2e:
        post = {}
        idx = int(torch.argmax(field))
        pi, pj, pk = idx // (shape[1] * shape[2]), (idx // shape[2]) % shape[1], idx % shape[2]
        row = field[pi, pj].cpu().numpy()
        while pk + 1 < shape[2] and row[pk + 1] >= ISOVALUE:
            pk += 1                                   # last sample of the row still above the isovalue: a border voxel
        for name in ("orient_reference", "select_seeded", "clean_reference"):
            ts = []
            for _ in range(3):
                run_c = eng.mt3d_run(field.data_ptr(), ISOVALUE, shape=shape, dtype=np.float32, flags=flags)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                if name == "orient_reference":
                    res = eng.mt3d_orient_reference()
                elif name == "select_seeded":
                    res = eng.mt3d_select_seeded(np.array([[min(pi, shape[0] - 2), min(pj, shape[1] - 2), min(pk, shape[2] - 2)]], np.int32))
                else:
                    # the reference's whole post-processing (quantize, tiny, clean, orient; tetrahedral.py:541-552); at 511
                    # voxels per axis its quantum is 1/19 of a voxel, so it merges a lot -- faithfully
                    cc = eng.mt3d_clean([shape[0] - 1, shape[1] - 1, shape[2] - 1], orient=True)
                    res = [int(cc.n_verts), int(cc.n_tris), int(cc.n_quantized), int(cc.n_tiny), int(cc.n_flat), int(cc.n_components)]
                ts.append((time.perf_counter() - t1) * 1e3)
            post[name] = {"ms": min(ts), "result": list(res), "n_tris_in": int(run_c.n_tris)}

    # CPU baseline sample: a block from the middle of this rank's field
    c0 = (n - 160) // 2
    p0 = min(n // 2, shape[0] - 34)
    sub = field[p0:p0 + 33, c0:c0 + 160, c0:c0 + 160].cpu().numpy()
    c5 = None
    if not args.no_c5 and not args.no_e2e:
        del host_field, hf, field
        torch.cuda.empty_cache()
        c5 = c5_strong(eng, world, rank, dev, stream)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    traffic, traffic_src = measured_traffic()
    st = stage_acc                                    # ms: 0 H2D, 1 classify, 2 count+scan, 3 verts, 4 tris
    field_bytes = float(np.prod(shape)) * 4
    # SURVEY 8(d) algorithmic bytes: 4 B per voxel read (stage 1), 24 B per vertex (stage 3), 12 B per triangle (stage 4);
    # the scan (stage 2) moves no algorithmic bytes -- it is pure overhead and is charged to the whole-step figure.
    stages = {"k_bitplane_tma (stage 1: field -> low/near bitplanes, the only full-field pass)": (st[1], field_bytes),
              "k_emit_verts (stage 3: positions + normals)": (st[3], c.n_verts * 24.0),
              "k_emit_tris (stage 4: indexed triangles)": (st[4], c.n_tris * 12.0)}
    per_stage = {k.split(" ")[0]: {"ms": v[0], "algorithmic_bytes": v[1],
                                   "gbs": (v[1] / (v[0] * 1e-3) / 1e9) if v[0] > 0 else None,
                                   "frac": (v[1] / (v[0] * 1e-3) / 1e9 / peak) if v[0] > 0 else None}
                 for k, v in stages.items()}
    per_stage["k_count_a+k_count_b+k_scan"] = {"ms": st[2], "algorithmic_bytes": 0.0, "gbs": 0.0, "frac": 0.0}
    kern_ms = float(st[1] + st[2] + st[3] + st[4])    # the four kernels of one extraction, from CUDA events on their stream
    dom = max(per_stage, key=lambda k: per_stage[k]["ms"])
    alg_total = float(n) ** 3 * 4 + c.n_verts * 24 + c.n_tris * 12        # SURVEY 8(d): field + V*(3p+3p) + T*12
    pipe_gbs = alg_total / (ms_step * 1e-3) / 1e9
    # CPU baseline: oracle port, 1 core, bounded sample of the same field family
    t_cpu, _ = time_oracle(sub, ISOVALUE, 1) if not args.no_e2e else (float('nan'), 0)
    cpu_val = sub.size / t_cpu / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "Gvoxels/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(n, world),
        "untimed_steps": {"warmup": args.warmup, "instrumented": n_inst + 1, "clock_preload": PRELOAD,
                          "note": "after the W warm-up steps: a CUDA-event instrumented pass for the per-stage times, then the "
                                  "same step repeated untimed so that nvidia-smi samples the clocks under this load"},
        "mtris_per_s": n_tris_all / (ms_step * 1e-3) / 1e6, "n_tris": n_tris_all, "n_verts": n_verts_all,
        "stage_ms": {"bitplane": st[1], "count_scan": st[2], "emit_verts": st[3], "emit_tris": st[4],
                     "wall_ms_per_step": wall / args.steps * 1e3},
        # one extraction = one launch each of four kernels; SURVEY 8(d) defines the algorithmic bytes per extraction, so the
        # roofline is taken over the four launches together (the scan kernel moves no algorithmic bytes of its own)
        "roofline": {"bound": "hbm", "kernel": "mt3d extraction = k_reset3 + k_bitplane_tma + k_count_a + k_count_b + k_scan + k_emit_verts + k_emit_tris + k_counts_out "
                                                "(largest share: %s, %.0f%% of the kernel time)" % (dom, 100.0 * per_stage[dom]["ms"] / kern_ms),
                     "achieved": alg_total / (kern_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": alg_total / (kern_ms * 1e-3) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_total, "kernel_ms": kern_ms, "per_stage": per_stage},
        "pipeline_roofline": {"algorithmic_bytes": alg_total, "achieved": pipe_gbs, "frac": pipe_gbs / peak,
                              "note": "whole step: (field + V*24 + T*12) / device time of the step"},
        "cpu_baseline": {"value": cpu_val, "unit": "Gvoxels/s", "cores": 1, "kind": "port",
                         "sample": "33x160x160 block from the middle of the same field, numpy oracle port (extract + normals)"},
        "e2e": {"value": e2e_val, "unit": "Gvoxels/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "h2d_copy_gbs_rank0_all_ranks_copying": h2d_gbs, "ms_per_call_rank0": [round(t * 1e3, 3) for t in e2e_times],
                "statistic": "median of %d calls after %d untimed ones (max over ranks)" % (E2E_CALLS, E2E_WARM), "value_from_mean": e2e_mean_val,
                "note": "Engine.mt3d_extract_host (volume uploaded once, plane by plane, by ctr_stage_upload on an upload context; ctr_mt3d_enqueue / _finish / _fetch per z-slab on two contexts, slab s+1 queued "
                        "while slab s runs, page-locked host buffers): H2D of the field and D2H of vertices, normals and "
                        "triangles inside the timed region"},
        "gpu_launches": int(launches), "clocks": clocks,
        "stepping": "two contexts on one stream take the steps in turn; step k+1 (and, on several GPUs, the all-gather of its "
                    "device counts behind it) is queued before the host waits for the counts of step k; every step is one "
                    "complete extraction",
        "f64_geom": f64, "c5_strong": c5,
        "post_passes": post,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--e2e-slabs", type=int, default=8, help="slabs of the pipelined host-array call (1 = run + fetch)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg and the CPU baseline (profiling runs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the 2048^3 strong-scaling leg (c5_strong)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the mesh of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
