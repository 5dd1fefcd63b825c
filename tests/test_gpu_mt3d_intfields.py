"""GPU: uint8 / int16 / uint16 fields in the 3D extraction.  An integer field gives exactly the arrays of the same call
on its float64 copy (both geometry modes) and, with fp32 geometry, of its float32 copy: counts, vertices, normals,
triangles, keys, lowmin bit for bit; cells and case codes as sets."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

INTS = [np.uint8, np.int16, np.uint16]
ALLCLOSE_BITS = sum(1 << (5 * t + 4) for t in range(6))      # the "all four corners allclose" bit of every tet code


def _flags(geom64, codes=True, minmax=True):
    from contourist_b200 import engine as E
    return (E.WANT_KEYS | E.WANT_NORMALS | (E.WANT_CODES if codes else 0) | (E.WANT_MINMAX if minmax else 0)
            | (E.GEOM_F64 if geom64 else 0))


def _run(engine, field, value, flags, **kw):
    c = engine.mt3d_run(field, value, flags=flags, **kw)
    out = engine.mt3d_fetch()
    return c, out


def _assert_same(a, b):
    (ca, oa), (cb, ob) = a, b
    for name in ("n_verts", "n_tris", "n_active_cells", "n_crossings", "n_codes"):
        assert getattr(ca, name) == getattr(cb, name), name
    for name in ("fmin", "fmax"):                             # NaN both: the run did not ask for them
        x, y = getattr(ca, name), getattr(cb, name)
        assert x == y or (np.isnan(x) and np.isnan(y)), (name, x, y)
    for name in ("verts", "normals", "tris", "keys", "lowmin"):
        if oa[name] is not None or ob[name] is not None:
            assert oa[name].dtype == ob[name].dtype and np.array_equal(oa[name], ob[name]), name
    if oa["cells"] is not None:
        pa, pb = np.argsort(oa["cells"]), np.argsort(ob["cells"])
        assert np.array_equal(oa["cells"][pa], ob["cells"][pb])
        assert np.array_equal(oa["codes"][pa], ob["codes"][pb])


def check_int_field(engine, field, value, geom64, codes=True):
    """Run the integer field and its float copies; return the integer run."""
    assert field.dtype in INTS
    flags = _flags(geom64, codes)
    ri = _run(engine, field, value, flags)
    assert ri[0].fmin == field.min() and ri[0].fmax == field.max()
    _assert_same(ri, _run(engine, field.astype(np.float64), value, flags))
    if not geom64:
        _assert_same(ri, _run(engine, field.astype(np.float32), value, flags))
    return ri


# ---------------------------------------------------------------------------------------------- 1. reference golden
@pytest.mark.parametrize("dt,shift", [(np.int16, 0), (np.uint8, 1), (np.uint16, 1)])
@pytest.mark.parametrize("geom64", [True, False])
def test_golden_ints7(engine, dt, shift, geom64):
    from contourist_b200 import engine as E
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    field = (g["field"] + shift).astype(dt)
    value = float(g["value"]) + shift
    c, raw = check_int_field(engine, field, value, geom64)
    o = E.canonical_mesh(raw)
    n0, n1, n2 = field.shape
    klow, khigh = g["key_low"], g["key_high"]
    pmin = np.minimum(klow, khigh)
    d = np.maximum(klow, khigh) - pmin
    gk = ((((pmin[:, 0] * n1 + pmin[:, 1]) * n2 + pmin[:, 2]).astype(np.uint64) << np.uint64(3))
          | (d[:, 0] * 4 + d[:, 1] * 2 + d[:, 2]).astype(np.uint64))
    srt = np.argsort(gk)
    assert np.array_equal(gk[srt], o["keys"])
    if geom64:
        assert np.array_equal(g["key_pos"][srt], o["verts"])
    else:
        assert np.array_equal(g["key_pos"][srt].astype(np.float32), o["verts"])
    assert len(g["tris"]) == c.n_tris


# ---------------------------------------------------------------------------------------------- 2. random fields
SHAPES = [(2, 2, 2), (9, 9, 129), (40, 40, 64), (7, 33, 96), (5, 6, 32)]


def _random_field(rng, shape, dt):
    info = np.iinfo(dt)
    mid = (int(info.min) + int(info.max)) // 2
    f = mid + rng.integers(-3, 4, size=shape)                 # narrow range: plateaus and exact contacts
    f = f.astype(dt)
    f.flat[rng.integers(0, f.size, size=max(1, f.size // 50))] = info.min
    f.flat[rng.integers(0, f.size, size=max(1, f.size // 50))] = info.max
    return f, mid


@pytest.mark.parametrize("shape", SHAPES, ids=["x".join(map(str, s)) for s in SHAPES])
@pytest.mark.parametrize("dt", INTS, ids=[np.dtype(d).name for d in INTS])
@pytest.mark.parametrize("geom64", [True, False])
def test_random_fields(engine, shape, dt, geom64):
    rng = np.random.default_rng(int(np.prod(shape)) * 7 + np.dtype(dt).itemsize * 3 + (np.dtype(dt).kind == "i"))
    f, mid = _random_field(rng, shape, dt)
    info = np.iinfo(dt)
    values = [mid, mid + 0.5, mid - 1.5, float(info.min) - 0.5, float(info.max) + 0.5, float(info.min), float(info.max),
              info.min + 0.5, info.max - 0.5, np.inf, -np.inf, 1e12, -1e12]
    for v in values:
        check_int_field(engine, f, float(v), geom64)


@pytest.mark.parametrize("dt", INTS, ids=[np.dtype(d).name for d in INTS])
def test_full_range_extremes(engine, dt):
    info = np.iinfo(dt)
    rng = np.random.default_rng(3)
    f = np.where(rng.random((12, 10, 64)) < 0.5, info.min, info.max).astype(dt)
    for v in (float(info.min), float(info.max), (float(info.min) + float(info.max)) / 2, info.min + 0.5, info.max - 0.5):
        for geom64 in (True, False):
            c, _ = check_int_field(engine, f, v, geom64)
            assert c.fmin == info.min and c.fmax == info.max


def test_misaligned_device_pointer(engine):
    """A device pointer that is not 16-byte aligned takes the generic stage-1 kernel."""
    import torch
    from contourist_b200 import engine as E
    rng = np.random.default_rng(5)
    f, mid = _random_field(rng, (8, 9, 64), np.uint16)
    flags = _flags(True, codes=False)
    want = _run(engine, f.astype(np.float64), mid + 0.5, flags)
    buf = torch.zeros(f.size + 8, dtype=torch.uint16, device="cuda")
    buf[1:1 + f.size] = torch.from_numpy(f.reshape(-1).astype(np.int32)).to("cuda").to(torch.uint16)
    torch.cuda.synchronize()
    c = engine.mt3d_run(buf.data_ptr() + 2, mid + 0.5, flags=flags | E.FIELD_ON_DEVICE, shape=f.shape, dtype=np.uint16)
    assert c.fmin == f.min() and c.fmax == f.max()
    _assert_same((c, engine.mt3d_fetch()), want)


def _off_alignment(field):
    """A device copy of `field` one sample past a 16-byte boundary: (buffer to keep alive, pointer)."""
    import torch
    tdt = {np.uint8: torch.uint8, np.int16: torch.int16, np.uint16: torch.uint16, np.float32: torch.float32,
           np.float64: torch.float64}[field.dtype.type]
    buf = torch.zeros(field.size + 16, dtype=tdt, device="cuda")
    flat = field.reshape(-1)
    src = torch.from_numpy(flat.astype(np.int32) if flat.dtype.kind in "iu" else flat)
    buf[1:1 + field.size] = src.to("cuda").to(tdt)
    torch.cuda.synchronize()
    return buf, buf.data_ptr() + field.itemsize


@pytest.mark.parametrize("layout", ["aligned", "off_alignment", "rows129"])
@pytest.mark.parametrize("dt", INTS, ids=[np.dtype(d).name for d in INTS])
def test_stage1_choice(engine, layout, dt):
    """Both stage-1 kernels give the float64 result: rows a multiple of 32 samples from an aligned buffer (TMA), the same
    field from a device pointer one sample off alignment and rows of 129 samples (generic)."""
    from contourist_b200 import engine as E
    rng = np.random.default_rng(7)
    f, mid = _random_field(rng, (12, 10, 129 if layout == "rows129" else 64), dt)
    for v in (mid, mid + 0.5, mid - 2.0):
        for geom64 in (True, False):
            if layout != "off_alignment":
                check_int_field(engine, f, float(v), geom64)
                continue
            flags = _flags(geom64)
            buf, ptr = _off_alignment(f)
            c = engine.mt3d_run(ptr, float(v), flags=flags | E.FIELD_ON_DEVICE, shape=f.shape, dtype=dt)
            ri = (c, engine.mt3d_fetch())
            del buf
            assert c.fmin == f.min() and c.fmax == f.max()
            _assert_same(ri, _run(engine, f.astype(np.float64), float(v), flags))
            if not geom64:
                _assert_same(ri, _run(engine, f.astype(np.float32), float(v), flags))


def _stage1_kernels(engine, field, value, off_alignment=False):
    """The stage-1 kernel instances of one run, as `k_bitplane_<path><first template argument`."""
    import re
    import torch
    from torch.profiler import ProfilerActivity, profile
    from contourist_b200 import engine as E
    flags = _flags(False, codes=False, minmax=False)
    arg, kw = field, {}
    if off_alignment:
        buf, arg = _off_alignment(field)
        flags |= E.FIELD_ON_DEVICE
        kw = dict(shape=field.shape, dtype=field.dtype.type)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.mt3d_run(arg, value, flags=flags, **kw)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("k_emit_verts" in n for n in names), "the profiler did not see the extraction's kernels"
    return sorted({m.group(1) for n in names for m in [re.search(r"(k_bitplane_\w+<[^,>]+)", n)] if m})


FLOATS = [np.float32, np.float64]
CTYPE = {np.uint8: "unsigned char", np.int16: "short", np.uint16: "unsigned short", np.float32: "float",
         np.float64: "double"}


def _field(rng, shape, dt):
    if dt in FLOATS:
        return rng.standard_normal(shape).astype(dt), 0.0
    return _random_field(rng, shape, dt)


@pytest.mark.parametrize("layout", ["aligned", "off_alignment", "rows129"])
@pytest.mark.parametrize("dt", INTS + FLOATS, ids=[np.dtype(d).name for d in INTS + FLOATS])
def test_stage1_kernel_that_runs(engine, dt, layout):
    """Rows of 32k samples from an aligned buffer take the TMA kernel of the field's sample type; the same rows from a
    device pointer one sample off alignment, and rows of 129 samples, its generic kernel."""
    rng = np.random.default_rng(9)
    f, mid = _field(rng, (9, 9, 129) if layout == "rows129" else (16, 12, 64), dt)
    kind = "tma" if layout == "aligned" else "generic"
    got = _stage1_kernels(engine, f, mid + 0.5, off_alignment=layout == "off_alignment")
    assert got == ["k_bitplane_%s<%s" % (kind, CTYPE[dt])]


@pytest.mark.parametrize("dt", FLOATS, ids=[np.dtype(d).name for d in FLOATS])
def test_minmax_partial_last_chunk(engine, dt):
    """fmin / fmax of float fields on the TMA path whose size in bytes is not a multiple of the kernel's 16 KiB chunk:
    the stale tail of the last chunk takes no part, in 3D and in 4D."""
    from contourist_b200 import engine as E
    rng = np.random.default_rng(13)
    for shape in ((5, 7, 64), (9, 33, 96)):
        f = (rng.standard_normal(shape) + 1.0).astype(dt)
        assert f.nbytes % 16384 != 0
        c = engine.mt3d_run(f, 1.0, flags=E.WANT_MINMAX)
        assert (c.fmin, c.fmax) == (f.min(), f.max()), shape
    for shape in ((4, 5, 6, 64), (3, 4, 5, 96)):
        f = (rng.standard_normal(shape) + 1.0).astype(dt)
        assert f.nbytes % 16384 != 0
        c = engine.mp4d_run(f, 1.0, flags=E.WANT_MINMAX)
        assert (c.fmin, c.fmax) == (f.min(), f.max()), shape


# ---------------------------------------------------------------------------------------------- 3. near hull
@pytest.mark.parametrize("geom64", [True, False])
def test_near_hull_large_magnitude(engine, geom64):
    rng = np.random.default_rng(11)
    f = (60000 + rng.integers(-1, 3, size=(16, 12, 64))).astype(np.uint16)
    seen = False
    for v in (60000.5, 59999.5, 60001.5):
        c, out = check_int_field(engine, f, v, geom64)
        seen = seen or bool(np.any(out["codes"].astype(np.int64) & ALLCLOSE_BITS))
    assert seen, "no tet was skipped by np.allclose: the exact path did not run"


# ---------------------------------------------------------------------------------------------- 4. pipelines
def _smooth_u16(shape=(48, 40, 64)):
    n0, n1, n2 = shape
    x, y, z = np.meshgrid(np.linspace(-1, 1, n0), np.linspace(-1, 1, n1), np.linspace(-1, 1, n2), indexing="ij")
    q = np.sin(3 * x) * np.cos(2 * y) + 0.7 * z * z
    return np.clip(np.round((q + 2.0) * 4096), 0, 65535).astype(np.uint16)


def test_enqueue_finish(engine):
    f = _smooth_u16()
    flags = _flags(False, codes=False)
    want = _run(engine, f, 8192.0, flags)
    engine.mt3d_enqueue(f, 8192.0, flags=flags)
    c = engine.mt3d_finish()
    _assert_same((c, engine.mt3d_fetch()), want)


def test_slab_sharding_concatenates(engine):
    from contourist_b200 import sharding
    f = _smooth_u16()
    flags = _flags(True, codes=False, minmax=False)
    cw, ow = _run(engine, f, 8192.5, flags)
    keys, verts, nt = [], [], 0
    for (a, b) in sharding.slab_bounds(f.shape[0], 3):
        lo, hi, kw = sharding.slab_with_halo(a, b, f.shape[0])
        c, o = _run(engine, np.ascontiguousarray(f[lo:hi]), 8192.5, flags, **kw)
        keys.append(o["keys"])
        verts.append(o["verts"])
        nt += int(c.n_tris)
    keys, verts = np.concatenate(keys), np.concatenate(verts)
    assert len(keys) == cw.n_verts and nt == cw.n_tris
    pa, pb = np.argsort(keys), np.argsort(ow["keys"])
    assert np.array_equal(keys[pa], ow["keys"][pb]) and np.array_equal(verts[pa], ow["verts"][pb])


@pytest.mark.parametrize("dt", [np.uint8, np.uint16])
def test_extract_host(engine, dt):
    from contourist_b200 import engine as E
    f = _smooth_u16()
    value = 8192.5
    if dt == np.uint8:
        f = (f >> 8).astype(np.uint8)
        value = 32.5
    flags = E.WANT_KEYS | E.WANT_NORMALS
    want = E.canonical_mesh(_run(engine, f, value, flags)[1])
    pinned = engine.pinned_empty("test_int_field", f.shape, dt)
    pinned[...] = f
    totals, out = engine.mt3d_extract_host(pinned, value, flags=flags, nslabs=4)
    got = E.canonical_mesh(out)
    assert totals["n_verts"] == len(want["keys"]) and totals["n_tris"] == len(want["tris"])
    for name in ("keys", "lowmin", "verts", "normals"):
        assert np.array_equal(got[name], want[name]), name
    assert np.array_equal(np.unique(np.sort(got["tris"], axis=1), axis=0), np.unique(np.sort(want["tris"], axis=1), axis=0))


def test_device_pointer(engine):
    import torch
    from contourist_b200 import engine as E
    f = _smooth_u16()
    flags = _flags(False, codes=False)
    want = _run(engine, f, 8192.0, flags)
    t = torch.from_numpy(f.astype(np.int32)).to("cuda").to(torch.uint16).contiguous()
    torch.cuda.synchronize()
    c = engine.mt3d_run(t.data_ptr(), 8192.0, flags=flags | E.FIELD_ON_DEVICE, shape=f.shape, dtype=np.uint16)
    _assert_same((c, engine.mt3d_fetch()), want)


# ---------------------------------------------------------------------------------------------- 5. facade
def _facade(field, value, seeds=None, post=True, orient=False):
    from contourist_b200 import tetrahedral
    n = [s - 1 for s in field.shape]
    g = tetrahedral.Grid3DContour(n[0], n[1], n[2], field, value, seeds)
    g.post_process = post
    g.reference_orientation = orient
    p, t = g.get_points_and_triangles()
    return np.array(p), np.array(t)


@pytest.mark.parametrize("post,orient", [(True, False), (False, True)])
def test_facade_int16(engine, post, orient):
    f = (_smooth_u16((24, 20, 33)).astype(np.int32) - 8192).astype(np.int16)
    p1, t1 = _facade(f, 0.5, post=post, orient=orient)
    p2, t2 = _facade(f.astype(np.float64), 0.5, post=post, orient=orient)
    assert len(t1) > 0
    assert np.array_equal(p1, p2) and np.array_equal(t1, t2)


def test_facade_seeded_uint8(engine):
    g = np.load(os.path.join(GOLDEN, "seeded3d_twodots.npz"))
    f8 = (g["field"] + 1).astype(np.uint8)
    seeds = [[tuple(int(x) for x in p) for p in s] for s in g["seeds"]]
    p1, t1 = _facade(f8, float(g["value"]) + 1, seeds=seeds)
    p2, t2 = _facade(f8.astype(np.float64), float(g["value"]) + 1, seeds=seeds)
    assert len(t1) > 0
    assert np.array_equal(p1, p2) and np.array_equal(t1, t2)


# ---------------------------------------------------------------------------------------------- 6. full size
@pytest.mark.parametrize("value", [2048.5, 2048.0])
def test_ct_like_512_uint16(engine, value):
    import torch
    from contourist_b200 import engine as E
    from contourist_b200.synthetic import ct_like
    q = ct_like(512)
    u = torch.clamp(torch.round(q * 4096), 0, 65535).to(torch.int32).to(torch.uint16).contiguous()
    f32 = u.to(torch.int32).to(torch.float32).contiguous()
    torch.cuda.synchronize()
    flags = _flags(False, codes=False) | E.FIELD_ON_DEVICE
    runs = []
    for t, dt in ((u, np.uint16), (f32, np.float32)):
        c = engine.mt3d_run(t.data_ptr(), value, flags=flags, shape=tuple(t.shape), dtype=dt)
        runs.append((c, engine.mt3d_fetch()))
    assert runs[0][0].n_tris > 1000000
    _assert_same(runs[0], runs[1])


# ---------------------------------------------------------------------------------------------- 7. rejections
def test_bad_dtype_code(engine):
    import ctypes
    from contourist_b200 import engine as E
    f = np.zeros((4, 4, 4), np.float32)
    p, _ = engine._mt3d_params(f, 0.5, (0, 0, 0), (1, 1, 1), 0, 0, None, 0, None, None, 0)
    p.dtype = 5
    c = E.Mt3dCounts()
    with pytest.raises(ValueError):
        engine._check(engine.lib.ctr_mt3d_run(engine.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_run")


@pytest.mark.parametrize("dt", INTS, ids=[np.dtype(d).name for d in INTS])
def test_2d_4d_device_int_rejected(engine, dt):
    import torch
    t = torch.zeros(4096, dtype=torch.float32, device="cuda")
    with pytest.raises(ValueError):
        engine.mt2d_run(t.data_ptr(), [0.5], shape=(16, 16), dtype=dt)
    with pytest.raises(ValueError):
        engine.mp4d_run(t.data_ptr(), 0.5, shape=(4, 4, 4, 4), dtype=dt)
    with pytest.raises(ValueError):
        engine.mt3d_run(t.data_ptr(), 0.5, shape=(4, 4, 4), dtype=np.int32)


def test_2d_4d_host_int_widened(engine):
    rng = np.random.default_rng(2)
    f2 = rng.integers(0, 5, size=(20, 24)).astype(np.uint16)
    c_i = engine.mt2d_run(f2, [1.5, 2.5])
    o_i = engine.mt2d_fetch()
    c_f = engine.mt2d_run(f2.astype(np.float64), [1.5, 2.5])
    o_f = engine.mt2d_fetch()
    assert c_i.n_segments == c_f.n_segments > 0
    assert np.array_equal(o_i["keys"], o_f["keys"]) and np.array_equal(o_i["pos"], o_f["pos"])
    f4 = rng.integers(0, 4, size=(6, 6, 6, 5)).astype(np.int16)
    c_i = engine.mp4d_run(f4, 1.5)
    o_i = engine.mp4d_fetch()
    c_f = engine.mp4d_run(f4.astype(np.float64), 1.5)
    o_f = engine.mp4d_fetch()
    assert c_i.n_tets == c_f.n_tets > 0
    assert np.array_equal(o_i["verts"], o_f["verts"]) and np.array_equal(o_i["tets"], o_f["tets"])
