"""GPU: per-vertex values of other fields on the 3D mesh (ctr_mt3d_interpolate, Engine.mt3d_interpolate, the façade's
vertex_fields).  Pinned by coordinate identity (the field of grid coordinates gives the vertex positions bit for bit)
and by oracle/mt3d_values.py:vertex_values."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))
DTYPES = [np.float64, np.float32, np.uint8, np.int16, np.uint16]


def _E():
    from contourist_b200 import engine as E
    return E


def _run(engine, field, value, geom64, extra=0, **kw):
    E = _E()
    c = engine.mt3d_run(field, value, flags=E.WANT_KEYS | (E.GEOM_F64 if geom64 else 0) | extra, **kw)
    return c, engine.mt3d_fetch()


def coords(shape, plane_offset=0, dtype=np.float64):
    c = np.stack(np.indices(shape), -1)
    c[..., 0] += plane_offset
    return c.astype(dtype)


def _random_attr(rng, shape, dt):
    if np.dtype(dt).kind == "f":
        return (rng.standard_normal(shape) * 100).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(info.min, int(info.max) + 1, size=shape).astype(dt)


# ---------------------------------------------------------------------------------------------- 1. coordinate identity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
@pytest.mark.parametrize("run_dt", [np.float64, np.float32])
def test_coordinates_give_positions_goldens(engine, path, geom64, run_dt):
    g = np.load(path)
    field = g["field"].astype(run_dt)
    c, out = _run(engine, field, float(g["value"]), geom64)
    assert c.n_verts > 0
    for adt in (np.float64, np.float32, np.int16):
        v = engine.mt3d_interpolate(coords(field.shape, dtype=adt))
        assert v.dtype == out["verts"].dtype and np.array_equal(v, out["verts"]), adt


@pytest.mark.parametrize("shape", [(6, 5, 32), (5, 7, 64), (4, 6, 129), (9, 3, 129)])
@pytest.mark.parametrize("geom64", [True, False])
def test_coordinates_give_positions_random_and_slabs(engine, shape, geom64):
    rng = np.random.default_rng(shape[2] * 31 + shape[0])
    for run_dt in (np.float64, np.float32):
        field = rng.standard_normal(shape).astype(run_dt)
        _, out = _run(engine, field, 0.1, geom64)
        assert np.array_equal(engine.mt3d_interpolate(coords(shape, dtype=np.float32)), out["verts"])
        # a slab of a taller volume: keys and positions are global, the attribute field is the slab's planes
        _, out = _run(engine, field, 0.1, geom64, i_lo=1, i_hi=shape[0] - 2, plane_offset=40)
        for adt in (np.float64, np.int16):
            assert np.array_equal(engine.mt3d_interpolate(coords(shape, 40, adt)), out["verts"])


def test_coordinates_integer_run_plateaus(engine):
    """uint16 run of the reference's integer golden (exact contacts: ratio-0.5 edges), float32 coordinates."""
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    for geom64 in (True, False):
        _, out = _run(engine, (g["field"] + 1).astype(np.uint16), float(g["value"]) + 1, geom64)
        assert np.array_equal(engine.mt3d_interpolate(coords(g["field"].shape, dtype=np.float32)), out["verts"])


# ---------------------------------------------------------------------------------------------- 2. oracle parity
@pytest.mark.parametrize("dt", DTYPES, ids=[np.dtype(d).name for d in DTYPES])
@pytest.mark.parametrize("ncomp", [0, 2, 3, 4])
def test_oracle_parity(engine, dt, ncomp):
    from oracle import mt3d_values
    rng = np.random.default_rng(ncomp * 10 + DTYPES.index(dt))
    shape = (9, 10, 37)
    field = rng.standard_normal(shape)
    ashape = shape if ncomp == 0 else shape + (ncomp,)
    attr = _random_attr(rng, ashape, dt)
    for geom64 in (True, False):
        gd = np.float64 if geom64 else np.float32
        _, out = _run(engine, field, 0.2, geom64)
        v = engine.mt3d_interpolate(attr)
        assert v.shape == ((len(out["keys"]),) if ncomp == 0 else (len(out["keys"]), ncomp))
        want = mt3d_values.vertex_values(field, 0.2, out["keys"], out["lowmin"], attr, gd)
        if geom64:
            assert np.array_equal(v, want)
        else:
            rng_a = float(attr.max()) - float(attr.min())
            np.testing.assert_allclose(v, want, rtol=1e-4, atol=1e-5 * rng_a)
        if np.dtype(dt).kind != "f":
            assert np.array_equal(v, engine.mt3d_interpolate(attr.astype(np.float64)))


# ---------------------------------------------------------------------------------------------- 3. after editing passes
def _by_key(keys, values, want_keys):
    o = np.argsort(keys)
    idx = o[np.searchsorted(keys, want_keys, sorter=o)]
    assert np.array_equal(keys[idx], want_keys)
    return values[idx]


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "seeded3d_*.npz"))),
                         ids=lambda p: os.path.basename(p))
def test_after_seeded_selection(engine, path):
    from contourist_b200 import tetrahedral
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    attr = _random_attr(np.random.default_rng(1), field.shape + (3,), np.float32)
    _, raw = _run(engine, field, value, True)
    raw_v = engine.mt3d_interpolate(attr)
    seeds = g["seeds"]
    start = tetrahedral.initial_voxels(field, value, seeds) if len(seeds) else np.zeros((0, 3), np.int32)
    nv, _, _ = engine.mt3d_select_seeded(start)
    sel = engine.mt3d_fetch()
    v = engine.mt3d_interpolate(attr)
    assert len(v) == nv == len(sel["keys"])
    assert np.array_equal(v, _by_key(raw["keys"], raw_v, sel["keys"]))


@pytest.mark.parametrize("geom64", [True, False])
def test_after_clean(engine, geom64):
    g = np.load(os.path.join(GOLDEN, "mt3d_noise8.npz"))
    field, value = g["field"], float(g["value"])
    attr = _random_attr(np.random.default_rng(2), field.shape, np.int16)
    _, raw = _run(engine, field, value, geom64)
    raw_v = engine.mt3d_interpolate(attr)
    cc = engine.mt3d_clean(np.array(field.shape) - 1, origin=(1.0, 2.0, 3.0), delta=(0.5, 0.5, 0.25), orient=True)
    fin = engine.mt3d_fetch()
    v = engine.mt3d_interpolate(attr)
    assert len(v) == cc.n_verts == len(fin["keys"])
    assert np.array_equal(v, _by_key(raw["keys"], raw_v, fin["keys"]))


# ---------------------------------------------------------------------------------------------- 4. sharding
@pytest.mark.parametrize("geom64", [True, False])
def test_slabs_match_the_full_run(engine, geom64):
    from contourist_b200 import sharding
    rng = np.random.default_rng(4)
    field = rng.standard_normal((23, 12, 40))
    attr = _random_attr(rng, field.shape + (2,), np.float64)
    _, full = _run(engine, field, 0.0, geom64)
    full_v = engine.mt3d_interpolate(attr)
    keys, vals = [], []
    for a, b in sharding.slab_bounds(field.shape[0], 4):
        lo, hi, kw = sharding.slab_with_halo(a, b, field.shape[0])
        _, out = _run(engine, np.ascontiguousarray(field[lo:hi]), 0.0, geom64, **kw)
        keys.append(out["keys"])
        vals.append(engine.mt3d_interpolate(np.ascontiguousarray(attr[lo:hi])))
    keys, vals = np.concatenate(keys), np.concatenate(vals)
    assert np.array_equal(np.sort(keys), np.sort(full["keys"]))
    assert np.array_equal(_by_key(keys, vals, full["keys"]), full_v)


# ---------------------------------------------------------------------------------------------- 5. paths
def test_device_fields_and_pipelines(engine):
    import torch
    E = _E()
    rng = np.random.default_rng(5)
    field = rng.standard_normal((10, 11, 48)).astype(np.float32)
    value = 0.05
    attrs = [_random_attr(rng, field.shape + (3,), np.float32), _random_attr(rng, field.shape + (4,), np.uint8),
             _random_attr(rng, field.shape + (2,), np.float64), _random_attr(rng, field.shape, np.int16)]
    _, out = _run(engine, field, value, False)
    want = [engine.mt3d_interpolate(a) for a in attrs]
    # the run's field on the device too
    dfield = torch.from_numpy(field).cuda()
    engine.mt3d_run(dfield.data_ptr(), value, flags=E.WANT_KEYS | E.FIELD_ON_DEVICE, shape=field.shape, dtype=np.float32)
    for a, w in zip(attrs, want):
        t = torch.from_numpy(a.reshape(-1).copy()).cuda()
        assert np.array_equal(engine.mt3d_interpolate(t.data_ptr(), shape=a.shape, dtype=a.dtype), w)
        # misaligned: the rows start one sample after an allocation boundary
        buf = torch.zeros(t.numel() + 1, dtype=t.dtype, device="cuda")
        buf[1:] = t
        torch.cuda.synchronize()
        assert np.array_equal(engine.mt3d_interpolate(buf.data_ptr() + a.itemsize, shape=a.shape, dtype=a.dtype), w)

    class DeviceValues(object):
        pass
    d = DeviceValues()
    d.__cuda_array_interface__ = dict(shape=want[-1].shape, typestr="<f4", data=(engine.mt3d_interpolate_device_ptr(), False),
                                      version=2)
    assert np.array_equal(torch.as_tensor(d, device="cuda").cpu().numpy(), want[-1])
    # a run finished through mt3d_enqueue / mt3d_finish, from a host field
    engine.mt3d_enqueue(field, value, flags=E.WANT_KEYS)
    engine.mt3d_finish()
    for a, w in zip(attrs, want):
        assert np.array_equal(engine.mt3d_interpolate(a), w)


def test_integer_run_with_float_attribute(engine):
    rng = np.random.default_rng(6)
    field = rng.integers(0, 7, size=(8, 9, 33)).astype(np.uint16)
    attr = _random_attr(rng, field.shape + (3,), np.float32)
    for geom64 in (True, False):
        _, a = _run(engine, field, 3.0, geom64)
        va = engine.mt3d_interpolate(attr)
        _, b = _run(engine, field.astype(np.float64), 3.0, geom64)
        assert np.array_equal(a["keys"], b["keys"])
        assert np.array_equal(va, engine.mt3d_interpolate(attr))


# ---------------------------------------------------------------------------------------------- 6. errors
def test_errors(engine):
    E = _E()
    field = np.random.default_rng(7).standard_normal((6, 6, 6))
    attr = np.zeros(field.shape)
    engine.mt3d_run(field, 0.0)                                        # no WANT_KEYS
    with pytest.raises(E.EngineError):
        engine.mt3d_interpolate(attr)
    engine.mt3d_run(field, 0.0, flags=E.WANT_KEYS | E.NO_GEOMETRY)
    with pytest.raises(E.EngineError):
        engine.mt3d_interpolate(attr)
    engine.mt3d_run(field, 0.0, flags=E.WANT_KEYS)
    for nc in (0, 5):
        with pytest.raises(ValueError):
            engine.mt3d_interpolate(np.zeros(field.shape + (nc,)))
    with pytest.raises(ValueError):
        engine.mt3d_interpolate(np.zeros((6, 6, 7)))                  # not the run's shape
    with pytest.raises(ValueError):
        engine.mt3d_interpolate(12345 * 256, shape=field.shape, dtype=np.int32)
    p = E.AttrParams()
    p.field, p.dtype, p.flags, p.ncomp = attr.ctypes.data, 9, 0, 1
    with pytest.raises(ValueError):
        engine._check(engine.lib.ctr_mt3d_interpolate(engine.h, p, None), "ctr_mt3d_interpolate")
    assert len(engine.mt3d_interpolate(attr)) > 0
    engine.mt3d_run(field, 0.0, flags=E.WANT_KEYS)                     # a new run drops the values
    with pytest.raises(E.EngineError):
        engine.mt3d_interpolate_device_ptr()
    engine.mt2d_run(field[0], [0.0])
    with pytest.raises(E.EngineError):
        engine.mt3d_interpolate(attr)


# ---------------------------------------------------------------------------------------------- 7. full size
def test_full_size_uint16_coordinates(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    q = synthetic.ct_like(n, device="cuda")
    f = torch.clamp(torch.round(q * 4096), 0, 65535).to(torch.int32).to(torch.uint16).contiguous()
    del q
    ax = torch.arange(n, device="cuda", dtype=torch.int16)
    grid = torch.stack([a.to(torch.int16) for a in torch.meshgrid(ax, ax, ax, indexing="ij")], -1).contiguous()
    torch.cuda.synchronize()
    c = engine.mt3d_run(f.data_ptr(), 2048.5, flags=E.WANT_KEYS | E.WANT_NORMALS, shape=(n, n, n), dtype=np.uint16)
    assert c.n_verts > 1000000
    verts = engine.mt3d_fetch()["verts"]
    v = engine.mt3d_interpolate(grid.data_ptr(), shape=(n, n, n, 3), dtype=np.int16)
    assert np.array_equal(v, verts)
    del grid, f
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- 8. façade
@pytest.mark.parametrize("post", [True, False])
def test_facade_grid3d(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_values
    g = np.load(os.path.join(GOLDEN, "mt3d_wave11.npz"))
    field, value = g["field"], float(g["value"])
    N = tuple(s - 1 for s in field.shape)
    attr = _random_attr(np.random.default_rng(8), field.shape + (3,), np.float32)
    fn = lambda i, j, k: i * 0.5 + j * j - k

    def make(vf):
        m = tetrahedral.Grid3DContour(*N, field, value, None)
        m.post_process = post
        if vf is not None:
            m.vertex_fields = vf
        return m

    plain = make(None)
    p0, t0 = plain.get_points_and_triangles()
    assert plain.vertex_values is None
    m = make([attr, fn])
    p1, t1 = m.get_points_and_triangles()
    assert np.array_equal(p0, p1) and np.array_equal(t0, t1)
    out = engine.mt3d_fetch()
    assert isinstance(m.vertex_values, list) and len(m.vertex_values) == 2
    assert np.array_equal(m.vertex_values[0], mt3d_values.vertex_values(field, value, out["keys"], out["lowmin"], attr))
    fs = np.fromfunction(fn, field.shape)
    assert np.array_equal(m.vertex_values[1], mt3d_values.vertex_values(field, value, out["keys"], out["lowmin"], fs))
    one = make(attr)
    one.get_points_and_triangles()
    assert np.array_equal(one.vertex_values, m.vertex_values[0])


@pytest.mark.parametrize("post", [True, False])
def test_facade_triangulated_isosurfaces(engine, post):
    from contourist_b200 import grid_field, tetrahedral
    from oracle import mt3d_values
    f = lambda x, y, z: x * x + y * y + z * z
    temp = lambda x, y, z: np.sin(3 * x) + y * z

    def make(vf):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.125, 0.125, 0.125), f, 0.5, [])
        t.post_process = post
        if vf is not None:
            t.vertex_fields = vf
        t.search_for_endpoints()
        return t

    plain = make(None)
    p0, t0 = plain.get_points_and_triangles()
    t = make(temp)
    p1, t1 = t.get_points_and_triangles()
    assert np.array_equal(p0, p1) and np.array_equal(t0, t1)
    out = engine.mt3d_fetch()
    samples = t.grid.samples(1)
    ts = grid_field.FunctionGrid(t.grid.mins, t.grid.maxes, t.grid.delta, temp).samples(1)
    assert t.vertex_values.shape == (len(p1),)
    assert np.array_equal(t.vertex_values, mt3d_values.vertex_values(samples, 0.5, out["keys"], out["lowmin"], ts))
