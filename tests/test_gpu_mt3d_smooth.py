"""GPU: Taubin smoothing of the 3D mesh on the device (ctr_mt3d_smooth, Engine.mt3d_smooth, the façades'
smooth_iterations), against oracle/mt3d_smooth.py applied to the engine's pre-smoothing fetch.  Positions and counts are
compared bit for bit; normals (summed with atomics) within the tolerances of check_normals."""
import ctypes
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN
from test_gpu_mt3d_components import check_oracle
from test_gpu_mt3d_keep import blob_field

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))
PARAMS = [(0, 0.5, -0.53), (1, 0.5, -0.53), (10, 0.5, -0.53), (4, 0.33, 0.0), (3, 1.0, -1.0)]


def _E():
    from contourist_b200 import engine as E
    return E


def _flags(geom64, normals=True):
    E = _E()
    return E.WANT_KEYS | (E.WANT_NORMALS if normals else 0) | (E.GEOM_F64 if geom64 else 0)


def check_normals(got, want, verts, tris, geom64):
    """fp64: angle below 1e-9 rad; fp32: components within 2e-6; vertices whose face normals cancel to below 1e-6 of
    the sum of their lengths are skipped (their direction is decided by rounding), vertices on no triangle compared
    exactly (they keep the old normal)"""
    from oracle import mt3d_smooth
    mag, parts = mt3d_smooth.face_normal_sums(verts, tris)
    none = parts == 0
    assert np.array_equal(got[none], want[none])
    ok = ~none & (mag >= 1e-6 * parts)
    g, w = got[ok].astype(np.float64), want[ok].astype(np.float64)
    if geom64:
        ang = np.arctan2(np.linalg.norm(np.cross(g, w), axis=1), (g * w).sum(axis=1))
        assert ang.max(initial=0) < 1e-9
    else:
        assert np.abs(g - w).max(initial=0) <= 2e-6


def check_smooth(engine, it, lam, mu, geom64):
    """Smooth the current device mesh and compare everything with the definition applied to the fetch before it;
    returns (pre, out)."""
    from oracle import mt3d_smooth
    pre = engine.mt3d_fetch()
    ptrs = engine.mt3d_device_ptrs()
    c = engine.mt3d_smooth(it, lam, mu)
    out = engine.mt3d_fetch()
    want, cnt = mt3d_smooth.smooth(pre["verts"], pre["tris"], it, lam, mu)
    assert (c.n_edges, c.n_fixed_verts) == (cnt["n_edges"], cnt["n_fixed_verts"])
    assert out["verts"].dtype == want.dtype and out["verts"].tobytes() == want.tobytes()
    for name in ("tris", "keys", "lowmin", "cells", "codes"):
        if pre[name] is not None:
            assert np.array_equal(out[name], pre[name]), name
    assert engine.mt3d_device_ptrs() == ptrs
    if pre["normals"] is not None:
        if it == 0:
            assert np.array_equal(out["normals"], pre["normals"])
        else:
            check_normals(out["normals"], mt3d_smooth.normals(want, pre["tris"], pre["normals"]), want, pre["tris"],
                          geom64)
    return pre, out


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_parity_goldens(engine, path, geom64):
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    for it, lam, mu in PARAMS:
        engine.mt3d_run(field, value, flags=_flags(geom64))
        check_smooth(engine, it, lam, mu, geom64)


@pytest.mark.parametrize("geom64", [True, False])
def test_parity_random_fields(engine, geom64):
    rng = np.random.default_rng(21)
    fields = [(rng.standard_normal((17, 20, 23)), 0.0),              # raw noise: many small pieces, box cuts
              (blob_field(40, 2), 0.15),
              ((blob_field(36, 9) > 0.1).astype(np.uint8), 0.5)]       # a mask: the staircase
    for field, value in fields:
        for it, lam, mu in PARAMS[1:4]:
            engine.mt3d_run(field, value, flags=_flags(geom64))
            check_smooth(engine, it, lam, mu, geom64)


# ---------------------------------------------------------------------------------------------- 2. after other passes
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "seeded3d_*.npz"))), ids=lambda p: os.path.basename(p))
def test_after_seeded_selection(engine, path):
    from contourist_b200 import tetrahedral
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    engine.mt3d_run(field, value, flags=_flags(True))
    seeds = g["seeds"]
    start = tetrahedral.initial_voxels(field, value, seeds) if len(seeds) else np.zeros((0, 3), np.int32)
    engine.mt3d_select_seeded(start)
    check_smooth(engine, 5, 0.5, -0.53, True)


@pytest.mark.parametrize("orient", [True, False])
@pytest.mark.parametrize("geom64", [True, False])
def test_after_clean(engine, orient, geom64):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    engine.mt3d_clean(np.array(field.shape) - 1, origin=(-1.0, -1.0, -1.0), delta=(1 / 32,) * 3, orient=orient)
    check_smooth(engine, 6, 0.5, -0.53, geom64)


@pytest.mark.parametrize("geom64", [True, False])
def test_after_orientation_filter_and_integer_runs(engine, geom64):
    field = blob_field(32, 5)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    engine.mt3d_orient_reference()
    pre, out = check_smooth(engine, 4, 0.5, -0.53, geom64)
    # the sign rule: the new normals never point against the gradient normals, whatever the winding
    assert ((out["normals"].astype(np.float64) * pre["normals"]).sum(axis=1) >= 0).all()
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    _, tab = engine.mt3d_components()
    engine.mt3d_keep_components(tab["n_tris"] >= np.median(tab["n_tris"]))
    check_smooth(engine, 4, 0.5, -0.53, geom64)
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    f16 = (g["field"] - 3).astype(np.int16)
    engine.mt3d_run(f16, float(g["value"]) - 3, flags=_flags(geom64))
    check_smooth(engine, 3, 0.5, -0.53, geom64)
    mask = (blob_field(30, 11) > 0.05).astype(np.uint8)
    engine.mt3d_run(mask, 0.5, flags=_flags(geom64))
    check_smooth(engine, 10, 0.5, -0.53, geom64)


def _device_snapshot(ptr, n, dtype):
    import torch

    class Dev(object):
        __cuda_array_interface__ = dict(shape=(n,), typestr=np.dtype(dtype).str, data=(ptr, False), version=3)
    return torch.as_tensor(Dev(), device="cuda").cpu().numpy().copy()


def test_nothing_written_to_normals_without_want_normals(engine):
    field = blob_field(24, 12)
    engine.mt3d_run(field, 0.1, flags=_flags(False))
    nptr = engine.mt3d_device_ptrs()[1]
    engine.mt3d_run(field, 0.1, flags=_flags(False, normals=False))
    assert engine.mt3d_device_ptrs()[1] is None
    n = len(engine.mt3d_fetch()["verts"]) * 3
    before = _device_snapshot(nptr, n, np.float32)
    check_smooth(engine, 5, 0.5, -0.53, False)
    assert np.array_equal(_device_snapshot(nptr, n, np.float32), before)


# ---------------------------------------------------------------------------------------------- 3. invariants
@pytest.mark.parametrize("geom64", [True, False])
def test_invariants_and_repeated_calls(engine, geom64):
    import torch
    from oracle import mt3d_smooth
    E = _E()
    field = blob_field(32, 13)
    pub = torch.zeros(2, dtype=torch.int64, device="cuda")
    engine.mt3d_publish_counts(pub.data_ptr())
    try:
        c = engine.mt3d_run(field, 0.1, flags=_flags(geom64) | E.WANT_CODES)
        torch.cuda.synchronize()
        published = pub.cpu().tolist()
        assert published == [c.n_verts, c.n_tris]
        pre, out = check_smooth(engine, 3, 0.5, -0.53, geom64)       # triangles, keys, lowmin, codes, pointers
        torch.cuda.synchronize()
        assert pub.cpu().tolist() == published
        _, _, fixed, _ = mt3d_smooth.neighbours(len(pre["verts"]), pre["tris"])
        assert fixed.sum() > 0 and np.array_equal(out["verts"][fixed], pre["verts"][fixed])
        assert (out["verts"][~fixed] != pre["verts"][~fixed]).any(axis=1).mean() > 0.5
        # a second call smooths the smoothed mesh; in fp64, 3 then 4 iterations equal 7
        engine.mt3d_smooth(4, 0.5, -0.53)
        two = engine.mt3d_fetch()["verts"]
        assert two.tobytes() == mt3d_smooth.smooth(out["verts"], pre["tris"], 4, 0.5, -0.53)[0].tobytes()
        if geom64:
            assert two.tobytes() == mt3d_smooth.smooth(pre["verts"], pre["tris"], 7, 0.5, -0.53)[0].tobytes()
    finally:
        engine.mt3d_publish_counts(None)


# ---------------------------------------------------------------------------------------------- 4. state
@pytest.mark.parametrize("geom64", [True, False])
def test_state_after_smoothing(engine, geom64):
    from oracle import mt3d_filter
    E = _E()
    g = np.load(os.path.join(GOLDEN, "mt3d_noise8.npz"))
    field, value = g["field"], float(g["value"])
    vf = np.random.default_rng(3).standard_normal(field.shape + (2,))
    engine.mt3d_run(field, value, flags=_flags(geom64))
    before = engine.mt3d_interpolate(vf)
    engine.mt3d_components()
    engine.mt3d_smooth(5)
    assert np.array_equal(engine.mt3d_interpolate(vf), before)        # the keys did not move
    out = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()                               # measured on the smoothed mesh
    check_oracle(lab, tab, out["verts"], out["tris"])
    keep = np.arange(len(tab)) % 2 == 0
    engine.mt3d_keep_components(keep)                                 # after measuring again: accepted
    t, used, _, _ = mt3d_filter.keep_components(out["tris"], lab, tab, keep)
    got = engine.mt3d_fetch()
    assert np.array_equal(got["tris"], t) and np.array_equal(got["verts"], out["verts"][used])
    # filter without measuring again, selection and clean-up after smoothing: refused
    engine.mt3d_run(field, value, flags=_flags(geom64))
    _, tab = engine.mt3d_components()
    engine.mt3d_smooth(2)
    with pytest.raises(E.EngineError, match="smoothing"):
        engine.mt3d_keep_components(np.ones(len(tab), bool))
    with pytest.raises(E.EngineError):
        engine.mt3d_select_seeded(np.zeros((0, 3), np.int32))
    with pytest.raises(E.EngineError, match="smoothed"):
        engine.mt3d_clean(np.array(field.shape) - 1)
    engine.mt3d_orient_reference()                                    # accepted, as is smoothing again
    check_smooth(engine, 2, 0.5, -0.53, geom64)
    # iterations == 0 writes nothing and changes no state
    engine.mt3d_run(field, value, flags=_flags(geom64))
    _, tab = engine.mt3d_components()
    check_smooth(engine, 0, 0.5, -0.53, geom64)
    engine.mt3d_keep_components(np.ones(len(tab), bool))
    engine.mt3d_clean(np.array(field.shape) - 1)


def test_errors(engine):
    E = _E()
    lib = engine.lib
    cnt = E.SmoothCounts()

    def call(eng, it=3, lam=0.5, mu=-0.53, reserved=0, p=True, out=True):
        sp = E.SmoothParams()
        sp.iterations, sp.reserved, sp.lam, sp.mu = it, reserved, lam, mu
        return eng.lib.ctr_mt3d_smooth(eng.h, ctypes.byref(sp) if p else None, ctypes.byref(cnt) if out else None)

    assert lib.ctr_mt3d_smooth(None, None, None) == -1
    fresh = E.Engine(0)
    try:
        assert call(fresh) == -5                                      # no run
    finally:
        fresh.close()
    field = np.random.default_rng(14).standard_normal((9, 8, 10))
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS)
    pre = engine.mt3d_fetch()
    bad = [dict(p=False), dict(out=False), dict(it=-1), dict(it=1001), dict(lam=0.0), dict(lam=1.5), dict(lam=np.nan),
           dict(mu=0.1), dict(mu=-1.5), dict(mu=np.nan), dict(reserved=1)]
    for kw in bad:
        assert call(engine, **kw) == -1, kw
    with pytest.raises(ValueError):
        engine.mt3d_smooth(3, lam=-0.5)
    # limits are accepted
    assert call(engine, it=0, lam=1.0, mu=-1.0) == 0 and call(engine, it=1, lam=1e-3, mu=-0.0) == 0
    engine.mt3d_run(field, 0.0, flags=E.NO_GEOMETRY)
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, i_lo=0, i_hi=5)                       # a slab
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, vert_id_base=7)
    assert call(engine) == -5
    # ids shifted after the run: detected before anything is written
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS)
    engine._check(lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    assert call(engine) == -5
    # every refusal left the positions and normals as they were
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS)
    for kw in bad[2:]:
        call(engine, **kw)
    after = engine.mt3d_fetch()
    assert np.array_equal(after["verts"], pre["verts"]) and np.array_equal(after["normals"], pre["normals"])
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS)
    engine._check(lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    call(engine)
    after = engine.mt3d_fetch()
    assert np.array_equal(after["verts"], pre["verts"]) and np.array_equal(after["normals"], pre["normals"])
    # a 2D run in between drops the 3D results
    engine.mt3d_run(field, 0.0)
    engine.mt2d_run(field[0], [0.0])
    assert call(engine) == -5
    # empty mesh: a valid no-op
    c = engine.mt3d_run(field + 10.0, 0.0)
    assert c.n_tris == 0
    assert call(engine) == 0 and (cnt.n_edges, cnt.n_fixed_verts) == (0, 0)
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt3d_keep_components([])
    assert call(engine) == 0 and (cnt.n_edges, cnt.n_fixed_verts) == (0, 0)


# ---------------------------------------------------------------------------------------------- 5. full size
def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS, shape=(n, n, n), dtype=np.float32)
    check_smooth(engine, 3, 0.5, -0.53, False)
    del f
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- 6. façades
@pytest.mark.parametrize("post", [True, False])
def test_facade_grid3d(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_smooth
    field = blob_field(24, 6).astype(np.float64)
    n = tuple(s - 1 for s in field.shape)
    vf = np.random.default_rng(6).standard_normal(field.shape + (2,))

    def make(iterations):
        m = tetrahedral.Grid3DContour(*n, field, 0.1, None)
        m.post_process = post
        m.reference_orientation = True
        m.vertex_fields = vf
        m.measure_components = True
        m.keep_components = 3
        m.smooth_iterations = iterations
        m.smooth_mu = -0.6
        return m

    plain = make(0)
    p0, t0 = plain.get_points_and_triangles()
    m = make(8)
    p1, t1 = m.get_points_and_triangles()
    assert np.array_equal(t1, t0) and p1.tobytes() == mt3d_smooth.smooth(p0, t0, 8, 0.5, -0.6)[0].tobytes()
    assert np.array_equal(m.vertex_values, plain.vertex_values)
    assert len(m.component_table) == 3
    check_oracle(m.triangle_components, m.component_table, p1, t1)


@pytest.mark.parametrize("post", [True, False])
def test_facade_triangulated_isosurfaces(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_smooth
    f = lambda x, y, z: np.minimum((x - 0.4) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + z * z + 0.05)

    def make(iterations):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.09, [])
        t.post_process = post
        t.geometry_dtype = np.float32
        t.measure_components = True
        t.keep_components = 1
        t.vertex_fields = lambda x, y, z: x * y
        t.smooth_iterations = iterations
        t.search_for_endpoints()
        return t

    plain = make(0)
    p0, t0 = plain.get_points_and_triangles()
    t = make(5)
    p1, t1 = t.get_points_and_triangles()
    assert p1.dtype == np.float32 and np.array_equal(t1, t0)
    assert p1.tobytes() == mt3d_smooth.smooth(p0, t0, 5, 0.5, -0.53)[0].tobytes()
    assert np.array_equal(t.vertex_values, plain.vertex_values) and len(t.component_table) == 1
    check_oracle(t.triangle_components, t.component_table, p1, t1)
