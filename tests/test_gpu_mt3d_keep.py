"""GPU: keeping or dropping connected components of the 3D mesh on the device (ctr_mt3d_keep_components,
Engine.mt3d_keep_components, the façade's keep_components), against oracle/mt3d_filter.py:keep_components applied to the
engine's pre-filter fetch.  Data movement is exact: every comparison is bit for bit unless it says otherwise."""
import ctypes
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, c1_golden
from test_gpu_mt3d_components import INT_FIELDS, check_oracle


def same_rows(tab, want):
    """integer fields and box bit for bit; area / volume (sums of another ctr_mt3d_components call, whose order may
    differ) within the tolerances of check_oracle"""
    assert len(tab) == len(want)
    for f in INT_FIELDS + ("lo", "hi"):
        assert np.array_equal(tab[f], want[f]), f
    assert (np.abs(tab["area"] - want["area"]) <= 1e-11 * want["area"]).all()
    side = (want["hi"] - want["lo"]).max(axis=1)
    assert (np.abs(tab["volume"] - want["volume"]) <= 2e-11 * want["area"] * side).all()

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))


def _E():
    from contourist_b200 import engine as E
    return E


def _flags(geom64):
    E = _E()
    return E.WANT_KEYS | E.WANT_NORMALS | (E.GEOM_F64 if geom64 else 0)


def _values_field(shape, ncomp=4):
    rng = np.random.default_rng(int(np.prod(shape)) % 1000)
    return rng.standard_normal(tuple(shape) + (ncomp,))


def _fetch_values(engine, n, ncomp, geom64):
    out = np.empty((n, ncomp), np.float64 if geom64 else np.float32)
    engine._check(engine.lib.ctr_mt3d_interpolate_fetch(engine.h, out.ctypes.data_as(ctypes.c_void_p)), "fetch")
    return out


def _masks(tab, rng):
    C = len(tab)
    largest = np.zeros(C, bool)
    if C:
        largest[np.argsort(-tab["n_tris"], kind="stable")[0]] = True
    return dict(random=rng.random(C) < 0.5, largest=largest, all=np.ones(C, bool), none=np.zeros(C, bool))


def check_keep(engine, keep, geom64, vfield=None):
    """Measure, filter by `keep` (a function of the table) and compare everything with the definition applied to the
    pre-filter fetch; returns (pre, out, oracle result)."""
    from oracle import mt3d_filter
    pre = engine.mt3d_fetch()
    vals = engine.mt3d_interpolate(vfield) if vfield is not None else None
    lab, tab = engine.mt3d_components()
    mask = np.asarray(keep(tab))
    bmask = mask if mask.dtype == bool else np.isin(np.arange(len(tab)), mask)     # a mask or component indices
    ptrs = engine.mt3d_device_ptrs()
    vptr = engine.mt3d_interpolate_device_ptr() if vfield is not None else None
    nv, nt = engine.mt3d_keep_components(mask)
    out = engine.mt3d_fetch()
    t, used, lab2, tab2 = mt3d_filter.keep_components(pre["tris"], lab, tab, bmask)
    assert (nv, nt) == (len(used), len(t))
    assert np.array_equal(out["tris"], t)
    for name in ("verts", "normals", "keys", "lowmin"):
        if pre[name] is not None:
            assert np.array_equal(out[name], pre[name][used]), name
    lab_f, tab_f = engine.mt3d_components_fetch()
    assert np.array_equal(lab_f, lab2) and tab_f.tobytes() == tab2.tobytes()
    assert engine.mt3d_device_ptrs() == ptrs                          # written back into the same buffers
    if vfield is not None:
        assert engine.mt3d_interpolate_device_ptr() == vptr
        got = _fetch_values(engine, nv, vals.shape[1], geom64)
        assert np.array_equal(got, vals[used])
    return pre, out, (t, used, lab2, tab2)


# ---------------------------------------------------------------------------------------------- 1. mesh parity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_parity_goldens(engine, path, geom64):
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    vf = _values_field(field.shape, 4 if geom64 else 3)
    rng = np.random.default_rng(7)
    engine.mt3d_run(field, value, flags=_flags(geom64))
    _, tab = engine.mt3d_components()
    for name, mask in _masks(tab, rng).items():
        engine.mt3d_run(field, value, flags=_flags(geom64))
        check_keep(engine, lambda t: mask, geom64, vf)


def blob_field(n, seed):
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    return gaussian_filter(rng.standard_normal((n, n + 3, n + 35)), 1.2, mode="wrap").astype(np.float32)


@pytest.mark.parametrize("geom64", [True, False])
def test_parity_many_components(engine, geom64):
    field = blob_field(48, 3)
    value = 0.2
    engine.mt3d_run(field, value, flags=_flags(geom64))
    _, tab = engine.mt3d_components()
    assert len(tab) >= 200 and (tab["n_boundary_edges"] > 0).sum() >= 20     # many, some cut by the box
    rng = np.random.default_rng(8)
    for name, mask in _masks(tab, rng).items():
        engine.mt3d_run(field, value, flags=_flags(geom64))
        check_keep(engine, lambda t: mask, geom64, _values_field(field.shape, 2))
    engine.mt3d_run(field, value, flags=_flags(geom64))                        # indices instead of a mask
    check_keep(engine, lambda t: np.flatnonzero(t["n_verts"] - t["n_edges"] + t["n_tris"] == 2), geom64)


# ---------------------------------------------------------------------------------------------- 2. components after
@pytest.mark.parametrize("geom64", [True, False])
def test_components_after_the_filter(engine, geom64):
    from oracle import mt3d_filter
    field = blob_field(40, 4)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    rng = np.random.default_rng(9)
    _, out, (t, used, lab2, tab2) = check_keep(engine, lambda tab: rng.random(len(tab)) < 0.6, geom64)
    lab3, tab3 = engine.mt3d_components()                             # measured again on the filtered mesh
    check_oracle(lab3, tab3, out["verts"], out["tris"])
    assert np.array_equal(lab3, lab2)
    same_rows(tab3, tab2)
    # twice equals once by the composed mask
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    pre = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    k1 = np.random.default_rng(10).random(len(tab)) < 0.6
    engine.mt3d_keep_components(k1)
    k2 = np.random.default_rng(11).random(int(k1.sum())) < 0.5
    engine.mt3d_keep_components(k2)
    both = k1.copy()
    both[np.flatnonzero(k1)[~k2]] = False
    t, used, lab4, tab4 = mt3d_filter.keep_components(pre["tris"], lab, tab, both)
    out = engine.mt3d_fetch()
    assert np.array_equal(out["tris"], t) and np.array_equal(out["verts"], pre["verts"][used])
    lab_f, tab_f = engine.mt3d_components_fetch()
    assert np.array_equal(lab_f, lab4) and tab_f.tobytes() == tab4.tobytes()


# ---------------------------------------------------------------------------------------------- 3. values
@pytest.mark.parametrize("geom64", [True, False])
def test_values_after_the_filter(engine, geom64):
    g = np.load(os.path.join(GOLDEN, "mt3d_noise8.npz"))
    field, value = g["field"], float(g["value"])
    vf = _values_field(field.shape, 4)
    engine.mt3d_run(field, value, flags=_flags(geom64))
    pre_vals = engine.mt3d_interpolate(vf)
    _, _, (t, used, _, _) = check_keep(engine, lambda tab: np.arange(len(tab)) % 3 != 1, geom64, vf)
    compacted = _fetch_values(engine, len(used), 4, geom64)
    fresh = engine.mt3d_interpolate(vf)
    assert np.array_equal(fresh, compacted) and np.array_equal(fresh, pre_vals[used])
    # values made before a clean-up are not of the current mesh: left as they were
    engine.mt3d_run(field, value, flags=_flags(geom64))
    stale = engine.mt3d_interpolate(vf[..., :1])
    engine.mt3d_clean(np.array(field.shape) - 1)
    engine.mt3d_components()
    engine.mt3d_keep_components(np.ones(len(engine.mt3d_components_fetch()[1]), bool))
    assert np.array_equal(_fetch_values(engine, len(stale), 1, geom64), stale)


# ---------------------------------------------------------------------------------------------- 4. after other passes
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "seeded3d_*.npz"))), ids=lambda p: os.path.basename(p))
def test_after_seeded_selection(engine, path):
    from contourist_b200 import tetrahedral
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    engine.mt3d_run(field, value, flags=_flags(True))
    seeds = g["seeds"]
    start = tetrahedral.initial_voxels(field, value, seeds) if len(seeds) else np.zeros((0, 3), np.int32)
    engine.mt3d_select_seeded(start)
    check_keep(engine, lambda tab: np.arange(len(tab)) % 2 == 0, True, _values_field(field.shape, 1))


@pytest.mark.parametrize("orient", [True, False])
@pytest.mark.parametrize("geom64", [True, False])
def test_after_clean(engine, orient, geom64):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    engine.mt3d_clean(np.array(field.shape) - 1, origin=(-1.0, -1.0, -1.0), delta=(1 / 32,) * 3, orient=orient)
    check_keep(engine, lambda tab: tab["n_tris"] >= np.median(tab["n_tris"]), geom64, _values_field(field.shape, 2))
    g = c1_golden()                                                  # one closed sphere: keep it
    engine.mt3d_run(g["field"], 0.5, flags=_flags(geom64))
    engine.mt3d_clean(np.array(g["field"].shape) - 1, origin=(-1.0, -1.0, -1.0), delta=(1 / 32,) * 3, orient=orient)
    check_keep(engine, lambda tab: tab["n_tris"] == tab["n_tris"].max(), geom64)


@pytest.mark.parametrize("geom64", [True, False])
def test_after_orientation_and_int16(engine, geom64):
    field = blob_field(32, 5)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    lab0, tab0 = engine.mt3d_components()
    engine.mt3d_orient_reference()                                   # only swaps corners: the labels stay valid
    ptrs = engine.mt3d_device_ptrs()
    keep = tab0["n_boundary_edges"] == 0
    engine.mt3d_keep_components(keep)
    assert engine.mt3d_device_ptrs() == ptrs
    lab_f, tab_f = engine.mt3d_components_fetch()
    assert np.array_equal(lab_f, np.cumsum(keep)[lab0[keep[lab0]]] - 1) and len(tab_f) == keep.sum()
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    engine.mt3d_orient_reference()
    check_keep(engine, lambda tab: tab["n_boundary_edges"] == 0, geom64)
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    f16 = (g["field"] - 3).astype(np.int16)
    engine.mt3d_run(f16, float(g["value"]) - 3, flags=_flags(geom64))
    check_keep(engine, lambda tab: np.arange(len(tab)) % 2 == 1, geom64, _values_field(f16.shape, 3))


# ---------------------------------------------------------------------------------------------- 5. errors
def test_errors(engine):
    E = _E()
    lib = engine.lib
    nv, nt = ctypes.c_int64(), ctypes.c_int64()

    def keep(eng, mask, n=None):
        mask = np.ascontiguousarray(mask, np.uint8)
        return eng.lib.ctr_mt3d_keep_components(eng.h, mask.ctypes.data_as(ctypes.c_void_p) if len(mask) else None,
                                                len(mask) if n is None else n, ctypes.byref(nv), ctypes.byref(nt))

    fresh = E.Engine(0)
    try:
        assert keep(fresh, []) == -5                                 # no run
    finally:
        fresh.close()
    field = np.random.default_rng(14).standard_normal((9, 8, 10))
    engine.mt3d_run(field, 0.0, flags=E.NO_GEOMETRY)
    assert keep(engine, []) == -5
    engine.mt3d_run(field, 0.0)
    assert keep(engine, []) == -5                                    # no components since the run
    _, tab = engine.mt3d_components()
    C = len(tab)
    assert C > 2
    assert keep(engine, np.ones(C - 1)) == -1                        # n_keep != C
    assert keep(engine, np.ones(C + 1), n=C + 1) == -1
    assert lib.ctr_mt3d_keep_components(engine.h, None, C, None, None) == -1     # keep == NULL with C > 0
    with pytest.raises(ValueError):
        engine.mt3d_keep_components(np.ones(C + 1, bool))
    with pytest.raises(ValueError):
        engine.mt3d_keep_components([C])
    # stale labels: after a selection, a clean-up, offset_ids; not after the orientation
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt3d_select_seeded(np.zeros((0, 3), np.int32))
    assert keep(engine, np.ones(C)) == -5
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt3d_clean(np.array(field.shape) - 1)
    assert keep(engine, np.ones(C)) == -5
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine._check(lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    assert keep(engine, np.ones(C)) == -5
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt3d_orient_reference()
    assert keep(engine, np.ones(C)) == 0
    # a selection after a filter; clean-up, orientation, components and interpolation are accepted
    with pytest.raises(E.EngineError):
        engine.mt3d_select_seeded(np.zeros((0, 3), np.int32))
    engine.mt3d_run(field, 0.0, flags=E.WANT_KEYS)
    engine.mt3d_components()
    engine.mt3d_keep_components([0, 2])
    engine.mt3d_orient_reference()
    engine.mt3d_clean(np.array(field.shape) - 1, orient=True)
    engine.mt3d_interpolate(field)
    engine.mt3d_components()
    # a 2D run in between drops the 3D results
    engine.mt2d_run(field[0], [0.0])
    assert keep(engine, np.ones(C)) == -5
    # empty mesh: a valid no-op; keeping nothing leaves an empty mesh
    c = engine.mt3d_run(field + 10.0, 0.0)
    assert c.n_tris == 0
    engine.mt3d_components()
    assert engine.mt3d_keep_components(np.zeros(0, bool)) == (0, 0)
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    assert engine.mt3d_keep_components([]) == (0, 0)
    out = engine.mt3d_fetch()
    assert out["verts"].shape == (0, 3) and out["tris"].shape == (0, 3)
    lab, tab = engine.mt3d_components_fetch()
    assert len(lab) == 0 and len(tab) == 0
    lab, tab = engine.mt3d_components()
    assert len(lab) == 0 and len(tab) == 0


# ---------------------------------------------------------------------------------------------- 6. full size
def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    from oracle import mt3d_filter
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS, shape=(n, n, n), dtype=np.float32)
    pre = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    big = int(np.argsort(-tab["n_tris"], kind="stable")[0])
    nv, nt = engine.mt3d_keep_components([big])
    assert nt == tab["n_tris"][big]
    t, used, lab2, tab2 = mt3d_filter.keep_components(pre["tris"], lab, tab, np.arange(len(tab)) == big)
    out = engine.mt3d_fetch()
    assert np.array_equal(out["tris"], t) and np.array_equal(out["verts"], pre["verts"][used])
    assert np.array_equal(out["normals"], pre["normals"][used])
    lab_f, tab_f = engine.mt3d_components_fetch()
    assert np.array_equal(lab_f, lab2) and tab_f.tobytes() == tab2.tobytes()
    del f
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- 7. façades
@pytest.mark.parametrize("post", [True, False])
def test_facade_grid3d(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_filter
    field = blob_field(24, 6).astype(np.float64)
    n = tuple(s - 1 for s in field.shape)
    vf = _values_field(field.shape, 2)

    def make(keep):
        m = tetrahedral.Grid3DContour(*n, field, 0.1, None)
        m.post_process = post
        m.reference_orientation = True
        m.vertex_fields = vf
        m.measure_components = True
        m.keep_components = keep
        return m

    full = make(None)
    p0, t0 = full.get_points_and_triangles()
    rule = lambda tab: tab["n_boundary_edges"] == 0
    m = make(rule)
    p1, t1 = m.get_points_and_triangles()
    tt, used, lab2, tab2 = mt3d_filter.keep_components(t0, full.triangle_components, full.component_table,
                                                       rule(full.component_table))
    assert np.array_equal(t1, tt) and np.array_equal(p1, p0[used])
    assert np.array_equal(m.vertex_values, full.vertex_values[used])
    assert np.array_equal(m.triangle_components, lab2)
    same_rows(m.component_table, tab2)
    check_oracle(m.triangle_components, m.component_table, p1, t1)
    m3 = make(3)
    p3, t3 = m3.get_points_and_triangles()
    assert len(m3.component_table) == 3
    assert sorted(m3.component_table["n_tris"]) == sorted(np.sort(full.component_table["n_tris"])[-3:])


@pytest.mark.parametrize("post", [True, False])
def test_facade_triangulated_isosurfaces(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_filter
    f = lambda x, y, z: np.minimum((x - 0.4) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + z * z + 0.05)

    def make(keep):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.09, [])
        t.post_process = post
        t.measure_components = True
        if keep is not None:
            t.keep_components = keep
        t.search_for_endpoints()
        return t

    full = make(None)
    p0, t0 = full.get_points_and_triangles()
    assert len(full.component_table) == 2
    t = make(1)
    p1, t1 = t.get_points_and_triangles()
    big = int(np.argmax(full.component_table["n_tris"]))
    assert len(t.component_table) == 1 and len(t1) == full.component_table["n_tris"][big]
    tt, used, lab2, tab2 = mt3d_filter.keep_components(t0, full.triangle_components, full.component_table,
                                                       np.arange(2) == big)
    assert np.array_equal(t1, tt) and np.array_equal(p1, p0[used]) and np.array_equal(t.triangle_components, lab2)
    same_rows(t.component_table, tab2)
    check_oracle(t.triangle_components, t.component_table, p1, t1)
