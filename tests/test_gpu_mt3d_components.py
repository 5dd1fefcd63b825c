"""GPU: connected components of the 3D mesh with per-component size and topology (ctr_mt3d_components,
Engine.mt3d_components, the façade's measure_components), against oracle/mt3d_components.py:components on the engine's
fetched mesh and against analytic surfaces."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, c1_golden

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))
INT_FIELDS = ("n_tris", "n_verts", "n_edges", "n_boundary_edges", "n_nonmanifold_edges", "first_tri")


def _E():
    from contourist_b200 import engine as E
    return E


def _run(engine, field, value, geom64, extra=0, **kw):
    E = _E()
    c = engine.mt3d_run(field, value, flags=(E.GEOM_F64 if geom64 else 0) | extra, **kw)
    return c, engine.mt3d_fetch()


def check_oracle(lab, tab, verts, tris):
    """labels and integer fields equal, box bit for bit, area within 1e-11 relative, volume within
    1e-11 * area * largest box side"""
    from oracle import mt3d_components
    want_lab, want = mt3d_components.components(verts, tris)
    assert lab.dtype == np.int32 and len(lab) == len(tris)
    assert tab.dtype == _E().COMPONENT_DTYPE and len(tab) == len(want)
    assert np.array_equal(lab, want_lab)
    for f in INT_FIELDS:
        assert np.array_equal(tab[f], want[f]), f
    assert np.array_equal(tab["lo"], want["lo"]) and np.array_equal(tab["hi"], want["hi"])
    assert (np.abs(tab["area"] - want["area"]) <= 1e-11 * want["area"]).all()
    side = (want["hi"] - want["lo"]).max(axis=1)
    assert (np.abs(tab["volume"] - want["volume"]) <= 1e-11 * want["area"] * side).all()
    return want


def chi(tab):
    return tab["n_verts"] - tab["n_edges"] + tab["n_tris"]


# ---------------------------------------------------------------------------------------------- 1. oracle parity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_oracle_parity_goldens(engine, path, geom64):
    g = np.load(path)
    _, out = _run(engine, g["field"], float(g["value"]), geom64)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])


@pytest.mark.parametrize("shape", [(6, 5, 32), (5, 7, 64), (4, 6, 129), (17, 9, 33), (40, 41, 43)])
@pytest.mark.parametrize("geom64", [True, False])
def test_oracle_parity_random(engine, shape, geom64):
    rng = np.random.default_rng(shape[2] * 31 + shape[0])
    field = rng.standard_normal(shape).astype(np.float32)
    _, out = _run(engine, field, 0.1, geom64)
    lab, tab = engine.mt3d_components()
    want = check_oracle(lab, tab, out["verts"], out["tris"])
    assert len(want) > 1


@pytest.mark.parametrize("geom64", [True, False])
def test_oracle_parity_int16_plateaus(engine, geom64):
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    _, out = _run(engine, (g["field"] - 3).astype(np.int16), float(g["value"]) - 3, geom64)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])


# ---------------------------------------------------------------------------------------------- 2. analytic surfaces
N = 64


def _grid(n=N):
    x = np.arange(n + 1, dtype=np.float64)
    return np.meshgrid(x, x, x, indexing="ij")


@pytest.mark.parametrize("geom64", [True, False])
def test_sphere_and_torus(engine, geom64):
    X, Y, Z = _grid()
    r = 0.35 * N
    sph = (X - N / 2) ** 2 + (Y - N / 2) ** 2 + (Z - N / 2) ** 2 - r * r
    _, out = _run(engine, sph, 0.0, geom64)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    assert len(tab) == 1 and chi(tab)[0] == 2 and tab["n_boundary_edges"][0] == 0 and tab["n_verts"][0] == len(out["verts"])
    assert abs(tab["area"][0] / (4 * np.pi * r * r) - 1) < 5e-3
    assert tab["volume"][0] > 0 and abs(tab["volume"][0] / (4 / 3 * np.pi * r ** 3) - 1) < 5e-3
    _run(engine, -sph, 0.0, geom64)                                    # the inside above the isovalue
    _, tabn = engine.mt3d_components()
    assert tabn["volume"][0] < 0 and abs(tabn["volume"][0] / tab["volume"][0] + 1) < 1e-6
    R, rr = 0.25 * N, 0.1 * N
    Xc, Yc, Zc = X - N / 2, Y - N / 2, Z - N / 2
    tor = (np.sqrt(Xc * Xc + Yc * Yc) - R) ** 2 + Zc * Zc - rr * rr
    _, out = _run(engine, tor, 0.0, geom64)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    assert len(tab) == 1 and chi(tab)[0] == 0 and tab["n_boundary_edges"][0] == 0
    assert abs(tab["area"][0] / (4 * np.pi ** 2 * R * rr) - 1) < 5e-3
    assert tab["volume"][0] > 0 and abs(tab["volume"][0] / (2 * np.pi ** 2 * R * rr * rr) - 1) < 1.5e-2


def test_two_spheres_and_a_cut_plane(engine):
    X, Y, Z = _grid()
    f = np.minimum((X - 40) ** 2 + (Y - 32) ** 2 + (Z - 32) ** 2 - 14.0 ** 2, (X - 14) ** 2 + (Y - 32) ** 2 + (Z - 32) ** 2 - 8.0 ** 2)
    _, out = _run(engine, f, 0.0, True)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    assert len(tab) == 2 and tab["first_tri"][0] == 0 and tab["first_tri"][1] > 0
    assert (chi(tab) == 2).all() and (tab["volume"] > 0).all()
    assert np.array_equal(np.bincount(lab), tab["n_tris"])
    X, Y, Z = _grid(16)
    _, out = _run(engine, X + 0.5 * Y + 0.25 * Z, 9.3, False)
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    assert len(tab) == 1 and tab["n_boundary_edges"][0] > 0 and chi(tab)[0] == 1


# ---------------------------------------------------------------------------------------------- 3. against orientation
@pytest.mark.parametrize("geom64", [True, False])
def test_against_orientation(engine, geom64):
    rng = np.random.default_rng(11)
    field = rng.standard_normal((30, 31, 35))
    for value in (0.4, -0.4):
        _, out = _run(engine, field, value, geom64)
        lab, tab = engine.mt3d_components()
        nc, _ = engine.mt3d_orient_reference()
        assert nc == len(tab)
        fin = engine.mt3d_fetch()
        lab2, tab2 = engine.mt3d_components()
        check_oracle(lab2, tab2, fin["verts"], fin["tris"])
        assert np.array_equal(lab, lab2)
        for f in INT_FIELDS:
            assert np.array_equal(tab[f], tab2[f])
        closed = tab2["n_boundary_edges"] == 0
        assert closed.any() and (tab2["volume"][closed] >= 0).all()
        tol = 1e-11 * tab["area"] * (tab["hi"] - tab["lo"]).max(axis=1)
        assert (np.abs(np.abs(tab2["volume"]) - np.abs(tab["volume"]))[closed] <= 2 * tol[closed]).all()


# ---------------------------------------------------------------------------------------------- 4. after mesh edits
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "seeded3d_*.npz"))),
                         ids=lambda p: os.path.basename(p))
def test_after_seeded_selection(engine, path):
    from contourist_b200 import tetrahedral
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    _run(engine, field, value, True)
    seeds = g["seeds"]
    start = tetrahedral.initial_voxels(field, value, seeds) if len(seeds) else np.zeros((0, 3), np.int32)
    engine.mt3d_select_seeded(start)
    sel = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, sel["verts"], sel["tris"])


@pytest.mark.parametrize("geom64", [True, False])
def test_after_clean_c1(engine, geom64):
    g = c1_golden()
    field = g["field"]
    _run(engine, field, 0.5, geom64)
    cc = engine.mt3d_clean(np.array(field.shape) - 1, origin=(-1.0, -1.0, -1.0), delta=(1 / 32,) * 3, orient=True)
    fin = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, fin["verts"], fin["tris"])
    assert len(tab) == cc.n_components
    closed = tab["n_boundary_edges"] == 0
    assert (tab["volume"][closed] >= 0).all()
    r = np.sqrt(0.5)
    assert abs(tab["volume"].sum() / (4 / 3 * np.pi * r ** 3) - 1) < 5e-3


# ---------------------------------------------------------------------------------------------- 5. full size
def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    c = engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS, shape=(n, n, n), dtype=np.float32)
    assert c.n_tris > 5000000
    out = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    lab2, tab2 = engine.mt3d_components()                           # repeat calls: integer outputs identical
    assert np.array_equal(lab, lab2)
    for fld in INT_FIELDS + ("lo", "hi"):
        assert np.array_equal(tab[fld], tab2[fld])
    nc, _ = engine.mt3d_orient_reference()
    assert nc == len(tab)
    del f
    torch.cuda.empty_cache()


def test_repeat_calls(engine):
    rng = np.random.default_rng(12)
    _run(engine, rng.standard_normal((20, 21, 70)), 0.0, False)
    first = engine.mt3d_components()
    for _ in range(3):
        lab, tab = engine.mt3d_components()
        assert np.array_equal(lab, first[0])
        for f in INT_FIELDS + ("lo", "hi"):
            assert np.array_equal(tab[f], first[1][f])


# ---------------------------------------------------------------------------------------------- 6. errors
def test_errors(engine):
    E = _E()
    fresh = E.Engine(0)
    try:
        with pytest.raises(E.EngineError):
            fresh.mt3d_components()                                    # no run
        fresh.mt3d_run(np.random.default_rng(13).standard_normal((8, 8, 8)), 0.0)
        assert fresh.lib.ctr_mt3d_components_fetch(fresh.h, None, None) != 0   # fetch before a call
        fresh.mt3d_components()
        assert fresh.lib.ctr_mt3d_components_fetch(fresh.h, None, None) == 0
        fresh.mt3d_run(np.random.default_rng(13).standard_normal((8, 8, 8)), 0.0)
        assert fresh.lib.ctr_mt3d_components_fetch(fresh.h, None, None) != 0   # a new run drops the results
    finally:
        fresh.close()
    field = np.random.default_rng(14).standard_normal((9, 8, 10))
    engine.mt3d_run(field, 0.0, flags=E.NO_GEOMETRY)
    with pytest.raises(E.EngineError):
        engine.mt3d_components()
    engine.mt3d_run(field, 0.0, i_lo=1, i_hi=7, plane_offset=0)     # a slab
    with pytest.raises(E.EngineError):
        engine.mt3d_components()
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    with pytest.raises(E.EngineError):
        engine.mt3d_components()                                       # ids outside [0, n_verts)
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt2d_run(field[0], [0.0])
    with pytest.raises(E.EngineError):
        engine.mt3d_components()
    assert engine.lib.ctr_mt3d_components_fetch(engine.h, None, None) != 0
    c = engine.mt3d_run(field + 10.0, 0.0)                             # empty mesh
    assert c.n_tris == 0
    lab, tab = engine.mt3d_components()
    assert len(lab) == 0 and len(tab) == 0


# ---------------------------------------------------------------------------------------------- 7. façades
@pytest.mark.parametrize("post", [True, False])
def test_facade_grid3d(engine, post):
    from contourist_b200 import tetrahedral
    g = np.load(os.path.join(GOLDEN, "mt3d_wave11.npz"))
    field, value = g["field"], float(g["value"])
    n = tuple(s - 1 for s in field.shape)

    def make(measure):
        m = tetrahedral.Grid3DContour(*n, field, value, None)
        m.post_process = post
        m.reference_orientation = True
        if measure:
            m.measure_components = True
        return m

    plain = make(False)
    p0, t0 = plain.get_points_and_triangles()
    assert plain.triangle_components is None and plain.component_table is None
    m = make(True)
    p1, t1 = m.get_points_and_triangles()
    assert np.array_equal(p0, p1) and np.array_equal(t0, t1)
    assert len(m.triangle_components) == len(t1)
    check_oracle(m.triangle_components, m.component_table, p1, t1)
    closed = m.component_table["n_boundary_edges"] == 0
    assert (m.component_table["volume"][closed] >= 0).all()


@pytest.mark.parametrize("post", [True, False])
def test_facade_triangulated_isosurfaces(engine, post):
    from contourist_b200 import tetrahedral
    f = lambda x, y, z: np.minimum((x - 0.4) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + z * z + 0.05)

    def make(measure):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.09, [])
        t.post_process = post
        if measure:
            t.measure_components = True
        t.search_for_endpoints()
        return t

    p0, t0 = make(False).get_points_and_triangles()
    t = make(True)
    p1, t1 = t.get_points_and_triangles()
    assert np.array_equal(p0, p1) and np.array_equal(t0, t1)
    assert len(t.triangle_components) == len(t1) and len(t.component_table) == 2
    check_oracle(t.triangle_components, t.component_table, p1, t1)
    if post:
        assert (t.component_table["volume"] > 0).all()
