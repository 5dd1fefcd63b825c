"""GPU: plane sections of the device mesh (ctr_mt3d_section, Engine.mt3d_section, the façades' sections option), against
oracle/mt3d_section.py applied to the engine's own fetch.  Segments, polyline membership, starts, flags, points and
junction planes are compared exactly; lengths and areas within rtol 1e-12."""
import ctypes

import numpy as np
import pytest

from test_gpu_mt3d_keep import blob_field

pytestmark = pytest.mark.gpu

ERR_BAD_ARG, ERR_STATE = -1, -5                                 # CTR_ERR_BAD_ARG, CTR_ERR_STATE


def _E():
    from contourist_b200 import engine as E
    return E


def _flags(geom64):
    E = _E()
    return E.WANT_KEYS | E.WANT_NORMALS | (E.GEOM_F64 if geom64 else 0)


def check_section(engine, normal, offsets):
    "section the current device mesh and compare with the definition on its fetch; returns the oracle's result"
    from oracle import mt3d_section
    mesh = engine.mt3d_fetch()
    seg, polys = engine.mt3d_section(normal, offsets)
    want = mt3d_section.section(mesh["verts"], mesh["tris"], normal, offsets, mesh["verts"].dtype)
    assert np.array_equal(seg["plane"], want["plane"])
    assert np.array_equal(seg["edges"], want["edges"])
    assert seg["points"].dtype == want["points"].dtype and np.array_equal(seg["points"], want["points"])
    assert len(polys) == len(want["polylines"])
    for got, ref in zip(polys, want["polylines"]):
        if ref is None:
            assert got is None
            continue
        assert got is not None and len(got) == len(ref)
        for (c, k, p, ln, ar), (rc, rk, rp, rln, rar) in zip(got, ref):
            assert (c, k) == (rc, rk) and np.array_equal(p, rp)
            np.testing.assert_allclose(ln, rln, rtol=1e-12)
            np.testing.assert_allclose(ar, rar, rtol=1e-12, atol=1e-12 * rln * rln)
    return want


def planes(mesh, normal, k):
    "k strictly increasing offsets spread over the mesh's extent along normal"
    s = mesh["verts"].astype(np.float64) @ np.asarray(normal, np.float64)
    return np.linspace(s.min(), s.max(), k + 2)[1:-1] + 1e-3


MESHES = ["raw", "smoothed", "decimated", "capped", "kept", "oriented"]


def prepare(engine, geom64, kind):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.2, flags=_flags(geom64))
    if kind == "smoothed":
        engine.mt3d_smooth(5)
    elif kind == "decimated":
        engine.mt3d_decimate(2.5)
        _, tab = engine.mt3d_components()
        assert tab["n_nonmanifold_edges"].sum() > 0            # the junction path runs
    elif kind == "capped":
        engine.mt3d_cap("low")
    elif kind == "kept":
        _, tab = engine.mt3d_components()
        engine.mt3d_keep_components(np.argsort(-tab["n_tris"], kind="stable")[:3])
    elif kind == "oriented":
        engine.mt3d_orient_reference()


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("kind", MESHES)
@pytest.mark.parametrize("normal", [(0.0, 0.0, 1.0), (0.3, -0.5, 0.8)])
@pytest.mark.parametrize("k", [1, 64, 300])
def test_parity(engine, geom64, kind, normal, k):
    prepare(engine, geom64, kind)
    want = check_section(engine, normal, planes(engine.mt3d_fetch(), normal, k))
    assert len(want["plane"]) > 0
    if kind == "decimated" and k > 1:
        assert want["junction"].any()


def test_capped_sections_are_closed_and_consistent(engine):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.2, flags=_flags(True))
    engine.mt3d_cap("low")
    mesh = engine.mt3d_fetch()
    _, polys = engine.mt3d_section((1.0, 0.0, 0.0), planes(mesh, (1.0, 0.0, 0.0), 20))
    assert all(p is not None and all(c and k for c, k, _, _, _ in p) for p in polys)


def test_read_only(engine):
    field = blob_field(32, 7)
    E = _E()
    engine.mt3d_run(field, 0.2, flags=_flags(False))
    labels, table = engine.mt3d_components()
    values = engine.mt3d_interpolate(field)
    ptrs = engine.mt3d_device_ptrs()
    before = engine.mt3d_fetch()
    engine.mt3d_section((0.2, 0.3, 0.9), planes(before, (0.2, 0.3, 0.9), 40))
    after = engine.mt3d_fetch()
    for key in ("verts", "normals", "tris", "keys", "lowmin"):
        assert np.array_equal(before[key], after[key])
    l2, t2 = engine.mt3d_components_fetch()
    assert np.array_equal(labels, l2) and table.tobytes() == t2.tobytes()
    v2 = np.empty_like(values)
    engine._check(engine.lib.ctr_mt3d_interpolate_fetch(engine.h, E._ptr(v2)), "ctr_mt3d_interpolate_fetch")
    assert np.array_equal(values, v2)
    assert engine.mt3d_device_ptrs() == ptrs
    engine.mt3d_keep_components(np.array([0]))                # still accepted: the component results are untouched


def _call(engine, normal, offsets, reserved=0, nplanes=None):
    E = _E()
    off = np.ascontiguousarray(np.asarray(offsets, np.float64))
    p = E.SectionParams()
    for a in range(3):
        p.normal[a] = normal[a]
    p.offsets = off.ctypes.data if len(off) else None
    p.nplanes = len(off) if nplanes is None else nplanes
    p.reserved = reserved
    c = E.SectionCounts()
    return engine.lib.ctr_mt3d_section(engine.h, ctypes.byref(p), ctypes.byref(c)), c


def test_errors(engine):
    from contourist_b200 import engine as E
    fresh = E.Engine(0)
    assert _call(fresh, (0.0, 0.0, 1.0), [1.0])[0] == ERR_STATE
    assert fresh.lib.ctr_mt3d_section_segments_fetch(fresh.h, None, None, None) == ERR_STATE
    fresh.close()
    field = blob_field(24, 5)
    engine.mt3d_run(field, 0.2, flags=_flags(False))
    assert engine.lib.ctr_mt3d_section_polylines_fetch(engine.h, *([None] * 8)) == ERR_STATE
    bad = [((0.0, 0.0, 0.0), [1.0], 0, None), ((np.nan, 0.0, 1.0), [1.0], 0, None), ((np.inf, 0.0, 1.0), [1.0], 0, None),
           ((0.0, 0.0, 1.0), [2.0, 1.0], 0, None), ((0.0, 0.0, 1.0), [1.0, 1.0], 0, None),
           ((0.0, 0.0, 1.0), [1.0, np.nan], 0, None), ((0.0, 0.0, 1.0), [1.0, np.inf], 0, None),
           ((0.0, 0.0, 1.0), [1.0], 1, None), ((0.0, 0.0, 1.0), [], 0, 0), ((0.0, 0.0, 1.0), np.arange(65537.0), 0, None)]
    for normal, offsets, reserved, nplanes in bad:
        assert _call(engine, normal, offsets, reserved, nplanes)[0] == ERR_BAD_ARG, (normal, offsets, reserved)
    assert engine.lib.ctr_mt3d_section(engine.h, None, None) == ERR_BAD_ARG
    assert _call(engine, (0.0, 0.0, 1.0), np.arange(65536.0))[0] == 0
    engine.mt3d_run(field, 0.2, flags=_flags(False) | E.NO_GEOMETRY)
    assert _call(engine, (0.0, 0.0, 1.0), [1.0])[0] == ERR_STATE
    engine.mt3d_run(field, 0.2, flags=_flags(False), i_lo=0, i_hi=12)
    assert _call(engine, (0.0, 0.0, 1.0), [1.0])[0] == ERR_STATE
    engine.mt3d_run(field, 0.2, flags=_flags(False))
    assert engine.lib.ctr_mt3d_offset_ids(engine.h, 7) == 0
    assert _call(engine, (0.0, 0.0, 1.0), [5.0])[0] == ERR_STATE


def test_empty_mesh(engine):
    field = blob_field(24, 5)
    engine.mt3d_run(field, 1e6, flags=_flags(True))
    rc, c = _call(engine, (0.0, 0.0, 1.0), [1.0, 2.0])
    assert rc == 0 and (c.n_segments, c.n_polylines, c.n_points, c.n_junction_planes) == (0, 0, 0, 0)
    seg, polys = engine.mt3d_section((0.0, 0.0, 1.0), [1.0, 2.0])
    assert len(seg["plane"]) == 0 and polys == [[], []]


def test_facade_sections(engine):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_section
    field = blob_field(24, 5).astype(np.float64)
    g = tetrahedral.GridContour3d(np.array(field.shape) - 1, field, 0.2, None, origin=(1.0, 2.0, 3.0), delta=(0.5, 0.5, 0.25))
    g.post_process = False
    g.full_scan = True
    g.sections = ((0.0, 0.0, 1.0), [4.0, 5.0, 6.0])
    points, tris = g.get_points_and_triangles()
    want = mt3d_section.section(points, tris, (0.0, 0.0, 1.0), [4.0, 5.0, 6.0])["polylines"]
    assert len(g.section_polylines) == 3
    for got, ref in zip(g.section_polylines, want):
        assert [np.array_equal(a[2], b[2]) for a, b in zip(got, ref)] == [True] * len(ref) and len(got) == len(ref)
