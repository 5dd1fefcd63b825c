"""GPU: quadric vertex-clustering decimation of the 3D mesh on the device (ctr_mt3d_decimate, Engine.mt3d_decimate, the
façades' decimate_cell), against oracle/mt3d_decimate.py applied to the engine's own pre-decimation fetch.  Counts,
triangles, keys and lowmin are compared exactly; positions within 1e-9 of the cell size (plus one fp32 spacing with
fp32 geometry); normals within the tolerances of check_normals."""
import ctypes
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, c1_golden
from test_gpu_mt3d_components import check_oracle
from test_gpu_mt3d_keep import blob_field
from test_gpu_mt3d_smooth import check_normals

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))
CELLS = [(1.0, (0.0, 0.0, 0.0)), (2.0, (0.0, 0.0, 0.0)), ((1.5, 2.5, 3.0), (0.3, -0.7, 0.1)), (4.0, (-0.5, 0.25, 1.0))]


def _E():
    from contourist_b200 import engine as E
    return E


def _flags(geom64, normals=True):
    E = _E()
    return E.WANT_KEYS | (E.WANT_NORMALS if normals else 0) | (E.GEOM_F64 if geom64 else 0)


def check_decimate(engine, cell, origin, geom64):
    """Decimate the current device mesh and compare everything with the definition applied to the fetch before it;
    returns (pre, out, member)."""
    from oracle import mt3d_decimate, mt3d_smooth
    pre = engine.mt3d_fetch()
    ptrs = engine.mt3d_device_ptrs()
    c = engine.mt3d_decimate(cell, origin)
    out = engine.mt3d_fetch()
    want, tris, member, cnt = mt3d_decimate.decimate(pre["verts"], pre["tris"], cell, origin)
    assert dict(n_verts=c.n_verts, n_tris=c.n_tris, n_clusters=c.n_clusters, n_collapsed=c.n_collapsed,
                n_duplicate=c.n_duplicate) == cnt
    assert np.array_equal(out["tris"], tris)
    if pre["keys"] is not None:
        assert np.array_equal(out["keys"], pre["keys"][member]) and np.array_equal(out["lowmin"], pre["lowmin"][member])
    assert out["verts"].dtype == want.dtype and out["verts"].shape == want.shape
    tol = 1e-9 * float(np.max(cell))
    if not geom64:
        tol = tol + np.spacing(np.abs(want)).astype(np.float64)
    assert (np.abs(out["verts"].astype(np.float64) - want.astype(np.float64)) <= tol).all()
    assert engine.mt3d_device_ptrs() == ptrs
    if pre["normals"] is not None:
        got = out["verts"]
        check_normals(out["normals"], mt3d_smooth.normals(got, tris, pre["normals"][member]), got, tris, geom64)
    return pre, out, member


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_parity_goldens(engine, path, geom64):
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    for cell, origin in CELLS:
        engine.mt3d_run(field, value, flags=_flags(geom64))
        check_decimate(engine, cell, origin, geom64)


@pytest.mark.parametrize("geom64", [True, False])
def test_parity_sphere_and_blobs(engine, geom64):
    g = c1_golden()
    fields = [(g["field"], 0.5), (blob_field(40, 2), 0.15), (np.random.default_rng(21).standard_normal((17, 20, 23)), 0.0)]
    for field, value in fields:
        for cell, origin in CELLS[1:]:
            engine.mt3d_run(field, value, flags=_flags(geom64))
            check_decimate(engine, cell, origin, geom64)


# ---------------------------------------------------------------------------------------------- 2. composition
@pytest.mark.parametrize("geom64", [True, False])
def test_after_filter_smoothing_and_clean(engine, geom64):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.1, flags=_flags(geom64))
    engine.mt3d_clean(np.array(field.shape) - 1, origin=(-1.0, -1.0, -1.0), delta=(1 / 32,) * 3, orient=True)
    _, tab = engine.mt3d_components()
    engine.mt3d_keep_components(tab["n_tris"] >= np.median(tab["n_tris"]))
    engine.mt3d_smooth(4)
    check_decimate(engine, 2 / 32, (-1.0, -1.0, -1.0), geom64)
    check_decimate(engine, 3 / 32, (-1.0, -1.0, -1.0), geom64)             # a further decimation is accepted


@pytest.mark.parametrize("geom64", [True, False])
def test_state_after_decimation(engine, geom64):
    E = _E()
    g = np.load(os.path.join(GOLDEN, "mt3d_noise8.npz"))
    field, value = g["field"], float(g["value"])
    vf = np.random.default_rng(3).standard_normal(field.shape + (2,))
    engine.mt3d_run(field, value, flags=_flags(geom64))
    before = engine.mt3d_interpolate(vf)
    _, tab = engine.mt3d_components()
    _, _, member = check_decimate(engine, 2.0, (0.0, 0.0, 0.0), geom64)
    # the filter refuses until the components are measured again
    with pytest.raises(E.EngineError, match="decimation"):
        engine.mt3d_keep_components(np.ones(len(tab), bool))
    out = engine.mt3d_fetch()
    lab, tab = engine.mt3d_components()
    check_oracle(lab, tab, out["verts"], out["tris"])
    engine.mt3d_keep_components(np.arange(len(tab)) % 2 == 0)
    # interpolation gives the member's values; selection and clean-up are refused; orientation and smoothing accepted
    engine.mt3d_run(field, value, flags=_flags(geom64))
    _, _, member = check_decimate(engine, 2.0, (0.5, 0.5, 0.5), geom64)
    assert np.array_equal(engine.mt3d_interpolate(vf), before[member])
    with pytest.raises(E.EngineError):
        engine.mt3d_select_seeded(np.zeros((0, 3), np.int32))
    with pytest.raises(E.EngineError, match="decimated"):
        engine.mt3d_clean(np.array(field.shape) - 1)
    engine.mt3d_orient_reference()
    pre = engine.mt3d_fetch()
    engine.mt3d_smooth(2)
    from oracle import mt3d_smooth
    assert engine.mt3d_fetch()["verts"].tobytes() == mt3d_smooth.smooth(pre["verts"], pre["tris"], 2, 0.5, -0.53)[0].tobytes()


def test_invariants(engine):
    import torch
    E = _E()
    field = blob_field(32, 13)
    pub = torch.zeros(2, dtype=torch.int64, device="cuda")
    engine.mt3d_publish_counts(pub.data_ptr())
    try:
        c = engine.mt3d_run(field, 0.1, flags=_flags(False) | E.WANT_CODES)
        torch.cuda.synchronize()
        published = pub.cpu().tolist()
        pre, out, _ = check_decimate(engine, 2.0, (0.0, 0.0, 0.0), False)
        torch.cuda.synchronize()
        assert pub.cpu().tolist() == published == [c.n_verts, c.n_tris]
        assert np.array_equal(out["cells"], pre["cells"]) and np.array_equal(out["codes"], pre["codes"])
        assert len(out["tris"]) < len(pre["tris"]) / 2
    finally:
        engine.mt3d_publish_counts(None)


def test_int16_run(engine):
    g = np.load(os.path.join(GOLDEN, "mt3d_ints7.npz"))
    f16 = (g["field"] - 3).astype(np.int16)
    for geom64 in (True, False):
        engine.mt3d_run(f16, float(g["value"]) - 3, flags=_flags(geom64))
        check_decimate(engine, 2.0, (0.0, 0.0, 0.0), geom64)
    mask = (blob_field(30, 11) > 0.05).astype(np.uint8)
    engine.mt3d_run(mask, 0.5, flags=_flags(False))
    check_decimate(engine, 3.0, (0.0, 0.0, 0.0), False)


# ---------------------------------------------------------------------------------------------- 3. errors
def test_errors(engine):
    E = _E()
    lib = engine.lib
    cnt = E.DecimateCounts()

    def call(eng, cell=(2.0, 2.0, 2.0), origin=(0.0, 0.0, 0.0), p=True, out=True):
        dp = E.DecimateParams()
        for a in range(3):
            dp.cell[a], dp.origin[a] = cell[a], origin[a]
        return eng.lib.ctr_mt3d_decimate(eng.h, ctypes.byref(dp) if p else None, ctypes.byref(cnt) if out else None)

    assert lib.ctr_mt3d_decimate(None, None, None) == -1
    fresh = E.Engine(0)
    try:
        assert call(fresh) == -5                                      # no run
    finally:
        fresh.close()
    field = np.random.default_rng(14).standard_normal((9, 8, 10))
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS | E.WANT_KEYS)
    pre = engine.mt3d_fetch()
    bad = [dict(p=False), dict(out=False), dict(cell=(0.0, 1.0, 1.0)), dict(cell=(1.0, -1.0, 1.0)),
           dict(cell=(1.0, 1.0, np.nan)), dict(cell=(np.inf, 1.0, 1.0)), dict(origin=(np.nan, 0.0, 0.0)),
           dict(origin=(0.0, -np.inf, 0.0)), dict(origin=(2.0 ** 21, 0.0, 0.0), cell=(1.0, 1.0, 1.0)),
           dict(cell=(1e-7, 1.0, 1.0))]                               # the last two: cell indices out of range
    for kw in bad:
        assert call(engine, **kw) == -1, kw
    engine.mt3d_run(field, 0.0, flags=E.NO_GEOMETRY)
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, i_lo=0, i_hi=5)                       # a slab
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, vert_id_base=7)
    assert call(engine) == -5
    # every refusal above left the mesh as it was
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS | E.WANT_KEYS)
    for kw in bad[2:]:
        call(engine, **kw)
    after = engine.mt3d_fetch()
    for name in ("verts", "normals", "tris", "keys"):
        assert np.array_equal(after[name], pre[name]), name
    # ids shifted after the run: detected before anything is written
    engine._check(lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    assert call(engine) == -5
    after = engine.mt3d_fetch()
    assert np.array_equal(after["verts"], pre["verts"]) and np.array_equal(after["normals"], pre["normals"])
    with pytest.raises(ValueError):
        engine.mt3d_decimate(0.0)
    # empty mesh: a valid no-op
    c = engine.mt3d_run(field + 10.0, 0.0)
    assert c.n_tris == 0
    assert call(engine) == 0 and (cnt.n_verts, cnt.n_tris, cnt.n_clusters) == (0, 0, 0)
    engine.mt3d_run(field, 0.0)
    engine.mt3d_components()
    engine.mt3d_keep_components([])
    assert call(engine) == 0 and (cnt.n_verts, cnt.n_tris) == (0, 0)


# ---------------------------------------------------------------------------------------------- 4. full size, façades
def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS | E.WANT_KEYS, shape=(n, n, n), dtype=np.float32)
    check_decimate(engine, 4.0, (0.0, 0.0, 0.0), False)
    del f
    torch.cuda.empty_cache()


@pytest.mark.parametrize("post", [True, False])
def test_facade_triangulated_isosurfaces(engine, post):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_decimate
    f = lambda x, y, z: np.minimum((x - 0.4) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + z * z + 0.05)

    def make(cell):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.09, [])
        t.post_process = post
        t.measure_components = True
        t.keep_components = 1
        t.vertex_fields = lambda x, y, z: x * y
        t.smooth_iterations = 2
        t.decimate_cell = cell
        t.search_for_endpoints()
        return t

    plain = make(None)
    p0, t0 = plain.get_points_and_triangles()
    t = make(2)
    p1, t1 = t.get_points_and_triangles()
    want, tris, member, _ = mt3d_decimate.decimate(p0, t0, 0.125, (-1.0, -1.0, -1.0))
    assert np.array_equal(t1, tris) and np.abs(p1 - want).max() <= 1e-9
    assert np.array_equal(t.vertex_values, plain.vertex_values[member])
    assert len(t.component_table) >= 1
    check_oracle(t.triangle_components, t.component_table, p1, t1)
