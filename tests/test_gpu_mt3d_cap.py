"""GPU: caps at the faces of the volume on the device (ctr_mt3d_cap, Engine.mt3d_cap, the façades' cap), against
oracle/mt3d_cap.py applied to the engine's own pre-cap fetch.  Counts, triangles, keys, lowmin, the new positions and
the old rows are compared exactly; the new normals within one ulp."""
import ctypes
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN
from test_gpu_mt3d_components import check_oracle
from test_gpu_mt3d_keep import blob_field
from test_oracle_cap_cpu import directed_edges_closed, signed_volume

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))
DTYPES = [np.float32, np.float64, np.uint8, np.int16, np.uint16]


def _E():
    from contourist_b200 import engine as E
    return E


def _flags(geom64, normals=True):
    E = _E()
    return E.WANT_KEYS | (E.WANT_NORMALS if normals else 0) | (E.GEOM_F64 if geom64 else 0)


def check_cap(engine, field, value, side, geom64, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0)):
    """Cap the current device mesh and compare everything with the definition applied to the fetch before it;
    returns (pre, out, counts)."""
    from oracle import mt3d_cap
    pre = engine.mt3d_fetch()
    c = engine.mt3d_cap(side)
    out = engine.mt3d_fetch()
    want, cnt = mt3d_cap.cap(pre, field, value, side, origin, delta, np.float64 if geom64 else np.float32)
    assert dict(n_verts=c.n_verts, n_tris=c.n_tris, n_cap_verts=c.n_cap_verts, n_cap_tris=c.n_cap_tris,
                n_missing=c.n_missing) == cnt
    for k in ("tris", "keys", "lowmin"):
        assert np.array_equal(out[k], want[k]), k
    assert out["verts"].dtype == want["verts"].dtype and out["verts"].tobytes() == want["verts"].tobytes()
    nV = len(pre["verts"])
    if pre["normals"] is not None:
        assert out["normals"][:nV].tobytes() == pre["normals"].tobytes()
        w = want["normals"][nV:]
        assert (np.abs(out["normals"][nV:] - w) <= np.spacing(np.abs(w))).all()
    return pre, out, c


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_parity_goldens(engine, path, geom64):
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    for side in ("high", "low"):
        engine.mt3d_run(field, value, flags=_flags(geom64))
        check_cap(engine, field, value, side, geom64)


@pytest.mark.parametrize("dtype", DTYPES, ids=[np.dtype(d).name for d in DTYPES])
@pytest.mark.parametrize("geom64", [True, False])
def test_parity_dtypes_origin_delta(engine, dtype, geom64):
    rng = np.random.default_rng(31)
    origin, delta = (0.5, -2.0, 10.25), (0.75, -0.5, 1.25)
    if np.dtype(dtype).kind == "f":
        field, value = rng.standard_normal((13, 17, 11)).astype(dtype), 0.05
    else:
        field, value = rng.integers(0, 9, (13, 17, 11)).astype(dtype), 4.5
    for side in ("high", "low"):
        engine.mt3d_run(field, value, origin=origin, delta=delta, flags=_flags(geom64))
        check_cap(engine, field, value, side, geom64, origin, delta)


# ---------------------------------------------------------------------------------------------- 2. after the cap
@pytest.mark.parametrize("geom64", [True, False])
def test_closed_components_and_volume(engine, geom64):
    field = blob_field(30, 5)
    value = 0.14
    # no sample within the extraction's allclose tolerance of the isovalue: no tetrahedron is skipped and no crossing
    # lies on a grid point, so the capped mesh must be closed
    assert np.abs(field.astype(np.float64) - value).min() > 1e-8 + 1e-5 * value
    origin, delta = (-1.0, 0.5, 2.0), (0.5, 0.25, 0.75)
    vol = {}
    for side in ("high", "low"):                                  # two runs
        c = engine.mt3d_run(field, value, origin=origin, delta=delta, flags=_flags(geom64))
        _, out, cc = check_cap(engine, field, value, side, geom64, origin, delta)
        assert cc.n_missing == 0 and cc.n_tris > c.n_tris
        lab, tab = engine.mt3d_components()
        want = check_oracle(lab, tab, out["verts"], out["tris"])
        assert (tab["n_boundary_edges"] == 0).all() and (tab["n_nonmanifold_edges"] == 0).all()
        assert np.array_equal(tab["n_verts"] - tab["n_edges"] + tab["n_tris"],
                              want["n_verts"] - want["n_edges"] + want["n_tris"])
        assert directed_edges_closed(out["tris"])
        vol[side] = signed_volume(out["verts"], out["tris"])
    box = float(np.prod((np.array(field.shape) - 1) * np.abs(np.array(delta))))
    assert abs(vol["low"] - vol["high"] - box) <= (1e-9 if geom64 else 1e-5) * box


@pytest.mark.parametrize("geom64", [True, False])
def test_passes_after_cap(engine, geom64):
    from oracle import mt3d_smooth
    field = blob_field(28, 9)
    value = 0.1
    engine.mt3d_run(field, value, flags=_flags(geom64))
    check_cap(engine, field, value, "high", geom64)
    _, tab = engine.mt3d_components()
    engine.mt3d_keep_components(np.argsort(-tab["n_tris"], kind="stable")[:3])
    pre = engine.mt3d_fetch()
    engine.mt3d_smooth(3)
    got = engine.mt3d_fetch()["verts"]
    assert got.tobytes() == mt3d_smooth.smooth(pre["verts"], pre["tris"], 3, 0.5, -0.53)[0].tobytes()
    c = engine.mt3d_decimate(2.0)
    assert c.n_tris > 0
    engine.mt3d_orient_reference()
    lab, tab = engine.mt3d_components()
    out = engine.mt3d_fetch()
    check_oracle(lab, tab, out["verts"], out["tris"])


@pytest.mark.parametrize("geom64", [True, False])
def test_interpolate_at_cap_vertices(engine, geom64):
    field = blob_field(24, 4)
    rng = np.random.default_rng(8)
    for a in (rng.standard_normal(field.shape + (3,)), rng.integers(0, 60000, field.shape).astype(np.uint16),
              rng.standard_normal(field.shape).astype(np.float32)):
        for side in ("high", "low"):
            engine.mt3d_run(field, 0.1, flags=_flags(geom64))
            c = engine.mt3d_cap(side)
            out = engine.mt3d_fetch()
            vals = engine.mt3d_interpolate(a)
            nV = c.n_verts - c.n_cap_verts
            p = (out["keys"][nV:] >> np.uint64(3)).astype(np.int64)
            assert (out["keys"][nV:] & np.uint64(7) == 0).all()
            gd = np.float64 if geom64 else np.float32
            want = a.reshape(field.size, -1)[p].astype(gd)
            assert np.array_equal(vals[nV:].reshape(len(p), -1), want)


@pytest.mark.parametrize("geom64", [True, False])
def test_smooth_then_cap(engine, geom64):
    field = blob_field(26, 2)
    value = 0.1
    origin, delta = (1.0, -1.0, 0.5), (0.5, 0.5, 0.25)
    for side in ("high", "low"):
        c = engine.mt3d_run(field, value, origin=origin, delta=delta, flags=_flags(geom64))
        engine.mt3d_smooth(5)
        _, out, cc = check_cap(engine, field, value, side, geom64, origin, delta)
        assert cc.n_missing == 0
        assert directed_edges_closed(out["tris"])                 # the rim joins
        gd = np.float64 if geom64 else np.float32
        shape = np.array(field.shape)
        pts = (out["keys"][c.n_verts:] >> np.uint64(3)).astype(np.int64)
        P = np.stack([pts // (shape[1] * shape[2]), (pts // shape[2]) % shape[1], pts % shape[2]], axis=1)
        on_face = ((P == 0) | (P == shape - 1)).any(axis=1)
        assert on_face.all()
        for a in range(3):                                        # the cap vertices lie exactly on the box faces
            for end in (0, shape[a] - 1):
                sel = P[:, a] == end
                assert (out["verts"][c.n_verts:][sel, a] == gd(end) * gd(delta[a]) + gd(origin[a])).all()


# ---------------------------------------------------------------------------------------------- 3. state and errors
def test_errors_and_states(engine):
    E = _E()
    lib = engine.lib
    cnt = E.CapCounts()

    def call(eng, side=0, reserved=0, p=True, out=True):
        cp = E.CapParams()
        cp.side, cp.reserved = side, reserved
        return eng.lib.ctr_mt3d_cap(eng.h, ctypes.byref(cp) if p else None, ctypes.byref(cnt) if out else None)

    assert lib.ctr_mt3d_cap(None, None, None) == -1
    fresh = E.Engine(0)
    try:
        assert call(fresh) == -5                                      # no run
    finally:
        fresh.close()
    field = np.random.default_rng(14).standard_normal((9, 8, 10))
    flags = E.WANT_NORMALS | E.WANT_KEYS

    def same(pre):
        after = engine.mt3d_fetch()
        for name in ("verts", "normals", "tris", "keys", "lowmin"):
            assert np.array_equal(after[name], pre[name]), name

    engine.mt3d_run(field, 0.0, flags=flags)
    pre = engine.mt3d_fetch()
    for kw in (dict(p=False), dict(out=False), dict(side=2), dict(side=-1), dict(reserved=1)):
        assert call(engine, **kw) == -1, kw
    same(pre)
    with pytest.raises(ValueError):
        engine.mt3d_cap("both")
    engine.mt3d_run(field, 0.0, flags=E.NO_GEOMETRY)
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, flags=E.WANT_NORMALS)                 # no keys
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, flags=flags, i_lo=0, i_hi=5)          # a slab
    assert call(engine) == -5
    engine.mt3d_run(field, 0.0, flags=flags, vert_id_base=7)
    assert call(engine) == -5
    # ids shifted after the run: detected before anything is written
    engine.mt3d_run(field, 0.0, flags=flags)
    engine._check(lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    shifted = engine.mt3d_fetch()
    assert call(engine) == -5
    same(shifted)
    # after a selection, clean-up, component filter, decimation, orientation or an earlier cap
    edits = [lambda: engine.mt3d_select_seeded(np.array([[2, 2, 2]], np.int32)),
             lambda: engine.mt3d_clean(np.array(field.shape) - 1),
             lambda: engine.mt3d_keep_components(np.ones(len(engine.mt3d_components()[1]), bool)),
             lambda: engine.mt3d_decimate(2.0),
             lambda: engine.mt3d_orient_reference(),
             lambda: engine.mt3d_cap("low")]
    for edit in edits:
        engine.mt3d_run(field, 0.0, flags=flags)
        edit()
        pre = engine.mt3d_fetch()
        assert call(engine) == -5
        same(pre)
    # accepted after smoothing, interpolation and components; select and clean refused after a cap
    engine.mt3d_run(field, 0.0, flags=flags)
    engine.mt3d_smooth(2)
    engine.mt3d_interpolate(field)
    engine.mt3d_components()
    assert call(engine, side=1) == 0 and cnt.n_cap_tris > 0
    with pytest.raises(E.EngineError):
        engine.mt3d_keep_components(np.ones(engine._comp_shape[1], bool))   # the components are stale
    engine.mt3d_run(field, 0.0, flags=flags)
    engine.mt3d_cap("high")
    with pytest.raises(E.EngineError, match="capped"):
        engine.mt3d_clean(np.array(field.shape) - 1)
    with pytest.raises(E.EngineError, match="capped"):
        engine.mt3d_select_seeded(np.array([[2, 2, 2]], np.int32))
    # an empty mesh gets the whole box (HIGH) or nothing (LOW)
    c = engine.mt3d_run(field + 10.0, 0.0, flags=flags)
    assert c.n_tris == 0
    assert call(engine, side=1) == 0 and (cnt.n_verts, cnt.n_tris) == (0, 0)
    engine.mt3d_run(field + 10.0, 0.0, flags=flags)
    n0, n1, n2 = field.shape
    assert call(engine, side=0) == 0
    assert cnt.n_tris == 4 * ((n0 - 1) * (n1 - 1) + (n0 - 1) * (n2 - 1) + (n1 - 1) * (n2 - 1))
    assert cnt.n_verts == n0 * n1 * n2 - (n0 - 2) * (n1 - 2) * (n2 - 2)


def test_abi():
    from contourist_b200 import engine as E
    lib = E.load_library()
    assert hasattr(lib, "ctr_mt3d_cap")
    assert ctypes.sizeof(E.CapParams) == 8 and ctypes.sizeof(E.CapCounts) == 40


# ---------------------------------------------------------------------------------------------- 4. full size, façades
@pytest.mark.parametrize("side", ["high", "low"])
def test_full_size_ct_like(engine, side):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    torch.cuda.synchronize()
    host = f.cpu().numpy()
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS | E.WANT_KEYS, shape=(n, n, n), dtype=np.float32)
    _, _, c = check_cap(engine, host, 0.5, side, False)
    if side == "low":                                             # the low region touches nearly the whole box
        assert c.n_cap_tris > 3_000_000
    del f, host
    torch.cuda.empty_cache()


def test_facades(engine):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_cap
    f = lambda x, y, z: np.minimum((x - 0.9) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + (z - 1.0) ** 2 + 0.05)

    def make(cap, post=False):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.3, [])
        t.post_process = post
        t.cap = cap
        t.measure_components = True
        t.search_for_endpoints()
        return t

    plain = make(None)
    p0, t0 = plain.get_points_and_triangles()
    grid = plain.grid
    field = grid.samples(1)
    for side in ("high", "low"):
        t = make(side)
        p1, t1 = t.get_points_and_triangles()
        pre = dict(verts=p0, tris=t0, keys=None, lowmin=None)
        eng = _E().default_engine()
        keys = eng.mt3d_fetch()["keys"]
        pre["keys"], pre["lowmin"] = keys[:len(p0)], np.zeros(len(p0), np.uint8)
        want, cnt = mt3d_cap.cap(pre, field, 0.3, side, tuple(grid.mins), tuple(grid.delta))
        assert np.array_equal(t1, want["tris"]) and np.array_equal(p1, want["verts"])
        assert (t.component_table["n_boundary_edges"] == 0).all()
    with pytest.raises(ValueError):
        make("high", post=True).get_points_and_triangles()
    g = tetrahedral.Grid3DContour(8, 9, 10, lambda x, y, z: (x - 4) ** 2 + (y - 4) ** 2 + z * z - 20.3, 0.0, [])
    g.post_process = False
    g.cap = "low"
    with pytest.raises(ValueError):
        g.get_points_and_triangles()                              # a seeded selection (here: no seeds)
    g.full_scan = True
    pts, tris = g.get_points_and_triangles()
    assert directed_edges_closed(tris)
    g.cap = "sideways"
    with pytest.raises(ValueError):
        g.get_points_and_triangles()
