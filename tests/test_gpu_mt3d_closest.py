"""GPU: closest points of the device mesh to query points (ctr_mt3d_closest, Engine.mt3d_closest, the façades'
closest_points), against oracle/mt3d_closest.py applied to the engine's own fetch: distance, triangle, point and n_found
are compared bit for bit."""
import ctypes

import numpy as np
import pytest

from test_gpu_mt3d_clip import BEFORE_ORDER, FIELDS, PASSES, _code, _flags, _pass_field, sphere_field
from test_gpu_mt3d_keep import blob_field

pytestmark = pytest.mark.gpu

ERR_BAD_ARG, ERR_STATE = -1, -5                                 # CTR_ERR_BAD_ARG, CTR_ERR_STATE


def _E():
    from contourist_b200 import engine as E
    return E


def check(engine, points, max_distance=np.inf, device=False):
    "query the device mesh and compare with the definition on its fetch; returns (result, counts)"
    import torch
    from oracle import mt3d_closest
    pre = engine.mt3d_fetch()
    want, nf = mt3d_closest.closest(pre["verts"], pre["tris"], points, max_distance, prune=True)
    if device:
        d = torch.as_tensor(np.ascontiguousarray(points), device="cuda")
        got, c = engine.mt3d_closest(d.data_ptr(), max_distance, n=len(points), dtype=points.dtype)
        del d
    else:
        got, c = engine.mt3d_closest(points, max_distance)
    assert c.n_found == nf, (c.n_found, nf)
    for k in ("distance", "triangle", "point"):
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k], equal_nan=True), k
    return got, c


def query_sets(mesh, rng, n_rand=2000, n_far=16):
    "random points in the box, far points, every vertex, every edge midpoint, points on triangle planes"
    v = mesh["verts"].astype(np.float64)
    t = mesh["tris"].astype(np.int64)
    lo, hi = v.min(axis=0), v.max(axis=0)
    c, ext = (lo + hi) / 2, (hi - lo).max()
    e = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    e = np.unique(np.sort(e, axis=1), axis=0)
    k = rng.integers(0, len(t), 2000)
    s, w = rng.uniform(-0.5, 1.5, (2, len(k), 1))
    a, b, cc = v[t[k, 0]], v[t[k, 1]], v[t[k, 2]]
    return {"random": rng.uniform(lo - 1, hi + 1, (n_rand, 3)),
            "far": c + rng.normal(size=(n_far, 3)) * 100 * ext,
            "vertices": mesh["verts"],
            "midpoints": (v[e[:, 0]] + v[e[:, 1]]) / 2,
            "planes": a + s * (b - a) + w * (cc - a)}


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("field", list(FIELDS))
def test_parity_query_sets(engine, geom64, field):
    f, v = FIELDS[field]
    engine.mt3d_run(f(), v, flags=_flags(geom64))
    mesh = engine.mt3d_fetch()
    rng = np.random.default_rng(1)
    for name, pts in query_sets(mesh, rng).items():
        got, c = check(engine, np.ascontiguousarray(pts))
        assert c.n_found == len(pts) and c.height > 0, name
        if name == "vertices":
            assert (got["distance"] == 0).all()


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("pdtype", [np.float32, np.float64])
@pytest.mark.parametrize("device", [False, True])
def test_point_inputs(engine, geom64, pdtype, device):
    engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(geom64))
    mesh = engine.mt3d_fetch()
    rng = np.random.default_rng(2)
    sets = query_sets(mesh, rng, n_rand=3000)
    pts = np.concatenate([sets["random"], sets["midpoints"][:2000], sets["vertices"][:500].astype(np.float64)]).astype(pdtype)
    for md in (np.inf, 1.5, 0.0):
        got, c = check(engine, pts, md, device=device)
        if md == 1.5:
            assert 0 < c.n_found < len(pts)


def test_tiny_meshes(engine):
    "one triangle (the root is a leaf), no triangles, and no points"
    f = np.ones((2, 2, 2))
    f[1, 0, 0] = 0.0                                  # a corner off the cube's diagonal: two triangles sharing an edge
    for geom64 in (False, True):
        engine.mt3d_run(f, 0.5, flags=_flags(geom64))
        mesh = engine.mt3d_fetch()
        v, t = mesh["verts"].astype(np.float64), mesh["tris"]
        uses = np.bincount(t.reshape(-1), minlength=len(v))
        u = int(np.nonzero(uses == 1)[0][0])
        others = np.delete(v, u, axis=0)
        rng = np.random.default_rng(12)
        normal = next(n for n in [v[u] - others.mean(axis=0)] + list(rng.normal(size=(1000, 3)))
                      if v[u] @ n > (others @ n).max())
        # keep only vertex u: its one triangle gives one piece, the other is dropped
        engine.mt3d_clip(tuple(normal), float((others @ normal).max() + v[u] @ normal) / 2, "high")
        assert len(engine.mt3d_fetch()["tris"]) == 1
        pts = np.random.default_rng(3).uniform(-1, 2, (100, 3))
        got, c = check(engine, pts)
        assert c.height == 0 and c.n_found == 100
        engine.mt3d_clip((1.0, 0.0, 0.0), -100.0, "low")           # nothing kept: no triangles
        got, c = check(engine, pts)
        assert c.height == 0 and c.n_found == 0 and (got["triangle"] == -1).all()
    got, c = engine.mt3d_closest(np.zeros((0, 3)))
    assert c.n_found == 0 and got["point"].shape == (0, 3)


BEFORE = {
    "selected": lambda e: e.mt3d_select_seeded(np.array([[16, 16, 3]], np.int32)),
    "cleaned": lambda e: e.mt3d_clean(np.array([31, 31, 31])),
    "kept": lambda e: e.mt3d_keep_components(np.argsort(-e.mt3d_components()[1]["n_tris"], kind="stable")[:3]),
    "smoothed": lambda e: e.mt3d_smooth(5),
    "decimated": lambda e: e.mt3d_decimate(2.5),
    "capped": lambda e: e.mt3d_cap("low"),
    "clipped": lambda e: e.mt3d_clip((0.6, 0.2, -0.4), 3.0, "high"),
    "oriented": lambda e: e.mt3d_orient_reference(),
}


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("before", list(BEFORE))
def test_parity_after_each_edit(engine, geom64, before):
    "a query before the edit and one after: the second is on the edited mesh (no stale tree)"
    engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(geom64))
    rng = np.random.default_rng(4)
    sets = query_sets(engine.mt3d_fetch(), rng, n_rand=1500)
    pts = np.concatenate([sets["random"], sets["planes"][:1000]])
    check(engine, pts)
    BEFORE[before](engine)
    check(engine, pts)
    check(engine, np.ascontiguousarray(engine.mt3d_fetch()["verts"]))


def test_positions_written_through_device_pointers(engine):
    "a tree per call: positions moved through mt3d_device_ptrs are seen by the next call"
    import torch
    from test_gpu_mt3d_clip import _from_device
    engine.mt3d_run(sphere_field(), 0.5, flags=_flags(False))
    pts = np.random.default_rng(5).uniform(0, 32, (1000, 3))
    check(engine, pts)
    v, _, _ = engine.mt3d_device_ptrs()
    V = len(engine.mt3d_fetch()["verts"])
    x = _from_device(v, (V, 3), "<f4", host=False)
    x.mul_(0.5)
    torch.cuda.synchronize()
    check(engine, pts)


def test_surface_to_surface_device_points(engine):
    "symmetric distances between a mesh and its decimation, each context's device vertices as the other's points"
    E = _E()
    from oracle import mt3d_closest
    other = E.Engine(0)
    try:
        for geom64 in (False, True):
            gd = np.float64 if geom64 else np.float32
            field = blob_field(32, 7)
            engine.mt3d_run(field, 0.2, flags=_flags(geom64))
            other.mt3d_run(field, 0.2, flags=_flags(geom64))
            other.mt3d_decimate(4.0)
            a, b = engine.mt3d_fetch(), other.mt3d_fetch()
            for src, dst, m_src, m_dst in ((engine, other, a, b), (other, engine, b, a)):
                ptr = src.mt3d_device_ptrs()[0]
                got, c = dst.mt3d_closest(ptr, n=len(m_src["verts"]), dtype=gd)
                want, nf = mt3d_closest.closest(m_dst["verts"], m_dst["tris"], m_src["verts"], prune=True)
                assert c.n_found == nf == len(m_src["verts"])
                for k in want:
                    assert np.array_equal(got[k], want[k], equal_nan=True), k
                assert got["distance"].max() > 0.0
    finally:
        other.close()


# ---------------------------------------------------------------------------------------------- 2. state
def test_state_unchanged_and_passes_accepted(engine):
    E = _E()
    f = blob_field(32, 7)
    engine.mt3d_run(f, 0.2, flags=_flags(False))
    engine.mt3d_interpolate(f)
    vptr = engine.mt3d_interpolate_device_ptr()
    seg, _ = engine.mt3d_section((0.0, 0.0, 1.0), [16.0])
    labels, tab = engine.mt3d_components()
    pre = engine.mt3d_fetch()
    ptrs = engine.mt3d_device_ptrs()
    engine.mt3d_closest(np.random.default_rng(6).uniform(0, 32, (5000, 3)))
    post = engine.mt3d_fetch()
    for k in ("verts", "normals", "tris", "keys", "lowmin"):
        assert np.array_equal(pre[k], post[k]), k
    assert engine.mt3d_device_ptrs() == ptrs and engine.mt3d_interpolate_device_ptr() == vptr
    labels2, tab2 = engine.mt3d_components_fetch()
    assert np.array_equal(labels, labels2) and np.array_equal(tab, tab2)
    S = len(seg["plane"])
    plane = np.empty(S, np.int32)
    engine._check(engine.lib.ctr_mt3d_section_segments_fetch(engine.h, plane.ctypes.data, None, None), "section fetch")
    assert np.array_equal(plane, seg["plane"])
    # the generation: the filter still accepts the measurement made before the query
    engine.mt3d_keep_components(np.ones(len(tab), bool))
    engine.mt3d_closest(np.zeros((1, 3)))


@pytest.mark.parametrize("before", BEFORE_ORDER)
def test_closest_accepted_after(engine, before):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    if before != "run":
        PASSES[before](engine, f)
    assert _code(lambda: check(engine, np.random.default_rng(7).uniform(0, 16, (300, 3)))) == 0, \
        engine.lib.ctr_last_error(engine.h).decode()


@pytest.mark.parametrize("name", list(PASSES))
def test_passes_after_closest(engine, name):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    engine.mt3d_closest(np.random.default_rng(8).uniform(0, 16, (300, 3)))
    got = _code(lambda: PASSES[name](engine, f))
    assert got == 0, (name, got, engine.lib.ctr_last_error(engine.h).decode())


# ---------------------------------------------------------------------------------------------- 3. errors
def _call(engine, points=None, n=None, dtype=1, flags=0, max_distance=np.inf, p=True, out=True):
    E = _E()
    from contourist_b200._bindings import ClosestCounts, ClosestParams
    cp = ClosestParams()
    if points is None:
        points = np.zeros((4, 3))
    cp.points = points if isinstance(points, int) else (points.ctypes.data if points is not None else None)
    cp.dtype, cp.flags = dtype, flags
    cp.n_points = len(points) if n is None else n
    cp.max_distance = max_distance
    c = ClosestCounts()
    return engine.lib.ctr_mt3d_closest(engine.h, ctypes.byref(cp) if p else None, ctypes.byref(c) if out else None)


def _fetch(engine):
    d = np.empty(4096)
    return engine.lib.ctr_mt3d_closest_fetch(engine.h, d.ctypes.data, None, None)


def test_errors(engine):
    import torch
    E = _E()
    assert engine.lib.ctr_mt3d_closest(None, None, None) == ERR_BAD_ARG
    assert engine.lib.ctr_mt3d_closest_fetch(None, None, None, None) == ERR_BAD_ARG
    fresh = E.Engine(0)
    try:
        assert _call(fresh) == ERR_STATE and _fetch(fresh) == ERR_STATE                 # no run
    finally:
        fresh.close()
    field = sphere_field(17)
    flags = _flags(False)
    engine.mt3d_run(field, 0.5, flags=flags)
    assert _fetch(engine) == ERR_STATE                                                   # no call since the run
    assert _call(engine) == 0 and _fetch(engine) == 0
    nanp = np.zeros((4, 3))
    nanp[2, 1] = np.nan
    infp = np.zeros((4, 3), np.float32)
    infp[3, 0] = np.inf
    bad = [dict(p=False), dict(out=False), dict(dtype=2), dict(dtype=-1), dict(flags=2), dict(flags=3), dict(n=-1),
           dict(n=1 << 31), dict(max_distance=np.nan), dict(max_distance=-1.0), dict(max_distance=-np.inf),
           dict(points=nanp), dict(points=infp, dtype=0), dict(points=np.zeros((4, 3)), flags=1)]
    for kw in bad:
        assert _call(engine, **kw) == ERR_BAD_ARG, kw
        assert _fetch(engine) == ERR_STATE, kw                                           # a failed call: no results
    cp_null = dict(points=0, n=4)
    assert _call(engine, **cp_null) == ERR_BAD_ARG
    assert _call(engine, points=0, n=0) == 0
    # a NaN among device points: found on the device, at the first host wait
    d = torch.zeros((1000, 3), dtype=torch.float64, device="cuda")
    d[777, 2] = float("nan")
    assert _call(engine, points=d.data_ptr(), n=1000, flags=1) == ERR_BAD_ARG and _fetch(engine) == ERR_STATE
    d32 = torch.zeros((10, 3), dtype=torch.float32, device="cuda")
    d32[0, 0] = float("-inf")
    assert _call(engine, points=d32.data_ptr(), n=10, dtype=0, flags=1) == ERR_BAD_ARG
    d[777, 2] = 0.0
    assert _call(engine, points=d.data_ptr(), n=1000, flags=1) == 0 and _fetch(engine) == 0
    for kw in (dict(flags=E.NO_GEOMETRY), dict(flags=flags, i_lo=0, i_hi=8), dict(flags=flags, vert_id_base=7)):
        engine.mt3d_run(field, 0.5, **kw)
        assert _call(engine) == ERR_STATE and _fetch(engine) == ERR_STATE, kw
    engine.mt3d_run(field, 0.5, flags=flags)
    engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    assert _call(engine) == ERR_STATE and _fetch(engine) == ERR_STATE
    engine.mt3d_run(field, 0.5, flags=flags)
    for bad_points in (np.zeros((3, 2)), np.zeros(3)):
        with pytest.raises(ValueError):
            engine.mt3d_closest(bad_points)
    with pytest.raises(ValueError):
        engine.mt3d_closest(np.full((2, 3), np.nan))
    with pytest.raises(ValueError):
        engine.mt3d_closest(d.data_ptr())
    with pytest.raises(ValueError):
        engine.mt3d_closest(d.data_ptr(), n=1000, dtype=np.int32)


def test_abi():
    E = _E()
    from contourist_b200._bindings import ClosestCounts, ClosestParams
    lib = E.load_library()
    assert hasattr(lib, "ctr_mt3d_closest") and hasattr(lib, "ctr_mt3d_closest_fetch")
    assert ctypes.sizeof(ClosestParams) == 32 and ctypes.sizeof(ClosestCounts) == 16


def test_fetch_into_device_memory(engine):
    import torch
    engine.mt3d_run(sphere_field(), 0.5, flags=_flags(False))
    pts = np.random.default_rng(9).uniform(0, 32, (777, 3))
    got, _ = engine.mt3d_closest(pts)
    d = torch.empty(777, dtype=torch.float64, device="cuda")
    t = torch.empty(777, dtype=torch.int32, device="cuda")
    q = torch.empty((777, 3), dtype=torch.float64, device="cuda")
    engine._check(engine.lib.ctr_mt3d_closest_fetch(engine.h, d.data_ptr(), t.data_ptr(), q.data_ptr()), "fetch")
    assert np.array_equal(d.cpu().numpy(), got["distance"]) and np.array_equal(t.cpu().numpy(), got["triangle"])
    assert np.array_equal(q.cpu().numpy(), got["point"])


# ---------------------------------------------------------------------------------------------- 4. façade, full size
def test_facade_closest_points(engine):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_closest
    f = lambda x, y, z: np.minimum((x - 0.3) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + (z - 0.6) ** 2 + 0.05)
    Q = np.random.default_rng(10).uniform(-1.2, 1.2, (500, 3))
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.3, [])
    t.post_process = False
    t.smooth_iterations = 3
    t.sections = ((0.0, 0.0, 1.0), [0.1])
    t.closest_points = Q
    t.search_for_endpoints()
    p, tr = t.get_points_and_triangles()
    want, nf = mt3d_closest.closest(p, tr, Q, prune=True)
    assert nf == len(Q)
    for k in want:
        assert np.array_equal(t.closest[k], want[k]), k
    t.closest_points = np.zeros((3, 2))
    with pytest.raises(ValueError):
        t.get_points_and_triangles()


def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS | E.WANT_KEYS, shape=(n, n, n), dtype=np.float32)
    del f
    torch.cuda.empty_cache()
    mesh = engine.mt3d_fetch()
    rng = np.random.default_rng(11)
    v = mesh["verts"].astype(np.float64)
    t = mesh["tris"][rng.integers(0, len(mesh["tris"]), 200)]
    on = (v[t[:, 0]] + v[t[:, 1]] + v[t[:, 2]]) / 3
    pts = np.concatenate([rng.uniform(0, n - 1, (300, 3)), on, v[rng.integers(0, len(v), 100)]])
    got, c = check(engine, pts)
    assert c.n_found == len(pts) and c.height >= 23
