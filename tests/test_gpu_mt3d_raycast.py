"""GPU: first hits of rays on the device mesh (ctr_mt3d_raycast, Engine.mt3d_raycast, the façades' rays), against
oracle/mt3d_raycast.py applied to the engine's own fetch: t, triangle, weights, point, side and n_hit are compared bit for
bit."""
import ctypes

import numpy as np
import pytest

from test_gpu_mt3d_clip import BEFORE_ORDER, FIELDS, PASSES, _code, _flags, _from_device, _pass_field, sphere_field
from test_gpu_mt3d_closest import BEFORE
from test_gpu_mt3d_keep import blob_field

pytestmark = pytest.mark.gpu

ERR_BAD_ARG, ERR_STATE = -1, -5                                 # CTR_ERR_BAD_ARG, CTR_ERR_STATE
KEYS = ("t", "triangle", "weights", "point", "side")


def _E():
    from contourist_b200 import engine as E
    return E


def check(engine, O, D, t_min=0.0, t_max=np.inf, device=False):
    "cast the rays at the device mesh and compare with the definition on its fetch; returns (result, counts)"
    import torch
    from oracle import mt3d_raycast
    pre = engine.mt3d_fetch()
    want, nh = mt3d_raycast.raycast(pre["verts"], pre["tris"], O, D, t_min, t_max, prune=True)
    if device:
        o = torch.as_tensor(np.ascontiguousarray(O), device="cuda")
        d = torch.as_tensor(np.ascontiguousarray(D), device="cuda")
        got, c = engine.mt3d_raycast(o.data_ptr(), d.data_ptr(), t_min, t_max, n=len(O), dtype=O.dtype)
        del o, d
    else:
        got, c = engine.mt3d_raycast(O, D, t_min, t_max)
    assert c.n_hit == nh, (c.n_hit, nh)
    for k in KEYS:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k], equal_nan=True), k
    return got, c


def ray_sets(mesh, rng, n=1500):
    """random rays in the box; rays aimed at vertices, edge midpoints and centroids; in-plane and axis-parallel rays;
    rays that miss the box; far origins; vertex-along-normal rays (with t_min > 0 when cast)"""
    v = mesh["verts"].astype(np.float64)
    t = mesh["tris"].astype(np.int64)
    lo, hi = v.min(axis=0), v.max(axis=0)
    ext = (hi - lo).max()
    k = t[rng.integers(0, len(t), n)]
    a, b, c = v[k[:, 0]], v[k[:, 1]], v[k[:, 2]]
    O = rng.uniform(lo - 2, hi + 2, (n, 3))
    axis = np.eye(3)[rng.integers(0, 3, n)] * rng.choice([-1.0, 1.0], (n, 1))
    far = (lo + hi) / 2 + rng.normal(size=(n, 3)) * 100 * ext
    iv = rng.integers(0, len(v), n)
    sets = {"random": (rng.uniform(lo, hi, (n, 3)), rng.normal(size=(n, 3))),
            "vertices": (O, a - O), "midpoints": (O, (a + b) / 2 - O), "centroids": (O, (a + b + c) / 3 - O),
            "in_plane": (a - 0.5 * (b - a), b - a),
            "axis": (rng.uniform(lo, hi, (n, 3)), axis),
            "axis_at_vertices": (a - 2 * ext * axis, axis),
            "miss_box": (np.broadcast_to(hi + ext, (n, 3)), rng.uniform(0.1, 1.0, (n, 3))),
            "far": (far, rng.uniform(lo, hi, (n, 3)) - far),
            "normals": (v[iv], mesh["normals"][iv].astype(np.float64))}
    for name, (o, d) in sets.items():                 # an edge of a zero-area triangle gives no direction
        sets[name] = (np.ascontiguousarray(o), np.ascontiguousarray(np.where((d == 0).all(axis=1, keepdims=True), [1.0, 0, 0], d)))
    return sets


def cast_sets(engine, rng, n=1500, dtype=np.float64, device=False):
    for name, (O, D) in ray_sets(engine.mt3d_fetch(), rng, n).items():
        t_min = 1e-3 if name == "normals" else 0.0
        got, c = check(engine, O.astype(dtype), D.astype(dtype), t_min=t_min, device=device)
        if name in ("centroids", "midpoints"):
            assert c.n_hit > 0.5 * len(O), name
        if name == "miss_box":
            assert c.n_hit == 0


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("field", list(FIELDS))
def test_parity_ray_sets(engine, geom64, field):
    f, v = FIELDS[field]
    engine.mt3d_run(f(), v, flags=_flags(geom64))
    cast_sets(engine, np.random.default_rng(1))


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("rdtype", [np.float32, np.float64])
@pytest.mark.parametrize("device", [False, True])
def test_ray_inputs(engine, geom64, rdtype, device):
    engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(geom64))
    cast_sets(engine, np.random.default_rng(2), n=700, dtype=rdtype, device=device)
    O, D = ray_sets(engine.mt3d_fetch(), np.random.default_rng(3), 2000)["random"]
    for t_min, t_max in ((0.0, 2.0), (-np.inf, np.inf), (1.0, 1.0), (np.inf, np.inf)):
        check(engine, O.astype(rdtype), D.astype(rdtype), t_min, t_max, device=device)


def test_tiny_meshes(engine):
    "one and two triangles (the root a leaf, and one node), no triangles, and no rays"
    f = np.ones((2, 2, 2))
    f[1, 0, 0] = 0.0                                  # a corner off the cube's diagonal: two triangles sharing an edge
    rng = np.random.default_rng(12)
    for geom64 in (False, True):
        engine.mt3d_run(f, 0.5, flags=_flags(geom64))
        mesh = engine.mt3d_fetch()
        v, t = mesh["verts"].astype(np.float64), mesh["tris"]
        assert len(t) == 2
        O = rng.uniform(-1, 2, (300, 3))
        aim = np.concatenate([v[t].mean(axis=1), (v[t[:, 0]] + v[t[:, 1]]) / 2, v])
        aim = aim[rng.integers(0, len(aim), 300)]
        got, c = check(engine, O, aim - O)
        assert c.height == 1 and c.n_hit > 0
        uses = np.bincount(t.reshape(-1), minlength=len(v))
        u = int(np.nonzero(uses == 1)[0][0])
        others = np.delete(v, u, axis=0)
        normal = next(n for n in [v[u] - others.mean(axis=0)] + list(rng.normal(size=(1000, 3)))
                      if v[u] @ n > (others @ n).max())
        engine.mt3d_clip(tuple(normal), float((others @ normal).max() + v[u] @ normal) / 2, "high")
        assert len(engine.mt3d_fetch()["tris"]) == 1
        tri = engine.mt3d_fetch()
        cen = tri["verts"][tri["tris"][0]].astype(np.float64).mean(axis=0)
        got, c = check(engine, O, cen - O)
        assert c.height == 0 and c.n_hit == 300
        engine.mt3d_clip((1.0, 0.0, 0.0), -100.0, "low")           # nothing kept: no triangles
        got, c = check(engine, O, cen - O)
        assert c.height == 0 and c.n_hit == 0 and (got["triangle"] == -1).all() and (got["side"] == 0).all()
    got, c = engine.mt3d_raycast(np.zeros((0, 3)), np.zeros((0, 3)))
    assert c.n_hit == 0 and got["point"].shape == (0, 3)


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("before", list(BEFORE))
def test_parity_after_each_edit(engine, geom64, before):
    "a cast before the edit and one after: the second is on the edited mesh (no stale tree)"
    engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(geom64))
    sets = ray_sets(engine.mt3d_fetch(), np.random.default_rng(4), 1000)
    O = np.concatenate([sets["random"][0], sets["centroids"][0]])
    D = np.concatenate([sets["random"][1], sets["centroids"][1]])
    check(engine, O, D)
    BEFORE[before](engine)
    check(engine, O, D)
    if len(engine.mt3d_fetch()["tris"]):              # the seeded selection may keep nothing
        cast_sets(engine, np.random.default_rng(5), n=500)


def test_positions_written_through_device_pointers(engine):
    "a tree per call: positions moved through mt3d_device_ptrs are seen by the next call"
    import torch
    engine.mt3d_run(sphere_field(), 0.5, flags=_flags(False))
    rng = np.random.default_rng(5)
    O = rng.uniform(0, 32, (1000, 3))
    D = rng.normal(size=(1000, 3))
    check(engine, O, D)
    v, _, _ = engine.mt3d_device_ptrs()
    V = len(engine.mt3d_fetch()["verts"])
    x = _from_device(v, (V, 3), "<f4", host=False)
    x.mul_(0.5)
    torch.cuda.synchronize()
    check(engine, O, D)


def test_thickness_from_own_device_pointers(engine):
    "every vertex along its normal, origins and directions the engine's own device arrays, t_min > 0"
    from oracle import mt3d_raycast
    for geom64 in (False, True):
        engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(geom64))
        mesh = engine.mt3d_fetch()
        v, nrm, _ = engine.mt3d_device_ptrs()
        V = len(mesh["verts"])
        got, c = engine.mt3d_raycast(v, nrm, 1e-3, n=V, dtype=np.float64 if geom64 else np.float32)
        want, nh = mt3d_raycast.raycast(mesh["verts"], mesh["tris"], mesh["verts"], mesh["normals"], 1e-3, prune=True)
        assert c.n_hit == nh and 0 < nh < V
        for k in KEYS:
            assert np.array_equal(got[k], want[k], equal_nan=True), k
        # the normals point up the field: the ray leaves through the far wall of the high region, from inside it
        assert (got["side"][got["triangle"] >= 0] == 1).mean() > 0.9


# ---------------------------------------------------------------------------------------------- 2. inside / outside
@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("field", ["sphere", "noise"])
def test_inside_outside_capped(engine, geom64, field):
    "on the HIGH-capped mesh the first hit's side tells the region of the origin"
    f, iso = FIELDS[field]
    f = f()
    engine.mt3d_run(f, iso, flags=_flags(geom64))
    engine.mt3d_cap("high")
    rng = np.random.default_rng(6)
    P = rng.uniform(0, np.array(f.shape) - 1, (200000, 3))
    i = np.minimum(np.floor(P).astype(np.int64), np.array(f.shape) - 2)
    corners = np.stack([f[i[:, 0] + a, i[:, 1] + b, i[:, 2] + c] for a in (0, 1) for b in (0, 1) for c in (0, 1)], axis=1)
    high, low = (corners >= iso).all(axis=1), (corners < iso).all(axis=1)
    O = np.concatenate([P[high][:1500], P[low][:1500]])
    D = rng.normal(size=(len(O), 3))
    got, c = check(engine, O, D)
    nh = min(1500, int(high.sum()))
    assert nh > 100 and len(O) - nh > 100
    assert (got["triangle"][:nh] >= 0).all() and (got["side"][:nh] == 1).all()
    assert (got["side"][nh:] != 1).all()


# ---------------------------------------------------------------------------------------------- 3. state
def test_state_unchanged_and_passes_accepted(engine):
    f = blob_field(32, 7)
    engine.mt3d_run(f, 0.2, flags=_flags(False))
    engine.mt3d_interpolate(f)
    vptr = engine.mt3d_interpolate_device_ptr()
    seg, _ = engine.mt3d_section((0.0, 0.0, 1.0), [16.0])
    labels, tab = engine.mt3d_components()
    q, _ = engine.mt3d_closest(np.random.default_rng(6).uniform(0, 32, (500, 3)))
    pre = engine.mt3d_fetch()
    ptrs = engine.mt3d_device_ptrs()
    rng = np.random.default_rng(7)
    engine.mt3d_raycast(rng.uniform(0, 32, (5000, 3)), rng.normal(size=(5000, 3)))
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
    dist = np.empty(500)
    engine._check(engine.lib.ctr_mt3d_closest_fetch(engine.h, dist.ctypes.data, None, None), "closest fetch")
    assert np.array_equal(dist, q["distance"])
    engine.mt3d_keep_components(np.ones(len(tab), bool))         # the generation: the measurement is still current
    engine.mt3d_raycast(np.zeros((1, 3)), np.ones((1, 3)))


@pytest.mark.parametrize("before", BEFORE_ORDER)
def test_raycast_accepted_after(engine, before):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    if before != "run":
        PASSES[before](engine, f)
    rng = np.random.default_rng(8)
    assert _code(lambda: check(engine, rng.uniform(0, 16, (300, 3)), rng.normal(size=(300, 3)))) == 0, \
        engine.lib.ctr_last_error(engine.h).decode()


@pytest.mark.parametrize("name", list(PASSES))
def test_passes_after_raycast(engine, name):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    rng = np.random.default_rng(9)
    engine.mt3d_raycast(rng.uniform(0, 16, (300, 3)), rng.normal(size=(300, 3)))
    got = _code(lambda: PASSES[name](engine, f))
    assert got == 0, (name, got, engine.lib.ctr_last_error(engine.h).decode())


def test_closest_and_raycast_alternate(engine):
    from test_gpu_mt3d_closest import check as check_closest
    engine.mt3d_run(blob_field(32, 7), 0.2, flags=_flags(True))
    rng = np.random.default_rng(10)
    for _ in range(3):
        check_closest(engine, rng.uniform(0, 32, (800, 3)))
        check(engine, rng.uniform(0, 32, (800, 3)), rng.normal(size=(800, 3)))
    d = np.empty(800)
    engine._check(engine.lib.ctr_mt3d_closest_fetch(engine.h, d.ctypes.data, None, None), "closest fetch")
    assert np.isfinite(d).all()


# ---------------------------------------------------------------------------------------------- 4. errors
def _call(engine, O=None, D=None, n=None, dtype=1, flags=0, t_min=0.0, t_max=np.inf, p=True, out=True):
    from contourist_b200._bindings import RayCounts, RayParams
    rp = RayParams()
    if O is None:
        O = np.zeros((4, 3))
    if D is None:
        D = np.ones((4, 3))
    rp.origins = O if isinstance(O, int) else O.ctypes.data
    rp.directions = D if isinstance(D, int) else D.ctypes.data
    rp.dtype, rp.flags = dtype, flags
    rp.n_rays = (4 if isinstance(O, int) else len(O)) if n is None else n
    rp.t_min, rp.t_max = t_min, t_max
    c = RayCounts()
    return engine.lib.ctr_mt3d_raycast(engine.h, ctypes.byref(rp) if p else None, ctypes.byref(c) if out else None)


def _fetch(engine):
    t = np.empty(4096)
    return engine.lib.ctr_mt3d_raycast_fetch(engine.h, t.ctypes.data, None, None, None, None)


def test_errors(engine):
    import torch
    E = _E()
    assert engine.lib.ctr_mt3d_raycast(None, None, None) == ERR_BAD_ARG
    assert engine.lib.ctr_mt3d_raycast_fetch(None, None, None, None, None, None) == ERR_BAD_ARG
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
    nan_o = np.zeros((4, 3))
    nan_o[2, 1] = np.nan
    inf_d = np.ones((4, 3), np.float32)
    inf_d[3, 0] = np.inf
    zero_d = np.ones((4, 3))
    zero_d[1] = 0.0
    bad = [dict(p=False), dict(out=False), dict(dtype=2), dict(dtype=-1), dict(flags=2), dict(flags=3), dict(n=-1),
           dict(n=1 << 31), dict(t_min=np.nan), dict(t_max=np.nan), dict(t_min=1.0, t_max=0.5),
           dict(t_min=np.inf, t_max=-np.inf), dict(O=nan_o), dict(O=np.zeros((4, 3), np.float32), D=inf_d, dtype=0),
           dict(D=zero_d), dict(flags=1)]
    for kw in bad:
        assert _call(engine, **kw) == ERR_BAD_ARG, kw
        assert _fetch(engine) == ERR_STATE, kw                                           # a failed call: no results
    assert _call(engine, O=0, n=4) == ERR_BAD_ARG and _call(engine, D=0, n=4) == ERR_BAD_ARG
    assert _call(engine, O=0, D=0, n=0) == 0
    # bad device rays: found on the device, at the first host wait
    o = torch.zeros((1000, 3), dtype=torch.float64, device="cuda")
    d = torch.ones((1000, 3), dtype=torch.float64, device="cuda")
    for t, idx, val in ((o, (777, 2), float("nan")), (d, (5, 0), float("-inf")), (d, (999,), 0.0)):
        keep = t[idx].clone()
        t[idx] = val
        assert _call(engine, O=o.data_ptr(), D=d.data_ptr(), n=1000, flags=1) == ERR_BAD_ARG and _fetch(engine) == ERR_STATE
        t[idx] = keep
    o32 = torch.zeros((10, 3), dtype=torch.float32, device="cuda")
    d32 = torch.ones((10, 3), dtype=torch.float32, device="cuda")
    d32[0] = 0.0
    assert _call(engine, O=o32.data_ptr(), D=d32.data_ptr(), n=10, dtype=0, flags=1) == ERR_BAD_ARG
    assert _call(engine, O=o.data_ptr(), D=d.data_ptr(), n=1000, flags=1) == 0 and _fetch(engine) == 0
    host = np.ones((1000, 3))
    assert _call(engine, O=o.data_ptr(), D=host.ctypes.data, n=1000, flags=1) == ERR_BAD_ARG
    for kw in (dict(flags=E.NO_GEOMETRY), dict(flags=flags, i_lo=0, i_hi=8), dict(flags=flags, vert_id_base=7)):
        engine.mt3d_run(field, 0.5, **kw)
        assert _call(engine) == ERR_STATE and _fetch(engine) == ERR_STATE, kw
    engine.mt3d_run(field, 0.5, flags=flags)
    engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    assert _call(engine) == ERR_STATE and _fetch(engine) == ERR_STATE
    engine.mt3d_run(field, 0.5, flags=flags)
    for bo, bd in ((np.zeros((3, 2)), np.ones((3, 2))), (np.zeros(3), np.ones(3)), (np.zeros((3, 3)), np.ones((2, 3)))):
        with pytest.raises(ValueError):
            engine.mt3d_raycast(bo, bd)
    with pytest.raises(ValueError):
        engine.mt3d_raycast(np.full((2, 3), np.nan), np.ones((2, 3)))
    with pytest.raises(ValueError):
        engine.mt3d_raycast(o.data_ptr(), d.data_ptr())
    with pytest.raises(ValueError):
        engine.mt3d_raycast(o.data_ptr(), d.data_ptr(), n=1000, dtype=np.int32)


def test_abi():
    E = _E()
    from contourist_b200._bindings import RayCounts, RayParams
    lib = E.load_library()
    assert hasattr(lib, "ctr_mt3d_raycast") and hasattr(lib, "ctr_mt3d_raycast_fetch")
    assert ctypes.sizeof(RayParams) == 48 and ctypes.sizeof(RayCounts) == 16


def test_fetch_into_device_memory(engine):
    import torch
    engine.mt3d_run(sphere_field(), 0.5, flags=_flags(False))
    rng = np.random.default_rng(11)
    got, _ = engine.mt3d_raycast(rng.uniform(0, 32, (777, 3)), rng.normal(size=(777, 3)))
    dev = dict(t=torch.empty(777, dtype=torch.float64, device="cuda"), triangle=torch.empty(777, dtype=torch.int32, device="cuda"),
               weights=torch.empty((777, 3), dtype=torch.float64, device="cuda"),
               point=torch.empty((777, 3), dtype=torch.float64, device="cuda"), side=torch.empty(777, dtype=torch.int8, device="cuda"))
    engine._check(engine.lib.ctr_mt3d_raycast_fetch(engine.h, *(dev[k].data_ptr() for k in KEYS)), "fetch")
    for k in KEYS:
        assert np.array_equal(dev[k].cpu().numpy(), got[k], equal_nan=True), k


# ---------------------------------------------------------------------------------------------- 5. façade, full size
def test_facade_rays(engine):
    from contourist_b200 import tetrahedral
    from oracle import mt3d_raycast
    f = lambda x, y, z: np.minimum((x - 0.3) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + (z - 0.6) ** 2 + 0.05)
    rng = np.random.default_rng(12)
    O = rng.uniform(-1.2, 1.2, (500, 3))
    D = rng.normal(size=(500, 3))
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.3, [])
    t.post_process = False
    t.smooth_iterations = 3
    t.closest_points = O
    t.rays = (O, D)
    t.search_for_endpoints()
    p, tr = t.get_points_and_triangles()
    want, nh = mt3d_raycast.raycast(p, tr, O, D, prune=True)
    assert 0 < nh < len(O)
    for k in want:
        assert np.array_equal(t.ray_hits[k], want[k], equal_nan=True), k
    t.rays = (np.zeros((3, 2)), np.ones((3, 2)))
    with pytest.raises(ValueError):
        t.get_points_and_triangles()


def camera_rays(n, res, rng=None):
    "a res x res pinhole camera outside the box [0, n-1]^3, aimed at its centre"
    c = np.full(3, (n - 1) / 2)
    eye = c + np.array([1.3, 0.9, 0.7]) * n
    fwd = (c - eye) / np.linalg.norm(c - eye)
    right = np.cross(fwd, [0.0, 0.0, 1.0])
    right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    s = (np.arange(res) + 0.5) / res * 2 - 1
    U, V = np.meshgrid(s, s, indexing="xy")
    D = fwd + 0.45 * (U.reshape(-1, 1) * right + V.reshape(-1, 1) * up)
    return np.broadcast_to(eye, D.shape).copy(), D


def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    from oracle import mt3d_raycast
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS | E.WANT_KEYS, shape=(n, n, n), dtype=np.float32)
    del f
    torch.cuda.empty_cache()
    mesh = engine.mt3d_fetch()
    rng = np.random.default_rng(13)
    Oc, Dc = camera_rays(n, 1024)
    cases = {"camera_1k": (Oc, Dc, 0.0), "random_1m": (rng.uniform(0, n - 1, (1 << 20, 3)), rng.normal(size=(1 << 20, 3)), 0.0)}
    for name, (O, D, t_min) in cases.items():
        got, c = engine.mt3d_raycast(O, D, t_min)
        idx = rng.integers(0, len(O), 150)
        want, _ = mt3d_raycast.raycast(mesh["verts"], mesh["tris"], O[idx], D[idx], t_min, prune=True)
        for k in KEYS:
            assert np.array_equal(got[k][idx], want[k], equal_nan=True), (name, k)
        assert c.height >= 23 and 0 < c.n_hit <= len(O)
    v, nrm, _ = engine.mt3d_device_ptrs()
    V = len(mesh["verts"])
    got, c = engine.mt3d_raycast(v, nrm, 1e-3, n=V, dtype=np.float32)
    idx = rng.integers(0, V, 150)
    want, _ = mt3d_raycast.raycast(mesh["verts"], mesh["tris"], mesh["verts"][idx], mesh["normals"][idx], 1e-3, prune=True)
    for k in KEYS:
        assert np.array_equal(got[k][idx], want[k], equal_nan=True), ("thickness", k)
    assert c.n_hit > 0.5 * V
