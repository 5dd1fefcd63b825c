"""GPU: clipping of the device mesh by a plane or a vertex value (ctr_mt3d_clip, Engine.mt3d_clip, the façades'
clip_halfspaces), against oracle/mt3d_clip.py applied to the engine's own fetch: counts, triangles, positions, normals,
keys, lowmin and carried vertex values are compared bit for bit."""
import ctypes
import re

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


def sphere_field(n=33):
    g = np.linspace(-1.0, 1.0, n)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    return X * X + Y * Y + Z * Z


def ct128():
    import torch
    from contourist_b200 import synthetic
    f = synthetic.ct_like(128, device="cuda")
    torch.cuda.synchronize()
    return f.cpu().numpy()


def mask_field():
    return (blob_field(24, 5) > 0.1).astype(np.uint8)


FIELDS = {"sphere": (sphere_field, 0.5), "noise": (lambda: blob_field(32, 7), 0.2), "ct128": (ct128, 0.5),
          "mask": (mask_field, 0.5)}


def values_of(engine, ncomp):
    "the current vertex values (ctr_mt3d_interpolate_fetch), [V, ncomp] in the geometry type"
    E = _E()
    flags, c = engine._last3
    out = np.empty((int(c.n_verts), ncomp), np.float64 if flags & E.GEOM_F64 else np.float32)
    engine._check(engine.lib.ctr_mt3d_interpolate_fetch(engine.h, out.ctypes.data), "ctr_mt3d_interpolate_fetch")
    return out


def check_clip(engine, normal=None, offset=0.0, keep="high", component=None, ncomp=0):
    "clip the device mesh and compare with the definition on its fetch; returns (oracle mesh, counts)"
    from oracle import mt3d_clip
    pre = engine.mt3d_fetch()
    vals = values_of(engine, ncomp) if ncomp else None
    gd = pre["verts"].dtype
    want, wc = mt3d_clip.clip(pre["verts"], pre["tris"], normals=pre["normals"], keys=pre["keys"], lowmin=pre["lowmin"],
                              values=vals, normal=normal, component=component, offset=offset, side=keep, geom_dtype=gd)
    c = engine.mt3d_clip(normal=normal, offset=offset, keep=keep, component=component)
    got = (c.n_verts, c.n_tris, c.n_new_verts, c.n_cut_tris, c.n_dropped_tris)
    assert got == tuple(wc[k] for k in ("n_verts", "n_tris", "n_new_verts", "n_cut_tris", "n_dropped_tris")), got
    post = engine.mt3d_fetch()
    for k in ("tris", "verts", "normals", "keys", "lowmin"):
        if want[k] is None:
            continue
        assert post[k].dtype == np.asarray(want[k]).dtype or k == "tris", k
        assert np.array_equal(post[k], np.asarray(want[k]).reshape(post[k].shape)), k
    if ncomp:
        assert np.array_equal(values_of(engine, ncomp), np.asarray(want["values"]).reshape(-1, ncomp))
    return want, wc


def _median_plane(mesh, normal):
    s = mesh["verts"].astype(np.float64) @ np.asarray(normal, np.float64)
    return float(np.median(s)) + 1e-3


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("field", list(FIELDS))
@pytest.mark.parametrize("keep", ["high", "low"])
def test_parity_plane(engine, geom64, field, keep):
    f, v = FIELDS[field]
    engine.mt3d_run(f(), v, flags=_flags(geom64))
    for normal in [(1.0, 0.0, 0.0), (0.3, -0.5, 0.8)]:
        engine.mt3d_run(f(), v, flags=_flags(geom64))
        _, wc = check_clip(engine, normal, _median_plane(engine.mt3d_fetch(), normal), keep)
        assert wc["n_new_verts"] > 0 and wc["n_dropped_tris"] > 0


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("field", ["sphere", "noise", "mask"])
@pytest.mark.parametrize("keep", ["high", "low"])
def test_parity_value(engine, geom64, field, keep):
    f, v = FIELDS[field]
    fld = f()
    engine.mt3d_run(fld, v, flags=_flags(geom64))
    n = fld.shape
    second = np.stack(np.meshgrid(*[np.arange(k, dtype=np.float64) for k in n], indexing="ij"), axis=-1)
    second = np.concatenate([second, np.sin(second[..., :1] * 0.3) * second[..., 1:2]], axis=-1)   # 4 components
    vals = engine.mt3d_interpolate(second)
    for comp in (0, 3):
        engine.mt3d_run(fld, v, flags=_flags(geom64))
        engine.mt3d_interpolate(second)
        _, wc = check_clip(engine, component=comp, offset=float(np.median(vals[:, comp])), keep=keep, ncomp=4)
        assert wc["n_new_verts"] > 0
    # a clip after a plane clip: the carried values are those of the clipped mesh
    engine.mt3d_run(fld, v, flags=_flags(geom64))
    engine.mt3d_interpolate(second[..., :1])
    check_clip(engine, (0.0, 1.0, 0.0), _median_plane(engine.mt3d_fetch(), (0.0, 1.0, 0.0)), keep, ncomp=1)
    check_clip(engine, component=0, offset=float(np.median(vals[:, 0])), keep=keep, ncomp=1)


BEFORE = {
    "smoothed": lambda e: e.mt3d_smooth(5),
    "decimated": lambda e: e.mt3d_decimate(2.5),
    "capped": lambda e: e.mt3d_cap("low"),
    "oriented": lambda e: e.mt3d_orient_reference(),
    "kept": lambda e: e.mt3d_keep_components(np.argsort(-e.mt3d_components()[1]["n_tris"], kind="stable")[:3]),
    "clipped": lambda e: e.mt3d_clip((0.0, 0.0, 1.0), 20.0, "low"),
}


@pytest.mark.parametrize("geom64", [False, True])
@pytest.mark.parametrize("before", list(BEFORE))
def test_parity_after_passes(engine, geom64, before):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.2, flags=_flags(geom64))
    BEFORE[before](engine)
    normal = (0.6, 0.2, -0.4)
    check_clip(engine, normal, _median_plane(engine.mt3d_fetch(), normal), "high")


def test_full_size_ct_like(engine):
    import torch
    from contourist_b200 import synthetic
    E = _E()
    n = 512
    f = synthetic.ct_like(n, device="cuda")
    engine.mt3d_run(f.data_ptr(), 0.5, flags=E.WANT_NORMALS | E.WANT_KEYS, shape=(n, n, n), dtype=np.float32)
    normal = (1.0, 2.0, 3.0)
    _, wc = check_clip(engine, normal, 3.0 * n + 0.25, "high")
    assert wc["n_cut_tris"] > 10000
    del f
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- 2. properties
@pytest.mark.parametrize("geom64", [False, True])
def test_rim_is_the_section_and_keys_are_the_kept_ends(engine, geom64):
    from oracle import mt3d_clip
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.2, flags=_flags(geom64))
    normal = (0.3, -0.5, 0.8)
    pre = engine.mt3d_fetch()
    d = _median_plane(pre, normal)
    seg, _ = engine.mt3d_section(normal, [d])
    c = engine.mt3d_clip(normal, d, "high")
    post = engine.mt3d_fetch()
    nk = c.n_verts - c.n_new_verts
    rim = post["verts"][nk:]
    assert np.array_equal(np.unique(rim, axis=0), np.unique(seg["points"].reshape(-1, 3), axis=0))
    # each new vertex's key is its kept end's: the edge's end with s >= d
    s = pre["verts"].astype(np.float64) @ np.asarray(normal)
    edges = np.unique(np.sort(seg["edges"].reshape(-1, 2), axis=1), axis=0)
    ends = {tuple(e) for e in edges}
    kept_end_keys = {int(pre["keys"][a if s[a] >= d else b]) for a, b in ends}
    assert set(post["keys"][nk:].tolist()) <= kept_end_keys
    assert len(mt3d_clip.SIDES) == 2


@pytest.mark.parametrize("geom64", [False, True])
def test_clip_then_smooth_keeps_the_cut(engine, geom64):
    field = blob_field(32, 7)
    engine.mt3d_run(field, 0.2, flags=_flags(geom64))
    normal = (0.0, 1.0, 0.0)
    c = engine.mt3d_clip(normal, _median_plane(engine.mt3d_fetch(), normal), "low")
    pre = engine.mt3d_fetch()
    engine.mt3d_smooth(10)
    post = engine.mt3d_fetch()
    nk = c.n_verts - c.n_new_verts
    assert np.array_equal(pre["verts"][nk:], post["verts"][nk:])
    assert not np.array_equal(pre["verts"][:nk], post["verts"][:nk])


def test_half_sphere_is_a_disc(engine):
    field = sphere_field(41)
    engine.mt3d_run(field, 0.5, flags=_flags(True))
    seg, polys = engine.mt3d_section((0.0, 0.0, 1.0), [20.0 + 1e-3])         # (the rim of the clip lies on the plane)
    c = engine.mt3d_clip((0.0, 0.0, 1.0), 20.0 + 1e-3, "high")
    _, tab = engine.mt3d_components()
    assert len(tab) == 1
    r = tab[0]
    assert int(r["n_verts"]) - int(r["n_edges"]) + int(r["n_tris"]) == 1
    assert int(r["n_boundary_edges"]) == len(seg["plane"]) and c.n_new_verts == len(seg["plane"])
    assert polys[0] is not None and len(polys[0]) == 1 and polys[0][0][0]


def test_noop_and_empty(engine):
    field = sphere_field()
    engine.mt3d_run(field, 0.5, flags=_flags(False))
    pre = engine.mt3d_fetch()
    ptrs = engine.mt3d_device_ptrs()
    c = engine.mt3d_clip((1.0, 0.0, 0.0), -100.0, "high")
    assert (c.n_verts, c.n_tris, c.n_new_verts, c.n_cut_tris, c.n_dropped_tris) == (len(pre["verts"]), len(pre["tris"]),
                                                                                   0, 0, 0)
    post = engine.mt3d_fetch()
    for k in ("verts", "normals", "tris", "keys", "lowmin"):
        assert np.array_equal(pre[k], post[k]), k
    assert engine.mt3d_device_ptrs() == ptrs
    engine.mt3d_cap("high")                                        # no state changed: the cap is still accepted
    engine.mt3d_run(field, 0.5, flags=_flags(False))
    c = engine.mt3d_clip((1.0, 0.0, 0.0), -100.0, "low")
    assert (c.n_verts, c.n_tris, c.n_dropped_tris) == (0, 0, len(pre["tris"]))
    engine.mt3d_components()
    engine.mt3d_smooth(2)
    engine.mt3d_decimate(2.0)
    engine.mt3d_section((0.0, 0.0, 1.0), [1.0])
    engine.mt3d_orient_reference()
    engine.mt3d_interpolate(field)
    assert engine.mt3d_fetch()["verts"].shape == (0, 3)


def _from_device(ptr, shape, typestr, host=True):
    "an array at a raw device address, as a torch tensor on the device or copied to the host"
    import torch

    class Dev(object):
        pass
    d = Dev()
    d.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, data=(ptr, False), version=2)
    x = torch.as_tensor(d, device="cuda")
    return x.cpu().numpy() if host else x


def test_growth_and_device_pointers(engine):
    "a value clip on a checkerboard of the vertex ids cuts most triangles and grows the mesh; pointers taken again"
    import torch
    from oracle import mt3d_clip
    field = sphere_field(17)
    engine.mt3d_run(field, 0.5, flags=_flags(False))
    engine.mt3d_interpolate(field)
    pre = engine.mt3d_fetch()
    vals = np.where(np.arange(len(pre["verts"])) % 2 == 0, 1.0, -1.0).astype(np.float32)
    # the checkerboard written over the engine's vertex values through their device pointer
    dst = _from_device(engine.mt3d_interpolate_device_ptr(), (len(vals),), "<f4", host=False)
    dst.copy_(torch.as_tensor(vals, device="cuda"))
    torch.cuda.synchronize()
    want, wc = mt3d_clip.clip(pre["verts"], pre["tris"], normals=pre["normals"], keys=pre["keys"], lowmin=pre["lowmin"],
                              values=vals, component=0, offset=0.0, side="high", geom_dtype=np.float32)
    c = engine.mt3d_clip(component=0, offset=0.0, keep="high")
    assert c.n_tris == wc["n_tris"] > len(pre["tris"]) and c.n_verts == wc["n_verts"]
    post = engine.mt3d_fetch()
    for k in ("verts", "normals", "tris", "keys", "lowmin"):
        assert np.array_equal(post[k], np.asarray(want[k]).reshape(post[k].shape)), k
    assert np.array_equal(values_of(engine, 1)[:, 0], want["values"])
    v, n, t = engine.mt3d_device_ptrs()
    V, T = c.n_verts, c.n_tris
    assert np.array_equal(_from_device(v, (V, 3), "<f4"), post["verts"])
    assert np.array_equal(_from_device(n, (V, 3), "<f4"), post["normals"])
    assert np.array_equal(_from_device(t, (T, 3), "<i4"), post["tris"])
    assert np.array_equal(_from_device(engine.mt3d_interpolate_device_ptr(), (V,), "<f4"), want["values"])


# ---------------------------------------------------------------------------------------------- 3. errors and pass order
def _call(engine, source=0, side=0, normal=(1.0, 0.0, 0.0), offset=0.0, component=0, reserved=0, p=True, out=True):
    E = _E()
    cp = E.ClipParams()
    cp.source, cp.side, cp.offset, cp.component, cp.reserved = source, side, offset, component, reserved
    for a in range(3):
        cp.normal[a] = normal[a]
    cnt = E.ClipCounts()
    return engine.lib.ctr_mt3d_clip(engine.h, ctypes.byref(cp) if p else None, ctypes.byref(cnt) if out else None)


def test_errors_leave_the_mesh(engine):
    E = _E()
    assert engine.lib.ctr_mt3d_clip(None, None, None) == ERR_BAD_ARG
    fresh = E.Engine(0)
    try:
        assert _call(fresh) == ERR_STATE                            # no run
    finally:
        fresh.close()
    field = sphere_field(17)
    flags = _flags(False)

    def same(pre):
        post = engine.mt3d_fetch()
        for k in ("verts", "normals", "tris", "keys", "lowmin"):
            assert np.array_equal(pre[k], post[k]), k

    engine.mt3d_run(field, 0.5, flags=flags)
    pre = engine.mt3d_fetch()
    bad = [dict(p=False), dict(out=False), dict(source=2), dict(side=2), dict(side=-1), dict(normal=(0.0, 0.0, 0.0)),
           dict(normal=(np.inf, 0.0, 0.0)), dict(normal=(np.nan, 1.0, 0.0)), dict(offset=np.inf), dict(offset=np.nan),
           dict(component=1), dict(reserved=1), dict(source=1, normal=(1.0, 0.0, 0.0)), dict(source=1, component=-1)]
    for kw in bad:
        assert _call(engine, **kw) == ERR_BAD_ARG, kw
    same(pre)
    assert _call(engine, source=1, normal=(0.0, 0.0, 0.0)) == ERR_STATE        # no interpolation
    engine.mt3d_interpolate(field)
    assert _call(engine, source=1, normal=(0.0, 0.0, 0.0), component=1) == ERR_BAD_ARG
    nanf = field.copy()
    nanf[:, :, 8:] = np.nan
    engine.mt3d_interpolate(nanf)
    assert _call(engine, source=1, normal=(0.0, 0.0, 0.0), offset=0.5) == ERR_BAD_ARG    # a NaN side value
    same(pre)
    engine.mt3d_smooth(1)                                          # values of an older mesh generation
    pre = engine.mt3d_fetch()
    assert _call(engine, source=1, normal=(0.0, 0.0, 0.0), offset=0.5) == ERR_STATE
    same(pre)
    for kw in (dict(flags=E.NO_GEOMETRY), dict(flags=flags, i_lo=0, i_hi=8), dict(flags=flags, vert_id_base=7)):
        engine.mt3d_run(field, 0.5, **kw)
        assert _call(engine, offset=8.0) == ERR_STATE, kw
    engine.mt3d_run(field, 0.5, flags=flags)
    engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, 1 << 20), "ctr_mt3d_offset_ids")
    pre = engine.mt3d_fetch()
    assert _call(engine, offset=8.0) == ERR_STATE
    same(pre)
    with pytest.raises(ValueError):
        engine.mt3d_clip()
    with pytest.raises(ValueError):
        engine.mt3d_clip((1.0, 0.0, 0.0), component=0)
    with pytest.raises(ValueError):
        engine.mt3d_clip((1.0, 0.0, 0.0), keep="both")


def test_abi():
    E = _E()
    assert hasattr(E.load_library(), "ctr_mt3d_clip")
    assert ctypes.sizeof(E.ClipParams) == 48 and ctypes.sizeof(E.ClipCounts) == 40


N = 17
SHAPE = np.array([N - 1] * 3)
PASSES = {
    "orient": lambda e, f: e.mt3d_orient_reference(),
    "components": lambda e, f: e.mt3d_components(),
    "keep": lambda e, f: e.mt3d_keep_components(np.ones(len(e.mt3d_components()[1]), bool)),
    "smooth": lambda e, f: e.mt3d_smooth(2),
    "section": lambda e, f: e.mt3d_section((0.0, 0.0, 1.0), [8.0]),
    "decimate": lambda e, f: e.mt3d_decimate(2.0),
    "select": lambda e, f: e.mt3d_select_seeded(np.array([[8, 8, 3]], np.int32)),
    "clean": lambda e, f: e.mt3d_clean(SHAPE),
    "cap": lambda e, f: e.mt3d_cap("high"),
    "interpolate": lambda e, f: e.mt3d_interpolate(f),
    "clip": lambda e, f: e.mt3d_clip((0.3, 0.0, 1.0), 10.0, "low"),
}
BEFORE_ORDER = ["run", "select", "clean", "keep", "smooth", "decimate", "cap", "orient", "clip", "interpolate", "section",
                "components"]


def _code(fn):
    E = _E()
    try:
        fn()
    except (E.EngineError, ValueError) as e:
        m = re.search(r"failed \((-?\d+)\)", str(e))
        return int(m.group(1)) if m else -1
    return 0


def _pass_field():
    g = np.linspace(-1.0, 1.0, N)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    return X * X + Y * Y + 1.3 * Z * Z


@pytest.mark.parametrize("before", BEFORE_ORDER)
def test_clip_accepted_after(engine, before):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    if before != "run":
        PASSES[before](engine, f)
    assert _code(lambda: PASSES["clip"](engine, f)) == 0, engine.lib.ctr_last_error(engine.h).decode()


def test_clip_refused_on_slab_and_shifted_ids(engine):
    f = _pass_field()
    for setup in ("slab", "offset_ids"):
        engine.mt3d_run(f, 0.5, flags=_flags(False), i_hi=N // 2 if setup == "slab" else None)
        if setup == "offset_ids":
            engine._check(engine.lib.ctr_mt3d_offset_ids(engine.h, 7), "ctr_mt3d_offset_ids")
        pre = engine.mt3d_fetch()
        assert _code(lambda: PASSES["clip"](engine, f)) == ERR_STATE, setup
        post = engine.mt3d_fetch()
        for k in pre:
            assert np.array_equal(pre[k], post[k]), (setup, k)


@pytest.mark.parametrize("name", [p for p in PASSES if p != "clip"])
def test_passes_after_clip(engine, name):
    f = _pass_field()
    engine.mt3d_run(f, 0.5, flags=_flags(False))
    PASSES["clip"](engine, f)
    pre = engine.mt3d_fetch()
    want = ERR_STATE if name in ("select", "clean", "cap") else 0
    got = _code(lambda: PASSES[name](engine, f))
    assert got == want, (name, got, engine.lib.ctr_last_error(engine.h).decode())
    if want:
        assert "clipped" in engine.lib.ctr_last_error(engine.h).decode()
        post = engine.mt3d_fetch()
        for k in pre:
            assert np.array_equal(pre[k], post[k]), (name, k)


# ---------------------------------------------------------------------------------------------- 4. façade
def test_facade_halfspaces_equal_engine_calls(engine):
    from contourist_b200 import tetrahedral
    f = lambda x, y, z: np.minimum((x - 0.3) ** 2 + y * y + z * z, (x + 0.5) ** 2 + y * y + (z - 0.6) ** 2 + 0.05)
    A = np.array([[1.0, 0.0, 0.0], [0.0, -1.0, 0.5], [0.2, 0.3, 1.0]])
    b = np.array([0.5, 0.4, 0.3])

    def make(clip):
        t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.0625,) * 3, f, 0.3, [])
        t.post_process = False
        t.want_normals = True
        t.clip_halfspaces = clip
        t.measure_components = True
        t.search_for_endpoints()
        return t

    plain = make(None)
    plain.get_points_and_triangles()
    for a, d in zip(A, b):
        engine.mt3d_clip(normal=a, offset=d, keep="low")
    want = engine.mt3d_fetch()
    _, want_tab = engine.mt3d_components()
    t = make((A, b))
    p, tr = t.get_points_and_triangles()
    assert np.array_equal(p, want["verts"]) and np.array_equal(tr, want["tris"])
    got_tab = t.component_table
    for k in ("n_tris", "n_verts", "n_edges", "n_boundary_edges", "n_nonmanifold_edges", "first_tri", "lo", "hi"):
        assert np.array_equal(got_tab[k], want_tab[k]), k
    for k in ("area", "volume"):                                # fp64 sums in an unspecified order
        np.testing.assert_allclose(got_tab[k], want_tab[k], rtol=1e-12, atol=1e-12)
    assert ((p.astype(np.float64) @ A.T) < b).all(axis=1).sum() > 0
