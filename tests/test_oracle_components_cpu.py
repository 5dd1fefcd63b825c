"""CPU: oracle/mt3d_components.py:components (the definition of ctr_mt3d_components) on analytic meshes, the layout of
ctr_mt3d_component, the new C ABI symbols and the façade's measure_components plumbing (no GPU here)."""
import ctypes

import numpy as np
import pytest

from oracle import mt3d, mt3d_components

N = 64


def wound_mesh(field, value):
    """oracle/mt3d.extract's mesh with every triangle wound like the engine's: cross(b - a, c - a) towards the high
    side of the field (the gradient normals at its corners)."""
    r = mt3d.extract(field, value)
    P, t = r["pos"], r["tris"].astype(np.int64).copy()
    g = mt3d.normals(field, value, r["keys"])
    fn = np.cross(P[t[:, 1]] - P[t[:, 0]], P[t[:, 2]] - P[t[:, 0]])
    flip = (fn * (g[t[:, 0]] + g[t[:, 1]] + g[t[:, 2]])).sum(axis=1) < 0
    t[flip] = t[flip][:, ::-1]
    return P, t


def grid(n=N):
    x = np.arange(n + 1, dtype=np.float64)
    return np.meshgrid(x, x, x, indexing="ij")


def chi(row):
    return int(row["n_verts"]) - int(row["n_edges"]) + int(row["n_tris"])


def sphere_field(c, r):
    X, Y, Z = grid()
    return (X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2 - r * r


def test_sphere_area_volume_and_sign():
    r = 0.35 * N
    f = sphere_field((N / 2,) * 3, r)
    P, t = wound_mesh(f, 0.0)
    lab, tab = mt3d_components.components(P, t)
    assert len(tab) == 1 and (lab == 0).all()
    c = tab[0]
    assert c["n_tris"] == len(t) and c["first_tri"] == 0 and c["n_verts"] == len(P)
    assert c["n_boundary_edges"] == 0 and c["n_nonmanifold_edges"] == 0 and chi(c) == 2
    assert abs(c["area"] / (4 * np.pi * r * r) - 1) < 5e-3
    assert c["volume"] > 0 and abs(c["volume"] / (4 / 3 * np.pi * r ** 3) - 1) < 5e-3
    assert np.array_equal(c["lo"], P.min(axis=0)) and np.array_equal(c["hi"], P.max(axis=0))
    # the inside high: every triangle faces the other way
    Pn, tn = wound_mesh(-f, 0.0)
    _, tabn = mt3d_components.components(Pn, tn)
    assert np.isclose(tabn[0]["volume"], -c["volume"], rtol=1e-12) and np.isclose(tabn[0]["area"], c["area"], rtol=1e-12)


def test_torus():
    R, rr = 0.25 * N, 0.1 * N
    X, Y, Z = grid()
    X, Y, Z = X - N / 2, Y - N / 2, Z - N / 2
    f = (np.sqrt(X * X + Y * Y) - R) ** 2 + Z * Z - rr * rr
    P, t = wound_mesh(f, 0.0)
    _, tab = mt3d_components.components(P, t)
    assert len(tab) == 1
    c = tab[0]
    assert chi(c) == 0 and c["n_boundary_edges"] == 0 and c["n_nonmanifold_edges"] == 0
    assert abs(c["area"] / (4 * np.pi ** 2 * R * rr) - 1) < 5e-3
    assert c["volume"] > 0 and abs(c["volume"] / (2 * np.pi ** 2 * R * rr * rr) - 1) < 1.5e-2


def test_two_spheres_numbered_by_first_triangle():
    X, Y, Z = grid()
    big, small = (40.0, 32.0, 32.0, 14.0), (14.0, 32.0, 32.0, 8.0)
    f = np.minimum(*[(X - s[0]) ** 2 + (Y - s[1]) ** 2 + (Z - s[2]) ** 2 - s[3] ** 2 for s in (big, small)])
    P, t = wound_mesh(f, 0.0)
    lab, tab = mt3d_components.components(P, t)
    assert len(tab) == 2
    assert tab["first_tri"][0] == 0 and tab["first_tri"][0] < tab["first_tri"][1]
    for k in range(2):
        assert lab[tab["first_tri"][k]] == k and (lab[: tab["first_tri"][k]] != k).all()
        assert chi(tab[k]) == 2 and tab[k]["n_boundary_edges"] == 0 and tab[k]["volume"] > 0
    assert np.array_equal(np.bincount(lab), tab["n_tris"])
    # the sphere around x = 14 comes first in the engine's x order; check sizes against the radii whatever the order
    rad = sorted((tab["area"] / (4 * np.pi)) ** 0.5)
    assert abs(rad[0] / 8 - 1) < 1e-2 and abs(rad[1] / 14 - 1) < 1e-2


def test_plane_cut_by_the_box_is_a_disc():
    X, Y, Z = grid(16)
    f = X + 0.5 * Y + 0.25 * Z
    P, t = wound_mesh(f, 9.3)
    _, tab = mt3d_components.components(P, t)
    assert len(tab) == 1 and tab[0]["n_boundary_edges"] > 0 and chi(tab[0]) == 1
    assert tab[0]["n_nonmanifold_edges"] == 0


def test_permuting_triangles_keeps_the_partition():
    X, Y, Z = grid(24)
    f = np.minimum((X - 6) ** 2 + (Y - 12) ** 2 + (Z - 12) ** 2 - 16, (X - 17) ** 2 + (Y - 12) ** 2 + (Z - 12) ** 2 - 20)
    P, t = wound_mesh(f, 0.0)
    lab, tab = mt3d_components.components(P, t)
    perm = np.random.default_rng(3).permutation(len(t))
    lab2, tab2 = mt3d_components.components(P, t[perm])
    assert len(tab2) == len(tab) == 2
    # same partition: a bijection between the labels
    pairs = np.unique(np.stack([lab[perm], lab2], 1), axis=0)
    assert len(pairs) == len(tab)
    m = dict(map(tuple, pairs))
    for k in range(len(tab)):
        a, b = tab[k], tab2[m[k]]
        for f_ in ("n_tris", "n_verts", "n_edges", "n_boundary_edges", "n_nonmanifold_edges"):
            assert a[f_] == b[f_]
        assert np.array_equal(a["lo"], b["lo"]) and np.array_equal(a["hi"], b["hi"])
        assert np.isclose(a["area"], b["area"], rtol=1e-12) and np.isclose(a["volume"], b["volume"], rtol=1e-12)
    assert (tab2["first_tri"] == np.sort(tab2["first_tri"])).all()


def test_vertex_touching_sheets_stay_apart_and_edge_counts():
    # two triangles sharing vertex 0 only; a fan of three triangles on one edge (non-manifold)
    P = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]], np.float64)
    lab, tab = mt3d_components.components(P, np.array([[0, 1, 2], [0, 3, 4]]))
    assert len(tab) == 2 and list(lab) == [0, 1] and list(tab["n_verts"]) == [3, 3]
    P = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1]], np.float64)
    lab, tab = mt3d_components.components(P, np.array([[0, 1, 2], [1, 0, 3], [0, 1, 4]]))
    assert len(tab) == 1 and tab[0]["n_edges"] == 7 and tab[0]["n_nonmanifold_edges"] == 1
    assert tab[0]["n_boundary_edges"] == 6 and tab[0]["n_verts"] == 5
    lab, tab = mt3d_components.components(P, np.zeros((0, 3), np.int32))
    assert len(lab) == 0 and len(tab) == 0


class CComponent(ctypes.Structure):
    _fields_ = [("n_tris", ctypes.c_int64), ("n_verts", ctypes.c_int64), ("n_edges", ctypes.c_int64),
                ("n_boundary_edges", ctypes.c_int64), ("n_nonmanifold_edges", ctypes.c_int64),
                ("first_tri", ctypes.c_int64), ("area", ctypes.c_double), ("volume", ctypes.c_double),
                ("lo", ctypes.c_double * 3), ("hi", ctypes.c_double * 3)]


def test_component_dtype_mirrors_the_header_struct():
    from contourist_b200 import engine
    dt = engine.COMPONENT_DTYPE
    assert dt.itemsize == ctypes.sizeof(CComponent) == 112
    for name, _ in CComponent._fields_:
        assert dt.fields[name][1] == getattr(CComponent, name).offset, name
    assert dt == mt3d_components.COMPONENT_DTYPE


def test_new_symbols_declared_and_exported():
    from test_capi_symbols import declared_symbols
    from contourist_b200 import build, engine
    syms = declared_symbols()
    for s in ("ctr_mt3d_components", "ctr_mt3d_components_fetch"):
        assert s in syms
    build.build()
    lib = engine.load_library()
    assert lib.ctr_mt3d_components(None, None) == -1       # null context, no CUDA touched
    assert lib.ctr_mt3d_components_fetch(None, None, None) == -1


class StubEngine(object):
    """Records the calls get_points_and_triangles makes; returns a two-triangle mesh."""

    def __init__(self):
        self.calls = []
        self.run_serial = 0

    def mt3d_run(self, field, value, origin, delta, flags):
        self.calls.append("run")
        return None

    def mt3d_clean(self, corner, **kw):
        self.calls.append("clean")

        class C(object):
            n_components, n_flipped = 1, 0
        return C()

    def mt3d_orient_reference(self):
        self.calls.append("orient")
        return 1, 0

    def mt3d_components(self):
        self.calls.append("components")
        tab = np.zeros(1, mt3d_components.COMPONENT_DTYPE)
        tab["n_tris"] = 2
        return np.zeros(2, np.int32), tab

    def mt3d_fetch(self):
        self.calls.append("fetch")
        return dict(verts=np.zeros((4, 3), np.float32), normals=None, tris=np.array([[0, 1, 2], [0, 2, 3]], np.int32))


@pytest.mark.parametrize("post_process", [True, False])
def test_facade_measures_components_after_the_last_edit(monkeypatch, post_process):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    stub = StubEngine()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    f = lambda x, y, z: x * x + y * y + z * z
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.5, 0.5, 0.5), f, 0.5, [])
    t.post_process = post_process
    t.reference_orientation = True
    t.measure_components = True
    points, tris = t.get_points_and_triangles()
    assert stub.calls[-2:] == ["components", "fetch"]
    assert ("clean" if post_process else "orient") in stub.calls[:-2]
    assert len(t.triangle_components) == len(tris) and t.component_table["n_tris"][0] == 2
    # unset: no pass, nothing left behind
    stub.calls = []
    t2 = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.5, 0.5, 0.5), f, 0.5, [])
    t2.post_process = post_process
    t2.get_points_and_triangles()
    assert "components" not in stub.calls and t2.triangle_components is None and t2.component_table is None
    assert tetrahedral.GridContour3d.measure_components is False
