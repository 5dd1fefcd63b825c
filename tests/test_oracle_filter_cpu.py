"""CPU: oracle/mt3d_filter.py:keep_components (the definition of ctr_mt3d_keep_components) on hand-made and extracted
meshes, the new C ABI symbol and the façade's keep_components plumbing (no GPU here)."""
import numpy as np
import pytest

from oracle import mt3d_components, mt3d_filter
from test_oracle_components_cpu import grid, wound_mesh

INT_FIELDS = ("n_tris", "n_verts", "n_edges", "n_boundary_edges", "n_nonmanifold_edges")


def sheets():
    # two triangles sharing only vertex 0 (two components), then a quad (two triangles, one component) apart
    P = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0],
                  [5, 5, 5], [6, 5, 5], [6, 6, 5], [5, 6, 5]], np.float64)
    T = np.array([[0, 1, 2], [5, 6, 7], [0, 3, 4], [5, 7, 8]], np.int32)
    return P, T


def test_vertex_touching_sheets_keep_the_shared_vertex():
    P, T = sheets()
    lab, tab = mt3d_components.components(P, T)
    assert list(lab) == [0, 1, 2, 1] and list(tab["first_tri"]) == [0, 1, 2]
    # drop the first sheet: vertex 0 stays for the other one, 1 and 2 go
    t, used, lab2, tab2 = mt3d_filter.keep_components(T, lab, tab, [False, True, True])
    assert list(used) == [0, 3, 4, 5, 6, 7, 8]
    assert np.array_equal(used[t], T[1:])
    assert list(lab2) == [0, 1, 0] and list(tab2["first_tri"]) == [0, 1]
    assert t.dtype == np.int32 and lab2.dtype == np.int32
    for f in INT_FIELDS + ("area", "volume", "lo", "hi"):
        assert np.array_equal(tab2[f], tab[1:][f]), f


def test_keep_all_is_the_identity_and_keep_none_is_empty():
    P, T = sheets()
    lab, tab = mt3d_components.components(P, T)
    t, used, lab2, tab2 = mt3d_filter.keep_components(T, lab, tab, np.ones(3, bool))
    assert np.array_equal(t, T) and np.array_equal(used, np.arange(len(P))) and np.array_equal(lab2, lab)
    assert tab2.tobytes() == tab.tobytes()
    t, used, lab2, tab2 = mt3d_filter.keep_components(T, lab, tab, np.zeros(3, bool))
    assert t.shape == (0, 3) and len(used) == 0 and len(lab2) == 0 and len(tab2) == 0
    t, used, lab2, tab2 = mt3d_filter.keep_components(np.zeros((0, 3), np.int32), np.zeros(0, np.int32),
                                                      np.zeros(0, mt3d_components.COMPONENT_DTYPE), np.zeros(0, bool))
    assert t.shape == (0, 3) and len(used) == 0 and len(tab2) == 0
    with pytest.raises(ValueError):
        mt3d_filter.keep_components(T, lab, tab, [True, False])


def test_numbering_and_first_tri_follow_the_compaction():
    P, T = sheets()
    lab, tab = mt3d_components.components(P, T)
    t, used, lab2, tab2 = mt3d_filter.keep_components(T, lab, tab, [True, False, True])
    assert list(lab2) == [0, 1] and list(tab2["first_tri"]) == [0, 1]
    assert np.array_equal(used[t], T[[0, 2]])
    for k in range(len(tab2)):
        assert lab2[tab2["first_tri"][k]] == k and (lab2[: tab2["first_tri"][k]] != k).all()


def blobs():
    X, Y, Z = grid(40)
    f = np.full(X.shape, 1.0)
    rng = np.random.default_rng(5)
    for _ in range(9):
        c = rng.uniform(-4, 44, 3)                       # some of them cut by the box
        r = rng.uniform(2.5, 7.0)
        f = np.minimum(f, ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) / (r * r))
    return wound_mesh(f, 0.8)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_filtered_mesh_measures_like_the_filter_of_its_components(seed):
    P, T = blobs()
    lab, tab = mt3d_components.components(P, T)
    assert len(tab) > 3
    keep = np.random.default_rng(seed).random(len(tab)) < 0.5
    t, used, lab2, tab2 = mt3d_filter.keep_components(T, lab, tab, keep)
    want_lab, want = mt3d_components.components(P[used], t)
    assert np.array_equal(lab2, want_lab) and len(tab2) == len(want) == keep.sum()
    for f in INT_FIELDS + ("first_tri", "lo", "hi"):
        assert np.array_equal(tab2[f], want[f]), f
    assert np.allclose(tab2["area"], want["area"], rtol=1e-12, atol=0)
    assert np.allclose(tab2["volume"], want["volume"], rtol=1e-9, atol=1e-9 * want["area"].max())
    # twice equals once by the composed mask
    keep2 = np.random.default_rng(seed + 10).random(len(tab2)) < 0.7
    t3, used3, lab3, tab3 = mt3d_filter.keep_components(t, lab2, tab2, keep2)
    both = keep.copy()
    both[np.flatnonzero(keep)[~keep2]] = False
    t4, used4, lab4, tab4 = mt3d_filter.keep_components(T, lab, tab, both)
    assert np.array_equal(t3, t4) and np.array_equal(used[used3], used4) and np.array_equal(lab3, lab4)
    assert tab3.tobytes() == tab4.tobytes()


def test_new_symbol_declared_and_exported():
    from test_capi_symbols import declared_symbols
    from contourist_b200 import build, engine
    assert "ctr_mt3d_keep_components" in declared_symbols()
    build.build()
    lib = engine.load_library()
    assert lib.ctr_mt3d_keep_components(None, None, 0, None, None) == -1    # null context, no CUDA touched


class StubEngine(object):
    """Records the calls get_points_and_triangles makes; a four-triangle mesh in three components."""

    def __init__(self):
        self.calls = []
        self.run_serial = 0
        self.kept = None

    def mt3d_run(self, field, value, origin, delta, flags):
        self.calls.append("run")
        return None

    def mt3d_clean(self, corner, **kw):
        self.calls.append("clean")

        class C(object):
            n_components, n_flipped = 3, 0
        return C()

    def mt3d_orient_reference(self):
        self.calls.append("orient")
        return 3, 0

    def mt3d_components(self):
        self.calls.append("components")
        tab = np.zeros(3, mt3d_components.COMPONENT_DTYPE)
        tab["n_tris"] = [1, 2, 1]
        tab["first_tri"] = [0, 1, 2]
        return np.array([0, 1, 2, 1], np.int32), tab

    def mt3d_keep_components(self, keep):
        self.calls.append("keep")
        self.kept = keep
        return 3, 2

    def mt3d_components_fetch(self):
        self.calls.append("components_fetch")
        tab = np.zeros(1, mt3d_components.COMPONENT_DTYPE)
        tab["n_tris"] = 2
        return np.zeros(2, np.int32), tab

    def mt3d_interpolate(self, field):
        self.calls.append("interpolate")
        return np.zeros(3)

    def mt3d_fetch(self):
        self.calls.append("fetch")
        return dict(verts=np.zeros((3, 3), np.float32), normals=None, tris=np.array([[0, 1, 2], [0, 2, 1]], np.int32))


def _make(post_process, **opts):
    from contourist_b200 import tetrahedral
    f = lambda x, y, z: x * x + y * y + z * z
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.5, 0.5, 0.5), f, 0.5, [])
    t.post_process = post_process
    t.reference_orientation = True
    for k, v in opts.items():
        setattr(t, k, v)
    return t


@pytest.mark.parametrize("post_process", [True, False])
def test_facade_filters_after_the_edits_and_before_values_and_measurement(monkeypatch, post_process):
    from contourist_b200 import engine as E
    stub = StubEngine()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    t = _make(post_process, keep_components=1, measure_components=True, vertex_fields=lambda x, y, z: x)
    points, tris = t.get_points_and_triangles()
    edit = "clean" if post_process else "orient"
    assert stub.calls == ["run", edit, "components", "keep", "interpolate", "components_fetch", "fetch"]
    assert list(stub.kept) == [1]                                   # the most triangles
    assert len(t.triangle_components) == len(tris) and t.component_table["n_tris"][0] == 2
    assert len(t.vertex_values) == len(points)


def test_facade_int_and_callable_rules(monkeypatch):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    stub = StubEngine()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    _make(True, keep_components=2).get_points_and_triangles()
    assert list(stub.kept) == [1, 0]                                # ties go to the smaller number
    _make(True, keep_components=0).get_points_and_triangles()
    assert len(stub.kept) == 0
    _make(True, keep_components=lambda tab: tab["n_tris"] == 1).get_points_and_triangles()
    assert list(stub.kept) == [True, False, True]
    seen = []
    _make(True, keep_components=lambda tab: seen.append(tab) or [2]).get_points_and_triangles()
    assert list(stub.kept) == [2] and list(seen[0]["n_tris"]) == [1, 2, 1]
    stub.calls = []
    _make(True, keep_components=1).get_points_and_triangles()   # without measure_components: no second fetch
    assert "components_fetch" not in stub.calls and stub.calls.count("components") == 1
    for bad in (-1, 1.5, True, "largest"):
        with pytest.raises((ValueError, TypeError)):
            tetrahedral.components_to_keep(np.zeros(2, mt3d_components.COMPONENT_DTYPE), bad)


def test_facade_option_unset_calls_nothing_new(monkeypatch):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    stub = StubEngine()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    _make(True).get_points_and_triangles()
    _make(False, measure_components=True).get_points_and_triangles()
    assert "keep" not in stub.calls and "components_fetch" not in stub.calls
    assert tetrahedral.GridContour3d.keep_components is None
