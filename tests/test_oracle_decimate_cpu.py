"""CPU: oracle/mt3d_decimate.py (the definition of ctr_mt3d_decimate) on hand-made meshes and on an extracted sphere,
the new C ABI symbol and the façade's decimate_cell plumbing (no GPU here)."""
import ctypes

import numpy as np
import pytest

from oracle import mt3d_components, mt3d_decimate
from test_oracle_components_cpu import wound_mesh
from test_oracle_filter_cpu import StubEngine, _make


def naive(verts, tris, cell, origin):
    """The definition written out cluster by cluster with a library solve, as a check on the vectorised oracle:
    (positions in float64 by member, tris, member)."""
    P = np.asarray(verts, np.float64)
    cell, origin = np.broadcast_to(np.asarray(cell, np.float64), (3,)), np.broadcast_to(np.asarray(origin, np.float64), (3,))
    q = [tuple(np.floor((p - origin) / cell).astype(int)) for p in P]
    lo = {k: origin + np.array(k) * cell for k in q}
    members = {}
    for v, k in enumerate(q):
        members.setdefault(k, []).append(v)
    A = {k: np.zeros((3, 3)) for k in members}
    g = {k: np.zeros(3) for k in members}
    for a, b, c in np.asarray(tris).tolist():
        n = np.cross(P[b] - P[a], P[c] - P[a])
        for v in (a, b, c):
            k = q[v]
            d = -np.dot(n, P[a] - lo[k])
            A[k] += np.outer(n, n)
            g[k] += d * n
    pos = {}
    for k, vs in members.items():
        m = np.mean([P[v] - lo[k] for v in vs], axis=0)
        lam = 1e-3 * np.trace(A[k])
        x = m if lam == 0 else np.linalg.solve(A[k] + lam * np.eye(3), lam * m - g[k])
        pos[min(vs)] = lo[k] + np.clip(x, 0, cell)
    rep = [min(members[k]) for k in q]
    kept, seen = [], set()
    for t in np.asarray(tris).tolist():
        r = [rep[v] for v in t]
        if len(set(r)) < 3 or frozenset(r) in seen:
            continue
        seen.add(frozenset(r))
        kept.append(r)
    member = sorted({v for t in kept for v in t})
    idx = {v: i for i, v in enumerate(member)}
    return (np.array([pos[v] for v in member]).reshape(-1, 3), np.array([[idx[v] for v in t] for t in kept]).reshape(-1, 3),
            np.array(member, np.int64), len(members))


def plane_grid(n, slope=(0.3, -0.2), offset=0.1):
    """an n x n grid of points on z = sx * x + sy * y + offset, two triangles per square"""
    ii, jj = np.meshgrid(np.arange(n, dtype=np.float64), np.arange(n, dtype=np.float64), indexing="ij")
    P = np.stack([ii.ravel(), jj.ravel(), slope[0] * ii.ravel() + slope[1] * jj.ravel() + offset], axis=1)
    T = []
    for i in range(n - 1):
        for j in range(n - 1):
            a, b, c, d = i * n + j, (i + 1) * n + j, (i + 1) * n + j + 1, i * n + j + 1
            T += [[a, b, c], [a, c, d]]
    return P, np.array(T, np.int32)


def cube_surface(k):
    """the surface of [0, 1]^3 with every face cut into k x k squares (shared vertices, outward winding)"""
    ids, P, T = {}, [], []

    def vid(p):
        key = tuple(int(round(x * k)) for x in p)
        if key not in ids:
            ids[key] = len(P)
            P.append(np.array(key, np.float64) / k)
        return ids[key]
    for ax in range(3):
        for side in (0, 1):
            u, w = [a for a in range(3) if a != ax]
            for i in range(k):
                for j in range(k):
                    quad = []
                    for di, dj in ((0, 0), (1, 0), (1, 1), (0, 1)):
                        p = np.zeros(3)
                        p[ax], p[u], p[w] = side, (i + di) / k, (j + dj) / k
                        quad.append(vid(p))
                    a, b, c, d = quad
                    tri = [[a, b, c], [a, c, d]]
                    n = np.zeros(3)
                    n[ax] = 1 if side else -1
                    for t in tri:
                        e = np.cross(P[t[1]] - P[t[0]], P[t[2]] - P[t[0]])
                        T.append(t if np.dot(e, n) > 0 else t[::-1])
    return np.array(P), np.array(T, np.int32)


def test_planar_grid_stays_on_its_plane_and_matches_the_naive_definition():
    P, T = plane_grid(12)
    for cell, origin in ((2.5, (0.3, -0.1, 0.0)), ((3.0, 1.7, 0.9), (-0.5, 0.2, -1.0))):
        V, t, member, c = mt3d_decimate.decimate(P, T, cell, origin)
        assert 0 < c["n_tris"] < len(T) and c["n_collapsed"] > 0
        # on its plane to rounding: the regularised 3 x 3 system has a condition number of about 1 / 1e-3 on a flat
        # cluster, so the residual is about 1e3 fp64 roundings of the cell size
        tol = 2e-12 * np.max(cell)
        assert np.abs(V[:, 2] - (0.3 * V[:, 0] - 0.2 * V[:, 1] + 0.1)).max() < tol
        W, tw, mw, nc = naive(P, T, cell, origin)
        assert np.array_equal(t, tw) and np.array_equal(member, mw) and c["n_clusters"] == nc
        assert np.abs(V - W).max() < tol


def test_cube_corner_inside_a_cell_is_kept_where_the_mean_cuts_it():
    P, T = cube_surface(10)
    cell, origin = 0.3, (0.15, 0.15, 0.15)                 # the corner (1, 1, 1) lies inside cell [0.75, 1.05)^3
    V, t, member, c = mt3d_decimate.decimate(P, T, cell, origin)
    corner = np.argmin(np.linalg.norm(V - 1.0, axis=1))
    err = np.linalg.norm(V[corner] - 1.0)
    # the members of the corner's cluster and their mean: the mean lies inside the cube, cutting the corner
    q, _ = mt3d_decimate.cells(P, cell, origin)
    inside = (q == q[member[corner]]).all(axis=1)
    cut = np.linalg.norm(P[inside].mean(axis=0) - 1.0)
    # the regularisation pulls the solution towards the mean by lambda / (w + lambda) per axis, with w = trace / 3 on
    # this symmetric corner: 3e-3 of the mean's distance (4.1e-4 against 0.137 here)
    assert (q[inside] == q[member[corner]]).all() and inside.sum() == 19
    assert cut > 0.1 and err < 3.4e-3 * cut and err < 5e-4
    assert np.abs(V - naive(P, T, cell, origin)[0]).max() < 2e-12 * cell
    # the corner vertex of the mesh itself is the only member: then the corner is kept exactly
    V, _, _, _ = mt3d_decimate.decimate(P, T, 0.3, (0.05, 0.05, 0.05))     # cell [0.95, 1.25)^3
    assert np.abs(V - 1.0).sum(axis=1).min() < 1e-12


def test_small_cells_leave_the_mesh_as_it_is():
    P, T = cube_surface(4)
    P = P + np.random.default_rng(2).uniform(-0.02, 0.02, P.shape)
    V, t, member, c = mt3d_decimate.decimate(P, T, 0.01, (-0.3, -0.3, -0.3))
    assert np.array_equal(t, T) and np.array_equal(member, np.arange(len(P)))
    assert c == dict(n_verts=len(P), n_tris=len(T), n_clusters=len(P), n_collapsed=0, n_duplicate=0)
    assert np.abs(V - P).max() < 1e-12
    V32, _, _, _ = mt3d_decimate.decimate(P.astype(np.float32), T, 0.01, (-0.3, -0.3, -0.3))
    assert V32.dtype == np.float32 and np.abs(V32 - P.astype(np.float32)).max() <= 1e-7


def test_every_vertex_lies_in_its_cluster_box():
    P, T = wound_mesh(sphere_field(24, 8.3), 0.0)
    for cell, origin in ((2.0, (0.0, 0.0, 0.0)), ((1.5, 2.5, 3.0), (0.7, -0.2, 0.4))):
        V, t, member, _ = mt3d_decimate.decimate(P, T, cell, origin)
        _, lo = mt3d_decimate.cells(P[member], cell, origin)
        assert (V >= lo).all() and (V <= lo + np.asarray(cell)).all()


def test_collapsed_and_duplicate_triangles():
    P = np.array([[0.1, 0.1, 0.0], [1.1, 0.1, 0.0], [0.1, 1.1, 0.0], [0.2, 0.2, 0.0], [1.2, 1.2, 0.0], [0.3, 0.1, 0.0],
                  [5.5, 5.5, 0.0]], np.float64)
    # clusters with cell 1: {0, 3, 5} {1} {2} {4} {6}
    T = np.array([[0, 1, 2],          # kept
                  [3, 1, 2],          # same three clusters: duplicate
                  [2, 1, 5],          # the other winding: duplicate
                  [0, 3, 1],          # two corners in one cluster: collapsed
                  [0, 3, 5],          # all three: collapsed
                  [1, 4, 2],          # kept
                  [3, 4, 1]], np.int32)   # its own triple {0, 4, 1}: kept
    V, t, member, c = mt3d_decimate.decimate(P, T, 1.0)
    assert c == dict(n_verts=4, n_tris=3, n_clusters=5, n_collapsed=2, n_duplicate=2)
    assert list(member) == [0, 1, 2, 4]                       # vertex 6 (no kept triangle) goes
    assert t.tolist() == [[0, 1, 2], [1, 3, 2], [0, 3, 1]]    # order and corner order kept
    W, tw, mw, nc = naive(P, T, 1.0, 0.0)
    assert np.array_equal(t, tw) and np.array_equal(member, mw) and nc == 5 and np.abs(V - W).max() < 1e-12


def test_empty_input_and_range():
    V, t, member, c = mt3d_decimate.decimate(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), 1.0)
    assert V.shape == (0, 3) and V.dtype == np.float32 and t.shape == (0, 3) and len(member) == 0
    assert c == dict(n_verts=0, n_tris=0, n_clusters=0, n_collapsed=0, n_duplicate=0)
    P, T = plane_grid(3)
    V, t, member, c = mt3d_decimate.decimate(P, np.zeros((0, 3), np.int32), 1.0)   # vertices but no triangles
    assert len(V) == 0 and c["n_clusters"] == len(P)
    mt3d_decimate.decimate(P, T, 1.0, (2.0 ** 20, 0.0, 0.0))                      # q = -2^20 at x = 0: in range
    for origin in ((2.0 ** 20 + 1, 0.0, 0.0), (0.0, -(2.0 ** 20) - 1, 0.0)):
        with pytest.raises(ValueError):
            mt3d_decimate.decimate(P, T, 1.0, origin)


def sphere_field(n, r):
    x = np.arange(n, dtype=np.float64) - (n - 1) / 2.0
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return np.sqrt(X * X + Y * Y + Z * Z) - r


def test_extracted_sphere_fewer_triangles_volume_kept():
    P, T = wound_mesh(sphere_field(40, 14.3), 0.0)
    _, tab0 = mt3d_components.components(P, T)
    vol0 = tab0["volume"][0]
    prev = len(T)
    for cell in (1.5, 2.0, 3.0, 4.0):
        V, t, _, c = mt3d_decimate.decimate(P, T, cell)
        assert c["n_tris"] < prev
        prev = c["n_tris"]
        _, tab = mt3d_components.components(V, t)
        assert len(tab) == 1
        rel = abs(tab["volume"][0] / vol0 - 1)
        if cell == 2.0:
            # this definition at a 2-voxel cell: 22 968 -> 1 920 triangles, still closed, enclosed volume -0.34 %
            # (1.5 voxels: -0.15 %; 3: -1.2 %; 4: -1.5 %)
            assert c["n_tris"] == 1920 and tab["n_boundary_edges"][0] == 0 and rel < 5e-3
        assert rel < 2e-2


def test_new_symbol_declared_exported_and_struct_layout():
    from test_capi_symbols import declared_symbols
    from contourist_b200 import build, engine
    assert "ctr_mt3d_decimate" in declared_symbols()
    assert ctypes.sizeof(engine.DecimateParams) == 48 and ctypes.sizeof(engine.DecimateCounts) == 40
    build.build()
    lib = engine.load_library()
    assert lib.ctr_mt3d_decimate(None, None, None) == -1           # null context, no CUDA touched


class DecimateStub(StubEngine):
    def __init__(self):
        StubEngine.__init__(self)
        self.decimated = None

    def mt3d_smooth(self, iterations, lam, mu):
        self.calls.append("smooth")

    def mt3d_decimate(self, cell, origin):
        self.calls.append("decimate")
        self.decimated = (tuple(cell), tuple(origin))


@pytest.mark.parametrize("post_process", [True, False])
def test_facade_decimates_after_smoothing_and_measures_again(monkeypatch, post_process):
    from contourist_b200 import engine as E
    stub = DecimateStub()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    t = _make(post_process, keep_components=1, measure_components=True, vertex_fields=lambda x, y, z: x,
              smooth_iterations=2, decimate_cell=2)
    t.get_points_and_triangles()
    edit = "clean" if post_process else "orient"
    assert stub.calls == ["run", edit, "components", "keep", "smooth", "decimate", "interpolate", "components", "fetch"]
    # cells of 2 voxels of the world grid (delta 0.5 from -1): aligned with the grid points
    assert stub.decimated == ((1.0, 1.0, 1.0), (-1.0, -1.0, -1.0))
    stub.calls = []
    _make(post_process, keep_components=1, measure_components=True, decimate_cell=(1, 2, 3)).get_points_and_triangles()
    assert stub.calls == ["run", edit, "components", "keep", "decimate", "components", "fetch"]
    assert stub.decimated == ((0.5, 1.0, 1.5), (-1.0, -1.0, -1.0))


def test_facade_default_does_not_decimate_and_flatten_still_raises(monkeypatch):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    stub = DecimateStub()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    _make(True, keep_components=1, measure_components=True).get_points_and_triangles()
    assert "decimate" not in stub.calls and stub.calls[-2] == "components_fetch"
    assert tetrahedral.GridContour3d.decimate_cell is None
    f = lambda x, y, z: x * x + y * y + z * z
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.5, 0.5, 0.5), f, 0.5, [], flatten=True)
    t.decimate_cell = 2
    with pytest.raises(NotImplementedError):
        t.get_points_and_triangles()
    assert "decimate" not in stub.calls
