"""CPU: oracle/mt3d_smooth.py (the definition of ctr_mt3d_smooth) on hand-made meshes and on extracted binary balls,
the new C ABI symbol and the façade's smooth_iterations plumbing (no GPU here)."""
import ctypes

import numpy as np
import pytest

from oracle import mt3d, mt3d_components, mt3d_smooth
from test_oracle_filter_cpu import StubEngine, _make


def naive(verts, tris, iterations, lam, mu):
    """The definition written out vertex by vertex, as a check on the vectorised oracle."""
    x = np.asarray(verts).astype(np.float64)
    uses = {}
    for t in np.asarray(tris).tolist():
        for a, b in ((t[0], t[1]), (t[1], t[2]), (t[2], t[0])):
            if a != b:
                k = (min(a, b), max(a, b))
                uses[k] = uses.get(k, 0) + 1
    nb = {v: set() for v in range(len(x))}
    fixed = set(range(len(x)))
    for (a, b), u in uses.items():
        nb[a].add(b)
        nb[b].add(a)
        fixed.discard(a)
        fixed.discard(b)
    for (a, b), u in uses.items():
        if u != 2:
            fixed.update((a, b))
    for _ in range(iterations):
        for w in [lam] + ([mu] if mu != 0 else []):
            y = x.copy()
            for v in range(len(x)):
                if v in fixed:
                    continue
                ns = sorted(nb[v])
                s = x[ns[0]].copy()
                for n in ns[1:]:
                    s = s + x[n]
                y[v] = x[v] + w * (s / len(ns) - x[v])
            x = y
    return x.astype(np.asarray(verts).dtype), len(uses), len(fixed)


def octahedron(scale=1.0):
    P = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.float64) * scale
    T = np.array([[0, 2, 4], [2, 1, 4], [1, 3, 4], [3, 0, 4], [2, 0, 5], [1, 2, 5], [3, 1, 5], [0, 3, 5]], np.int32)
    return P, T


def grid_patch(n=6):
    ii, jj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    P = np.stack([ii.ravel(), jj.ravel(), np.zeros(n * n)], axis=1).astype(np.float64)
    T = []
    for i in range(n - 1):
        for j in range(n - 1):
            a, b, c, d = i * n + j, (i + 1) * n + j, (i + 1) * n + j + 1, i * n + j + 1
            T += [[a, b, c], [a, c, d]]                 # every cell cut along the same diagonal
    return P, np.array(T, np.int32)


def test_flat_regular_patch_stays_put_bit_for_bit():
    P, T = grid_patch(6)
    for dtype in (np.float64, np.float32):
        Q, c = mt3d_smooth.smooth(P.astype(dtype), T, 7, 0.5, -0.53)
        assert Q.dtype == dtype and np.array_equal(Q, P.astype(dtype))
        assert c == dict(n_edges=5 * 6 * 2 + 25, n_fixed_verts=20)       # the 4 * 5 border vertices


def test_single_triangle_and_open_strip_are_fixed():
    P = np.random.default_rng(1).random((3, 3))
    Q, c = mt3d_smooth.smooth(P, [[0, 1, 2]], 5, 0.5, -0.53)
    assert np.array_equal(Q, P) and c == dict(n_edges=3, n_fixed_verts=3)
    P = np.random.default_rng(2).random((8, 3))
    T = [[k, k + 1, k + 2] for k in range(6)]
    Q, c = mt3d_smooth.smooth(P, T, 5, 0.5, -0.53)
    assert np.array_equal(Q, P) and c == dict(n_edges=13, n_fixed_verts=8)


def test_closed_mesh_moves_and_matches_the_naive_definition():
    P, T = octahedron()
    P = P + np.random.default_rng(3).normal(0, 0.1, P.shape)
    for it, lam, mu in ((1, 0.5, -0.53), (4, 0.33, -0.34), (3, 1.0, 0.0), (2, 0.5, -1.0)):
        for dtype in (np.float64, np.float32):
            Q, c = mt3d_smooth.smooth(P.astype(dtype), T, it, lam, mu)
            W, ne, nf = naive(P.astype(dtype), T, it, lam, mu)
            assert Q.tobytes() == W.tobytes()
            assert c == dict(n_edges=ne, n_fixed_verts=nf) == dict(n_edges=12, n_fixed_verts=0)
            assert not np.array_equal(Q, P.astype(dtype))


def test_non_manifold_fan():
    P, T = octahedron()
    P = np.vstack([P + np.random.default_rng(4).normal(0, 0.1, P.shape), [[2.0, 2.0, 0.0]]])
    T = np.vstack([T, [[0, 2, 6]]])                    # a fin on edge {0, 2}: three uses
    Q, c = mt3d_smooth.smooth(P, T, 3, 0.5, -0.53)
    assert c == dict(n_edges=14, n_fixed_verts=3)
    fixed = [0, 2, 6]
    assert np.array_equal(Q[fixed], P[fixed]) and (Q[[1, 3, 4, 5]] != P[[1, 3, 4, 5]]).any(axis=1).all()
    W, _, _ = naive(P, T, 3, 0.5, -0.53)
    assert Q.tobytes() == W.tobytes()


def test_degenerate_triangles_with_repeated_ids():
    P, T = octahedron()
    P = P + np.random.default_rng(5).normal(0, 0.1, P.shape)
    # (1, 1, 1): self-edges only, no use of anything; (4, 4, 3): {3, 4} used twice more -> non-manifold
    Q, c = mt3d_smooth.smooth(P, np.vstack([T, [[1, 1, 1]]]), 3, 0.5, -0.53)
    Q0, c0 = mt3d_smooth.smooth(P, T, 3, 0.5, -0.53)
    assert Q.tobytes() == Q0.tobytes() and c == c0
    Q, c = mt3d_smooth.smooth(P, np.vstack([T, [[4, 4, 3]]]), 3, 0.5, -0.53)
    assert c == dict(n_edges=12, n_fixed_verts=2) and np.array_equal(Q[[3, 4]], P[[3, 4]])
    W, _, _ = naive(P, np.vstack([T, [[4, 4, 3]]]), 3, 0.5, -0.53)
    assert Q.tobytes() == W.tobytes()
    # a vertex on no triangle is fixed
    Q, c = mt3d_smooth.smooth(np.vstack([P, [[9.0, 9.0, 9.0]]]), T, 2, 0.5, -0.53)
    assert c["n_fixed_verts"] == 1 and np.array_equal(Q[6], [9.0, 9.0, 9.0])


def test_zero_iterations_is_the_identity():
    P, T = octahedron()
    Q, c = mt3d_smooth.smooth(P.astype(np.float32), T, 0, 0.5, -0.53)
    assert Q.dtype == np.float32 and np.array_equal(Q, P.astype(np.float32)) and c["n_edges"] == 12
    Q, c = mt3d_smooth.smooth(np.zeros((0, 3)), np.zeros((0, 3), np.int32), 3, 0.5, -0.53)
    assert Q.shape == (0, 3) and c == dict(n_edges=0, n_fixed_verts=0)


def ball(n, c, r):
    x = np.arange(n, dtype=np.float64)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return (((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) <= r * r).astype(np.uint8)


def spread(Q, c):
    d = np.linalg.norm(Q - np.asarray(c, np.float64), axis=1)
    return np.sqrt(((d - d.mean()) ** 2).mean()), d.mean()


def test_n_edges_equals_the_components_count():
    from test_oracle_components_cpu import wound_mesh
    P, T = wound_mesh(ball(20, (9.5, 9.2, 12.0), 6.3).astype(np.float64), 0.5)
    _, tab = mt3d_components.components(P, T)
    _, c = mt3d_smooth.smooth(P, T, 0, 0.5, -0.53)
    assert c["n_edges"] == tab["n_edges"].sum()
    P, T = grid_patch(5)
    _, tab = mt3d_components.components(P, T)
    assert mt3d_smooth.smooth(P, T, 0, 0.5, -0.53)[1]["n_edges"] == tab["n_edges"].sum()


def test_binary_ball_gets_rounder_without_shrinking():
    # uint8 mask of a ball, isovalue 0.5: the one-voxel staircase.  Numbers of this definition (lambda 0.5, mu -0.53):
    # RMS of |p - c| about its mean 0.281 -> 0.208 (10 iterations) -> 0.181 (20); mean radius 10.338 -> 10.341
    c = (16, 16, 16)
    r = mt3d.extract(ball(33, c, 10.3), 0.5)
    P, T = r["pos"], r["tris"]
    rms0, mean0 = spread(P, c)
    assert abs(rms0 - 0.281) < 0.005 and abs(mean0 - 10.338) < 0.005
    Q10, cnt = mt3d_smooth.smooth(P, T, 10, 0.5, -0.53)
    assert cnt["n_fixed_verts"] == 0
    rms10, mean10 = spread(Q10, c)
    Q20, _ = mt3d_smooth.smooth(P, T, 20, 0.5, -0.53)
    rms20, mean20 = spread(Q20, c)
    assert rms10 < 0.215 and rms20 < 0.188 and rms20 < rms10 < rms0
    assert abs(mean10 - mean0) < 0.01 and abs(mean20 - mean0) < 0.015     # Taubin: no shrinkage
    # plain Laplacian smoothing (mu = 0) shrinks: 10.338 -> 10.264 -> 10.19 in this definition
    L10, _ = mt3d_smooth.smooth(P, T, 10, 0.5, 0.0)
    L20, _ = mt3d_smooth.smooth(P, T, 20, 0.5, 0.0)
    assert spread(L10, c)[1] < mean0 - 0.05 and spread(L20, c)[1] < spread(L10, c)[1] - 0.05
    # n then m iterations equal n + m in fp64
    Q5, _ = mt3d_smooth.smooth(P, T, 5, 0.5, -0.53)
    assert mt3d_smooth.smooth(Q5, T, 5, 0.5, -0.53)[0].tobytes() == Q10.tobytes()


def test_ball_cut_by_the_box_corner_keeps_the_cut_on_the_faces():
    r = mt3d.extract(ball(24, (0, 0, 0), 10.3), 0.5)
    P, T = r["pos"], r["tris"]
    Q, cnt = mt3d_smooth.smooth(P, T, 10, 0.5, -0.53)
    assert cnt["n_fixed_verts"] == 126
    _, _, fixed, _ = mt3d_smooth.neighbours(len(P), T)
    assert fixed.sum() == 126 and np.array_equal(Q[fixed], P[fixed])
    assert (P[fixed].min(axis=1) == 0).all()                      # the boundary is the cut on the box faces
    assert (Q.min(axis=0) == 0).all() and (Q[~fixed] != P[~fixed]).any(axis=1).mean() > 0.9


def test_normals_definition():
    P, T = octahedron(2.0)
    old = -P / 2.0                                                # pointing the other way: the sign rule flips
    n = mt3d_smooth.normals(P, T, old)
    assert np.allclose(n, -P / 2.0, atol=1e-15)
    n = mt3d_smooth.normals(P, T[:, ::-1], P / 2.0)               # winding does not matter
    assert np.allclose(n, P / 2.0, atol=1e-15)
    # a vertex on no triangle, or whose face normals cancel, keeps its old normal
    P2 = np.vstack([P, [[5.0, 5.0, 5.0]]])
    old2 = np.vstack([P / 2.0, [[0.0, 0.0, 1.0]]]).astype(np.float32)
    n = mt3d_smooth.normals(P2.astype(np.float32), T, old2)
    assert n.dtype == np.float32 and np.array_equal(n[6], [0, 0, 1])
    flat = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float64)
    n = mt3d_smooth.normals(flat, [[0, 1, 2], [0, 2, 1]], np.ones((3, 3)))
    assert np.array_equal(n, np.ones((3, 3)))
    mag, parts = mt3d_smooth.face_normal_sums(flat, [[0, 1, 2], [0, 2, 1]])
    assert (mag == 0).all() and np.allclose(parts, 2.0)


def test_new_symbol_declared_exported_and_struct_layout():
    from test_capi_symbols import declared_symbols
    from contourist_b200 import build, engine
    assert "ctr_mt3d_smooth" in declared_symbols()
    assert ctypes.sizeof(engine.SmoothParams) == 24 and ctypes.sizeof(engine.SmoothCounts) == 16
    build.build()
    lib = engine.load_library()
    assert lib.ctr_mt3d_smooth(None, None, None) == -1             # null context, no CUDA touched


class SmoothStub(StubEngine):
    def __init__(self):
        StubEngine.__init__(self)
        self.smoothed = None

    def mt3d_smooth(self, iterations, lam, mu):
        self.calls.append("smooth")
        self.smoothed = (iterations, lam, mu)


@pytest.mark.parametrize("post_process", [True, False])
def test_facade_smooths_after_the_filter_and_measures_again(monkeypatch, post_process):
    from contourist_b200 import engine as E
    stub = SmoothStub()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    t = _make(post_process, keep_components=1, measure_components=True, vertex_fields=lambda x, y, z: x,
              smooth_iterations=4, smooth_lambda=0.4, smooth_mu=-0.45)
    t.get_points_and_triangles()
    edit = "clean" if post_process else "orient"
    # the filter's results describe the unsmoothed mesh: measured again, not fetched
    assert stub.calls == ["run", edit, "components", "keep", "smooth", "interpolate", "components", "fetch"]
    assert stub.smoothed == (4, 0.4, -0.45)
    stub.calls = []
    _make(post_process, measure_components=True, smooth_iterations=2).get_points_and_triangles()
    assert stub.calls == ["run", edit, "smooth", "components", "fetch"] and stub.smoothed == (2, 0.5, -0.53)


def test_facade_defaults_do_not_smooth_and_smooth_still_raises(monkeypatch):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    stub = SmoothStub()
    monkeypatch.setattr(E, "default_engine", lambda *a, **k: stub)
    _make(True, keep_components=1, measure_components=True).get_points_and_triangles()
    assert "smooth" not in stub.calls and stub.calls[-2] == "components_fetch"
    g = tetrahedral.GridContour3d
    assert (g.smooth_iterations, g.smooth_lambda, g.smooth_mu) == (0, 0.5, -0.53)
    f = lambda x, y, z: x * x + y * y + z * z
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.5, 0.5, 0.5), f, 0.5, [], smooth=True)
    t.smooth_iterations = 3
    with pytest.raises(NotImplementedError):
        t.get_points_and_triangles()
    assert "smooth" not in stub.calls
