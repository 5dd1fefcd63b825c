"""CPU: the definition of ctr_mt3d_closest (oracle/mt3d_closest.py) on small meshes, its pruned path against brute force,
and the façade's closest_points checks."""
import numpy as np
import pytest

from oracle import mt3d_closest

TRI = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def _one(verts, tris, p, **kw):
    r, n = mt3d_closest.closest(verts, tris, np.asarray([p], np.float64), **kw)
    return r["point"][0], r["distance"][0], r["triangle"][0], n


# region of Ericson's walk -> (query point, closest point, d2)
REGIONS = {
    "a": ((-1.0, -1.0, 0.5), (0.0, 0.0, 0.0), 2.25),
    "b": ((2.0, -1.0, 0.0), (1.0, 0.0, 0.0), 2.0),
    "ab": ((0.5, -1.0, 1.0), (0.5, 0.0, 0.0), 2.0),
    "c": ((-1.0, 2.0, 0.0), (0.0, 1.0, 0.0), 2.0),
    "ac": ((-1.0, 0.5, 0.0), (0.0, 0.5, 0.0), 1.0),
    "bc": ((1.0, 1.0, 0.0), (0.5, 0.5, 0.0), 0.5),
    "inside": ((0.25, 0.25, 2.0), (0.25, 0.25, 0.0), 4.0),
}


@pytest.mark.parametrize("region", list(REGIONS))
def test_single_triangle_regions(region):
    p, q, d2 = REGIONS[region]
    got, dist, t, n = _one(TRI, [[0, 1, 2]], p)
    assert np.array_equal(got, q) and dist == np.sqrt(d2) and t == 0 and n == 1
    # the corner order does not move the answer on a regular triangle
    got, dist, t, _ = _one(TRI, [[1, 2, 0]], p)
    assert np.array_equal(got, q) and dist == np.sqrt(d2)


DEGENERATE = {
    "collinear": ([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [2.0, 0.0, 0.0]], (0.5, 1.0, 0.0), (0.5, 0.0, 0.0)),
    "collinear_beyond": ([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [2.0, 0.0, 0.0]], (3.0, 1.0, 0.0), (2.0, 0.0, 0.0)),
    "repeated_ab": ([[0.0, 0.0, 0.0], [0.0, 0.0, 0.0], [1.0, 0.0, 0.0]], (0.5, 1.0, 0.0), (0.5, 0.0, 0.0)),
    "repeated_ac": ([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 0.0]], (0.5, 1.0, 0.0), (0.5, 0.0, 0.0)),
    "repeated_bc": ([[1.0, 0.0, 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]], (0.25, -2.0, 0.0), (0.25, 0.0, 0.0)),
    "point": ([[1.0, 1.0, 1.0]] * 3, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
}


@pytest.mark.parametrize("case", list(DEGENERATE))
def test_degenerate_triangles_take_the_segment_rule(case):
    v, p, q = DEGENERATE[case]
    got, dist, t, n = _one(np.array(v), [[0, 1, 2]], p)
    assert np.array_equal(got, q) and t == 0 and n == 1
    assert dist == np.sqrt(np.sum((np.array(p) - np.array(q)) ** 2))


def test_degenerate_triangles_never_give_nan():
    rng = np.random.default_rng(3)
    v = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [2.0, 0.0, 0.0], [0.5, 0.0, 0.0], [0.0, 0.0, 0.0],
                  [1e-300, 0.0, 0.0], [1.0, 1e-17, 0.0]])
    tris = np.array([[0, 1, 2], [0, 0, 1], [1, 0, 0], [0, 3, 1], [0, 4, 0], [4, 4, 4], [0, 5, 1], [0, 1, 6], [6, 1, 0]])
    P = np.concatenate([rng.normal(size=(400, 3)) * 3, v, (v[:, None] + v[None]).reshape(-1, 3) / 2])
    for t in range(len(tris)):
        r, n = mt3d_closest.closest(v, tris[t:t + 1], P)
        assert n == len(P) and np.isfinite(r["point"]).all() and np.isfinite(r["distance"]).all(), tris[t]
        # never farther than the triangle's corners, never nearer than the exact segment / triangle allows
        corners = np.sqrt(((P[:, None, :] - v[tris[t]][None]) ** 2).sum(axis=2)).min(axis=1)
        assert (r["distance"] <= corners * (1 + 1e-12)).all()


def test_equal_distance_smallest_index_wins():
    up = TRI + [0.0, 0.0, 1.0]
    down = TRI - [0.0, 0.0, 1.0]
    v = np.concatenate([up, down])
    for tris in ([[0, 1, 2], [3, 4, 5]], [[3, 4, 5], [0, 1, 2]]):
        got, dist, t, _ = _one(v, tris, (0.25, 0.25, 0.0))
        assert t == 0 and dist == 1.0
    # the two triangles on an edge: its midpoint is at distance 0 from both
    v = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 1.0, 0.0]])
    got, dist, t, _ = _one(v, [[3, 2, 1], [0, 1, 2]], (0.5, 0.5, 0.0))
    assert t == 0 and dist == 0.0


def test_max_distance_is_inclusive():
    p = (0.25, 0.25, 2.0)
    assert _one(TRI, [[0, 1, 2]], p, max_distance=2.0)[2:] == (0, 1)
    got, dist, t, n = _one(TRI, [[0, 1, 2]], p, max_distance=np.nextafter(2.0, 0.0))
    assert (t, n) == (-1, 0) and dist == np.inf and np.isnan(got).all()
    assert _one(TRI, [[0, 1, 2]], p, max_distance=0.0)[2:] == (-1, 0)
    with pytest.raises(ValueError):
        _one(TRI, [[0, 1, 2]], p, max_distance=-1.0)
    with pytest.raises(ValueError):
        _one(TRI, [[0, 1, 2]], p, max_distance=np.nan)
    with pytest.raises(ValueError):
        _one(TRI, [[0, 1, 2]], (np.nan, 0.0, 0.0))


def test_empty_mesh():
    r, n = mt3d_closest.closest(TRI, np.zeros((0, 3), np.int32), np.ones((4, 3)))
    assert n == 0 and (r["distance"] == np.inf).all() and (r["triangle"] == -1).all() and np.isnan(r["point"]).all()
    r, n = mt3d_closest.closest(TRI, [[0, 1, 2]], np.zeros((0, 3)))
    assert n == 0 and r["point"].shape == (0, 3)


def _mesh(seed, n=12):
    "a bumpy closed UV sphere in fp32, with a few zero-area and repeated-corner triangles appended"
    rng = np.random.default_rng(seed)
    th = np.linspace(0, np.pi, n + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, 2 * n, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    ring = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], axis=-1).reshape(-1, 3)
    v = np.concatenate([[[0, 0, 1]], ring, [[0, 0, -1]]]) * (1 + 0.1 * rng.random((len(ring) + 2, 1)))
    m = 2 * n
    idx = lambda r, c: 1 + r * m + (c % m)
    tris = [(0, idx(0, c), idx(0, c + 1)) for c in range(m)] + \
           [(len(v) - 1, idx(n - 2, c + 1), idx(n - 2, c)) for c in range(m)]
    for r in range(n - 2):
        for c in range(m):
            tris += [(idx(r, c), idx(r + 1, c), idx(r + 1, c + 1)), (idx(r, c), idx(r + 1, c + 1), idx(r, c + 1))]
    tris = np.array(tris, np.int64)
    extra = rng.integers(0, len(v), size=(6, 1))
    tris = np.concatenate([tris, np.concatenate([extra, extra, rng.integers(0, len(v), (6, 1))], axis=1)])
    return (v * 10).astype(np.float32), tris


@pytest.mark.parametrize("seed", range(4))
def test_pruned_equals_brute_force(seed):
    v, tris = _mesh(seed)
    rng = np.random.default_rng(100 + seed)
    e = tris[:, :2]
    P = np.concatenate([rng.uniform(-15, 15, (300, 3)), rng.uniform(-1500, 1500, (20, 3)), v[:50].astype(np.float64),
                        (v[e[:, 0]] + v[e[:, 1]])[:200] / 2])
    for md in (np.inf, 2.0):
        a, na = mt3d_closest.closest(v, tris, P, max_distance=md)
        b, nb = mt3d_closest.closest(v, tris, P, max_distance=md, prune=True)
        assert na == nb
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), (k, md)
    assert (a["distance"][320:370] == 0).all()


def test_vertices_are_at_distance_zero():
    v, tris = _mesh(7)
    used = np.unique(tris)
    for prune in (False, True):
        r, n = mt3d_closest.closest(v, tris, v[used], prune=prune)
        assert n == len(used) and (r["distance"] == 0).all()
        assert np.array_equal(r["point"], v[used].astype(np.float64))


def test_facade_closest_points_checks():
    from contourist_b200 import tetrahedral
    t = tetrahedral.GridContour3d((4, 4, 4), np.zeros((5, 5, 5)), 0.5, None)
    for bad in (np.zeros((3, 2)), np.zeros(3), [[0.0, np.nan, 0.0]], [[np.inf, 0.0, 0.0]]):
        t.closest_points = bad
        with pytest.raises(ValueError):
            t._closest_points()
    t.closest_points = [[1, 2, 3]]
    assert t._closest_points().dtype == np.float64
