"""CPU: the definition of ctr_mt3d_raycast (oracle/mt3d_raycast.py) on small meshes, its pruned path against brute force,
and the façade's rays checks."""
import numpy as np
import pytest

from oracle import mt3d_raycast
from test_oracle_closest_cpu import _mesh

TRI = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def _cast(verts, tris, O, D, **kw):
    return mt3d_raycast.raycast(verts, tris, np.asarray(O, np.float64).reshape(-1, 3), np.asarray(D, np.float64).reshape(-1, 3), **kw)


def _same(a, b):
    for k in a:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k], equal_nan=True), k


def adversarial_rays(v, tris, rng, n=300):
    "random rays in and around the box, rays aimed at vertices, edge midpoints and centroids, in-plane, axis-parallel"
    v = v.astype(np.float64)
    lo, hi = v.min(axis=0), v.max(axis=0)
    ext = (hi - lo).max()
    t = tris[rng.integers(0, len(tris), n)]
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    O = rng.uniform(lo - ext, hi + ext, (n, 3))
    axis = np.eye(3)[rng.integers(0, 3, n)] * rng.choice([-1.0, 1.0], (n, 1))
    sets = {"random": (rng.uniform(lo - 1, hi + 1, (n, 3)), rng.normal(size=(n, 3))),
            "vertices": (O, a - O),
            "midpoints": (O, (a + b) / 2 - O),
            "centroids": (O, (a + b + c) / 3 - O),
            "in_plane": (a - (b - a), b - a),
            "axis": (rng.uniform(lo, hi, (n, 3)), axis),
            "axis_at_vertices": (a - 2 * ext * axis, axis),
            "miss_box": (np.broadcast_to(hi + ext, (n, 3)), rng.uniform(0.1, 1.0, (n, 3))),
            "far": ((lo + hi) / 2 + rng.normal(size=(n, 3)) * 1e6, (lo + hi) / 2 + rng.normal(size=(n, 3)))}
    sets["far"] = (sets["far"][0], sets["far"][1] - sets["far"][0])
    for k, (o, d) in sets.items():                    # an edge of a zero-area triangle gives no direction
        sets[k] = (o, np.where((d == 0).all(axis=1, keepdims=True), [1.0, 0.0, 0.0], d))
    return sets


@pytest.mark.parametrize("seed", range(3))
def test_pruned_equals_brute_force(seed):
    v, tris = _mesh(seed)
    rng = np.random.default_rng(200 + seed)
    for name, (O, D) in adversarial_rays(v, tris, rng).items():
        for t_min, t_max in ((0.0, np.inf), (-np.inf, np.inf), (0.5, 1.5)):
            a, na = _cast(v, tris, O, D, t_min=t_min, t_max=t_max)
            b, nb = _cast(v, tris, O, D, t_min=t_min, t_max=t_max, prune=True)
            assert na == nb, name
            _same(a, b)


def test_watertight_closed_mesh():
    "rays from an interior point through every vertex and every edge midpoint of a closed mesh all hit, from inside"
    v, tris = _mesh(5, n=16)
    tris = tris[:-6]                                  # the closed sphere, without the appended zero-area triangles
    V = v.astype(np.float64)
    e = np.unique(np.sort(np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]]), axis=1), axis=0)
    targets = np.concatenate([V, (V[e[:, 0]] + V[e[:, 1]]) / 2])
    for o in ([0.0, 0.0, 0.0], [0.3, -0.7, 0.1]):
        O = np.broadcast_to(np.array(o), targets.shape)
        for D in (targets - O, (targets - O) * 3.0):
            r, n = _cast(v, tris, O, D)
            assert n == len(targets)
            assert (r["side"] == r["side"][0]).all()  # a consistently wound closed surface: always the same side
            q, nq = _cast(v, tris, O, D, prune=True)
            _same(r, q)


def test_weights_recombine_to_point():
    v, tris = _mesh(3)
    rng = np.random.default_rng(7)
    O, D = adversarial_rays(v, tris, rng)["centroids"]
    r, n = _cast(v, tris, O, D)
    assert n == len(O)
    V = v.astype(np.float64)
    t = tris[r["triangle"]]
    rec = (r["weights"][:, :1] * V[t[:, 0]] + r["weights"][:, 1:2] * V[t[:, 1]]) + r["weights"][:, 2:] * V[t[:, 2]]
    assert np.abs(rec - r["point"]).max() <= 8 * np.finfo(np.float64).eps * np.abs(V).max()
    assert np.allclose(r["weights"].sum(axis=1), 1.0, rtol=0, atol=1e-14)
    assert (r["weights"] >= 0).all()


def test_side_is_minus_sign_of_d_dot_normal():
    rng = np.random.default_rng(9)
    n = 2000
    a, b, c = rng.normal(size=(3, n, 3))
    nrm = np.cross(b - a, c - a)
    good = np.linalg.norm(nrm, axis=1) > 0.5
    cen = (a + b + c) / 3
    O = cen + rng.normal(size=(n, 3)) * 3
    D = cen - O
    good &= np.abs(np.einsum("ij,ij->i", D / np.linalg.norm(D, axis=1)[:, None], nrm / np.linalg.norm(nrm, axis=1)[:, None])) > 0.1
    V = np.concatenate([a, b, c])
    tris = np.stack([np.arange(n), n + np.arange(n), 2 * n + np.arange(n)], axis=1)
    for i in np.nonzero(good)[0][:300]:
        r, k = _cast(V, tris[i:i + 1], O[i], D[i])
        assert k == 1 and r["side"][0] == -np.sign(D[i] @ nrm[i])


def test_t_range_is_inclusive():
    O, D = [0.25, 0.25, 2.0], [0.0, 0.0, -1.0]
    r, n = _cast(TRI, [[0, 1, 2]], O, D)
    assert n == 1 and r["t"][0] == 2.0 and np.array_equal(r["point"][0], [0.25, 0.25, 0.0])
    assert np.array_equal(r["weights"][0], [0.5, 0.25, 0.25]) and r["side"][0] == 1
    assert _cast(TRI, [[0, 1, 2]], O, D, t_max=2.0)[1] == 1
    assert _cast(TRI, [[0, 1, 2]], O, D, t_min=2.0)[1] == 1
    assert _cast(TRI, [[0, 1, 2]], O, D, t_max=np.nextafter(2.0, 0.0))[1] == 0
    r, n = _cast(TRI, [[0, 1, 2]], O, D, t_min=np.nextafter(2.0, 3.0))
    assert n == 0 and r["t"][0] == np.inf and r["triangle"][0] == -1 and r["side"][0] == 0
    assert np.isnan(r["weights"]).all() and np.isnan(r["point"]).all()
    # from below: the back of the triangle
    r, n = _cast(TRI, [[0, 1, 2]], [0.25, 0.25, -2.0], [0.0, 0.0, 0.5])
    assert n == 1 and r["t"][0] == 4.0 and r["side"][0] == -1


def test_duplicates_tie_to_the_smaller_index():
    O, D = [0.25, 0.25, 2.0], [0.0, 0.0, -1.0]
    for tris in ([[0, 1, 2], [0, 1, 2]], [[1, 2, 0], [0, 1, 2]], [[0, 2, 1], [0, 1, 2]]):
        for prune in (False, True):
            r, n = _cast(TRI, tris, O, D, prune=prune)
            assert n == 1 and r["triangle"][0] == 0 and r["t"][0] == 2.0
    # the two triangles of a square, through their shared edge: one hit, the smaller index
    v = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 1.0, 0.0]])
    r, n = _cast(v, [[3, 2, 1], [0, 1, 2]], [0.5, 0.5, 1.0], [0.0, 0.0, -1.0])
    assert n == 1 and r["triangle"][0] == 0 and r["t"][0] == 1.0


def test_axis_parallel_directions():
    v, tris = _mesh(11)
    V = v.astype(np.float64)
    rng = np.random.default_rng(13)
    for k in range(3):
        for s in (-1.0, 1.0):
            D = np.zeros((200, 3))
            D[:, k] = s
            O = rng.uniform(-12, 12, (200, 3))
            O[:, k] = -s * 40.0
            a, na = _cast(v, tris, O, D)
            b, nb = _cast(v, tris, O, D, prune=True)
            _same(a, b)
            assert 0 < na < 200
    # aimed exactly at vertices along an axis
    D = np.tile([0.0, 0.0, -1.0], (len(V), 1))
    O = V + [0.0, 0.0, 50.0]
    r, n = _cast(v, tris, O, D)
    assert n == len(np.unique(tris))
    _same(r, _cast(v, tris, O, D, prune=True)[0])


def test_empty_mesh_and_no_rays():
    r, n = _cast(TRI, np.zeros((0, 3), np.int32), np.zeros((4, 3)), np.ones((4, 3)))
    assert n == 0 and (r["t"] == np.inf).all() and (r["triangle"] == -1).all() and (r["side"] == 0).all()
    assert np.isnan(r["weights"]).all() and np.isnan(r["point"]).all()
    r, n = _cast(TRI, [[0, 1, 2]], np.zeros((0, 3)), np.zeros((0, 3)))
    assert n == 0 and r["point"].shape == (0, 3) and r["side"].dtype == np.int8


def test_bad_rays_raise():
    for kw in (dict(O=[np.nan, 0, 0], D=[0, 0, 1]), dict(O=[0, 0, 0], D=[0, 0, np.inf]), dict(O=[0, 0, 0], D=[0, 0, 0])):
        with pytest.raises(ValueError):
            _cast(TRI, [[0, 1, 2]], kw["O"], kw["D"])
    for t_min, t_max in ((1.0, 0.0), (np.nan, 1.0), (0.0, np.nan)):
        with pytest.raises(ValueError):
            _cast(TRI, [[0, 1, 2]], [0, 0, 1], [0, 0, -1], t_min=t_min, t_max=t_max)


def test_facade_rays_checks():
    from contourist_b200 import tetrahedral
    t = tetrahedral.GridContour3d((4, 4, 4), np.zeros((5, 5, 5)), 0.5, None)
    for bad in (np.zeros((3, 3)), (np.zeros((3, 2)), np.zeros((3, 2))), (np.zeros((3, 3)), np.ones((2, 3))),
                ([[0.0, np.nan, 0.0]], [[1.0, 0.0, 0.0]]), ([[0.0, 0.0, 0.0]], [[np.inf, 0.0, 0.0]]),
                ([[0.0, 0.0, 0.0]], [[0.0, 0.0, 0.0]])):
        t.rays = bad
        with pytest.raises(ValueError):
            t._rays()
    t.rays = ([[1, 2, 3]], [[0, 0, 1]])
    O, D = t._rays()
    assert O.dtype == D.dtype == np.float64
