"""CPU: the definition of ctr_mt3d_clip (oracle/mt3d_clip.py) on small meshes, and the façade's clip_halfspaces checks."""
import numpy as np
import pytest

from oracle import mt3d_clip, mt3d_section


def _cross(v, t):
    p = np.asarray(v, np.float64)[np.asarray(t, np.int64)]
    return np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])


def _area(v, t):
    return 0.5 * np.linalg.norm(_cross(v, t), axis=1).sum()


def sphere(n=24):
    "a closed UV sphere of radius 1, outward"
    th = np.linspace(0, np.pi, n + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, 2 * n, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    ring = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], axis=-1).reshape(-1, 3)
    verts = np.concatenate([[[0, 0, 1]], ring, [[0, 0, -1]]]).astype(np.float64)
    m = 2 * n
    idx = lambda r, c: 1 + r * m + (c % m)
    tris = []
    for c in range(m):
        tris.append((0, idx(0, c), idx(0, c + 1)))
        tris.append((len(verts) - 1, idx(n - 2, c + 1), idx(n - 2, c)))
    for r in range(n - 2):
        for c in range(m):
            tris.append((idx(r, c), idx(r + 1, c), idx(r + 1, c + 1)))
            tris.append((idx(r, c), idx(r + 1, c + 1), idx(r, c + 1)))
    tris = np.array(tris, np.int64)
    assert (np.einsum("ij,ij->i", _cross(verts, tris), verts[tris].mean(axis=1)) > 0).all()
    return verts, tris


TRI = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


@pytest.mark.parametrize("side", ["high", "low"])
@pytest.mark.parametrize("pattern", range(8))
def test_single_triangle_patterns(side, pattern):
    # corner i high iff bit i of pattern: value clip on s = +1 / -1
    s = np.array([1.0 if (pattern >> i) & 1 else -1.0 for i in range(3)])
    nrm = np.tile([0.0, 0.0, 1.0], (3, 1))
    out, c = mt3d_clip.clip(TRI, [[0, 1, 2]], normals=nrm, values=s, component=0, offset=0.0, side=side,
                            geom_dtype=np.float64)
    kept = [(s[i] >= 0) == (side == "high") for i in range(3)]
    nk = sum(kept)
    want_pieces = {0: 0, 1: 1, 2: 2, 3: 1}[nk]
    assert c["n_tris"] == want_pieces == len(out["tris"])
    assert c["n_dropped_tris"] == (nk == 0) and c["n_cut_tris"] == (0 < nk < 3)
    assert c["n_new_verts"] == (2 if 0 < nk < 3 else 0)
    if nk == 3:
        assert np.array_equal(out["tris"], [[0, 1, 2]])
        return
    # the walk: tokens in corner order, kept corners renumbered, crossings appended
    toks = []
    for i in range(3):
        if kept[i]:
            toks.append(("c", i))
        if kept[i] != kept[(i + 1) % 3]:
            toks.append(("x", i))
    # ids of the tokens: kept corners renumbered in order, the two crossings nk, nk + 1 in walk order
    ids = [sum(kept[:tok[1]]) if tok[0] == "c" else nk + [t for t in toks if t[0] == "x"].index(tok) for tok in toks]
    want = [] if not ids else [[ids[0], ids[1], ids[2]]] + ([[ids[0], ids[2], ids[3]]] if len(ids) == 4 else [])
    assert out["tris"].tolist() == want
    if len(out["tris"]):
        # every piece faces the source's way; crossings lie on the cut (values 0) and at the edge midpoints
        assert (_cross(out["verts"], out["tris"])[:, 2] >= 0).all() and _area(out["verts"], out["tris"]) > 0
        assert np.array_equal(out["normals"][nk:], np.tile([0.0, 0.0, 1.0], (2, 1)))
        assert np.all(out["values"][nk:] == 0.0)


def test_shared_edge_gets_one_vertex():
    v = np.array([[0.0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]])
    t = np.array([[0, 1, 2], [1, 3, 2]])
    out, c = mt3d_clip.clip(v, t, normal=(1.0, 1.0, 0.0), offset=1.0, side="low", geom_dtype=np.float64)
    # kept: vertex 0 (s = 0); {1, 2} lie on the plane (s = 1 >= 1: high), vertex 3 high: triangle 1 dropped
    assert c == dict(n_verts=3, n_tris=1, n_new_verts=2, n_cut_tris=1, n_dropped_tris=1)
    out, c = mt3d_clip.clip(v, t, normal=(1.0, 0.0, 0.0), offset=0.5, side="low", geom_dtype=np.float64)
    # kept 0, 2; edges {0, 1}, {1, 2} (crossed by both triangles: one vertex), {2, 3}... x = 0.5 crosses {0, 1},
    # {1, 2} and {2, 3}: three new vertices, numbered by first use
    assert c == dict(n_verts=5, n_tris=3, n_new_verts=3, n_cut_tris=2, n_dropped_tris=0)
    assert np.array_equal(out["verts"][2:], [[0.5, 0, 0], [0.5, 0.5, 0], [0.5, 1, 0]])
    assert out["tris"].tolist() == [[0, 2, 3], [0, 3, 1], [4, 1, 3]]


@pytest.mark.parametrize("normal", [(0.0, 0.0, 1.0), (1.0, 2.0, 3.0), (-0.3, 0.7, 0.2)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_high_plus_low_is_the_whole(normal, dtype):
    v, t = sphere()
    v = v.astype(dtype)
    d = 0.137
    hi, _ = mt3d_clip.clip(v, t, normal=normal, offset=d, side="high", geom_dtype=dtype)
    lo, _ = mt3d_clip.clip(v, t, normal=normal, offset=d, side="low", geom_dtype=dtype)
    whole = _area(v, t)
    tol = 1e-12 if dtype == np.float64 else 1e-6
    assert abs(_area(hi["verts"], hi["tris"]) + _area(lo["verts"], lo["tris"]) - whole) <= tol * whole


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_rim_points_are_the_section_points(dtype):
    v, t = sphere()
    v = v.astype(dtype)
    normal, d = (0.3, -0.5, 0.8), 0.21
    out, c = mt3d_clip.clip(v, t, normal=normal, offset=d, side="high", geom_dtype=dtype)
    _, _, pts = mt3d_section.segments(v, t, normal, [d], dtype)
    rim = out["verts"][c["n_verts"] - c["n_new_verts"]:]
    seg = np.unique(pts.reshape(-1, 3), axis=0)
    assert len(rim) == len(seg) and np.array_equal(np.unique(rim, axis=0), seg)


def test_noop_and_empty():
    v, t = sphere()
    keys = np.arange(len(v), dtype=np.uint64)
    out, c = mt3d_clip.clip(v, t, keys=keys, normal=(0, 0, 1.0), offset=-5.0, side="high", geom_dtype=np.float64)
    assert c == dict(n_verts=len(v), n_tris=len(t), n_new_verts=0, n_cut_tris=0, n_dropped_tris=0)
    assert np.array_equal(out["verts"], v) and np.array_equal(out["tris"], t) and np.array_equal(out["keys"], keys)
    out, c = mt3d_clip.clip(v, t, keys=keys, normal=(0, 0, 1.0), offset=5.0, side="high", geom_dtype=np.float64)
    assert c == dict(n_verts=0, n_tris=0, n_new_verts=0, n_cut_tris=0, n_dropped_tris=len(t))
    assert out["verts"].shape == (0, 3) and out["tris"].shape == (0, 3) and len(out["keys"]) == 0
    out, c = mt3d_clip.clip(np.zeros((0, 3)), np.zeros((0, 3), int), normal=(1.0, 0, 0), offset=0.0, side="low",
                            geom_dtype=np.float64)
    assert c["n_verts"] == 0 and c["n_tris"] == 0


def test_nan_and_bad_ids_raise():
    with pytest.raises(ValueError):
        mt3d_clip.clip(TRI, [[0, 1, 2]], values=np.array([0.0, np.nan, 1.0]), component=0, offset=0.0, side="high",
                       geom_dtype=np.float64)
    with pytest.raises(ValueError):
        mt3d_clip.clip(TRI, [[0, 1, 3]], normal=(1.0, 0, 0), offset=0.0, side="high", geom_dtype=np.float64)


def test_repeated_id_triangle():
    out, c = mt3d_clip.clip(TRI, [[0, 0, 1]], normal=(1.0, 0, 0), offset=0.5, side="low", geom_dtype=np.float64)
    # corners 0, 0 kept, 1 not: tokens 0, 0, x(0,1), x(1,0) -- one crossing vertex, a degenerate fan; vertex 2 is
    # kept although no triangle uses it, so the crossing is vertex 2
    assert c["n_new_verts"] == 1 and c["n_tris"] == 2 and c["n_verts"] == 3
    assert out["tris"].tolist() == [[0, 0, 2], [0, 2, 2]]


def test_six_plane_box_of_a_sphere():
    v, t = sphere(32)
    A = np.array([[1.0, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]])
    b = np.array([0.61, 0.53, 0.47, 0.71, 0.66, 0.58])
    mesh = dict(verts=v, tris=t)
    for a, d in zip(A, b):
        mesh, _ = mt3d_clip.clip(mesh["verts"], mesh["tris"], normal=a, offset=d, side="low", geom_dtype=np.float64)
    tr = mesh["tris"].astype(np.int64)
    e = np.sort(np.concatenate([tr[:, [0, 1]], tr[:, [1, 2]], tr[:, [2, 0]]]), axis=1)
    ue, cnt = np.unique(e, axis=0, return_counts=True)
    assert set(cnt.tolist()) <= {1, 2} and (cnt == 1).sum() > 0
    p = mesh["verts"]
    for (i, j) in ue[cnt == 1]:
        # a rim edge lies on one of the planes, both of its ends
        on = [np.allclose(p[[i, j]] @ a, d, atol=1e-12) for a, d in zip(A, b)]
        assert any(on)
    assert ((p @ A.T) < b + 1e-12).all()


def test_facade_validation():
    from contourist_b200 import tetrahedral
    f = np.zeros((5, 5, 5))
    for bad in [np.zeros((2, 3)), (np.zeros((2, 2)), np.zeros(2)), (np.zeros((2, 3)), np.zeros(3)),
                (np.array([[1.0, 0, np.inf]]), np.zeros(1)), (np.array([[1.0, 0, 0]]), np.array([np.nan])),
                (np.array([[0.0, 0, 0]]), np.zeros(1))]:
        m = tetrahedral.Grid3DContour(4, 4, 4, f, 0.5, None)
        m.clip_halfspaces = bad
        with pytest.raises(ValueError):
            m.get_points_and_triangles()
    m = tetrahedral.Grid3DContour(4, 4, 4, f, 0.5, None)
    m.clip_halfspaces = ([[1, 0, 0], [0, 1, 0]], [1, 2])
    A, b = m._halfspaces()
    assert A.dtype == np.float64 and A.shape == (2, 3) and b.shape == (2,)
