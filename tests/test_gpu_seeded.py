"""GPU: seeded extraction (ctr_mt3d_select_seeded, SURVEY.md 8(f3)) against the oracle's restatement of the
reference tracker and against the reference's own seeded runs (tests/golden/seeded3d_*.npz)."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import mt3d

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "seeded3d_*.npz")))


def run_seeded(engine, field, value, seeds, geom64=True):
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    flags = E.WANT_KEYS | E.WANT_NORMALS | (E.GEOM_F64 if geom64 else 0)
    full = engine.mt3d_run(field, value, flags=flags)
    n_full = (int(full.n_verts), int(full.n_tris))
    start = tetrahedral.initial_voxels(field, value, seeds) if len(seeds) else np.zeros((0, 3), np.int32)
    nv, nt, ncell = engine.mt3d_select_seeded(start)
    raw = engine.mt3d_fetch()
    assert raw["verts"].shape == (nv, 3) and raw["tris"].shape == (nt, 3) and raw["normals"].shape == (nv, 3)
    assert len(np.unique(raw["keys"])) == nv
    if nt:
        assert raw["tris"].min() >= 0 and raw["tris"].max() < nv and len(np.unique(raw["tris"])) == nv
    o = E.canonical_mesh(raw)
    r = mt3d.extract_seeded(field, value, seeds, np.float64 if geom64 else np.float32)
    assert np.array_equal(o["keys"], r["keys"])
    assert np.array_equal(o["lowmin"], r["lowmin"])
    assert np.array_equal(np.sort(o["tris"], axis=1), np.sort(r["tris"], axis=1))
    assert ncell == len(r["cells"])
    if geom64:
        assert np.array_equal(o["verts"], r["pos"])
    else:
        np.testing.assert_allclose(o["verts"], r["pos"], rtol=1e-4, atol=1e-5)
    nr = mt3d.normals(field, value, r["keys"], np.float64 if geom64 else np.float32)
    np.testing.assert_allclose(o["normals"], nr, rtol=1e-9 if geom64 else 1e-4, atol=1e-11 if geom64 else 1e-4)
    return n_full, (nv, nt), r


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("geom64", [True, False])
def test_reference_seeded_runs(engine, path, geom64):
    g = np.load(path)
    n_full, (nv, nt), r = run_seeded(engine, g["field"], float(g["value"]), g["seeds"], geom64)
    assert (nv, nt) == (int(g["n_keys"]), int(g["n_tris"]))                # the reference tracker's own counts
    gv = g["voxels"]
    n1, n2 = g["field"].shape[1] - 1, g["field"].shape[2] - 1
    assert np.isin(r["cells"], (gv[:, 0] * n1 + gv[:, 1]) * n2 + gv[:, 2]).all()
    if "wave_sheet" not in path:
        assert nt < n_full[1]


def test_integer_field_walks_through_connector_voxels(engine):
    """Samples exactly on the isovalue: border voxels that emit nothing still carry the flood fill."""
    rng = np.random.default_rng(12)
    f = rng.integers(-2, 3, size=(14, 13, 15)).astype(np.float64)
    f[3:11, 2:11, 3:12] = -2.0                                 # a moat two voxels wide: more than one component
    f[6:8, 6:7, 7:8] = 2.0
    seeds = [[(6, 6, 7), (6, 6, 9)]]
    n_full, n_sel, r = run_seeded(engine, f, 0.0, seeds)
    assert 0 < n_sel[1] < n_full[1]
    # two low pockets in a high background, 4 samples apart: separate surfaces ...
    two = np.full((9, 6, 6), 1.0)
    two[2, 2, 2] = two[6, 2, 2] = -1.0
    seed = [[(2, 2, 2), (2, 2, 5)]]
    n_full, n_sel, r = run_seeded(engine, two, 0.0, seed)
    assert n_sel[1] * 2 == n_full[1]
    # ... until a sample between them sits exactly on the isovalue: its voxels emit nothing (all corners high) but are
    # border voxels (min <= value, tetrahedral.py:383-394), and the reference's flood fill walks across them
    two[4, 2, 2] = 0.0
    n_full2, n_sel2, r = run_seeded(engine, two, 0.0, seed)
    assert n_full2 == n_full and n_sel2 == n_full


def test_many_seeds_and_no_seeds(engine):
    n = 44
    x, y, z = np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing="ij")
    rng = np.random.default_rng(9)
    f = np.zeros((n, n, n))
    cen = rng.uniform(6, n - 6, (10, 3))
    for c in cen:
        f += np.exp(-((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2) / rng.uniform(6.0, 14.0))
    f32 = f.astype(np.float32)
    seeds = []
    for c in cen[:4]:
        p = tuple(int(round(v)) for v in c)
        q = (p[0], p[1], 0)
        if f32[p] > 0.5 > f32[q]:
            seeds.append([p, q])
    assert len(seeds) >= 2
    n_full, n_sel, r = run_seeded(engine, f32, 0.5, seeds, geom64=False)
    assert 0 < n_sel[1] < n_full[1]
    n_full, n_sel, r = run_seeded(engine, f32, 0.5, [])
    assert n_sel == (0, 0)
    # every crossing segment as seed = the full scan
    lo = [int(np.clip(int(c) - 10, 0, n - 20)) for c in cen[0]]
    sub = np.ascontiguousarray(f32[lo[0]:lo[0] + 20, lo[1]:lo[1] + 20, lo[2]:lo[2] + 20]).astype(np.float64)
    base = sub[:19, :19, :19] - 0.5
    segs = []
    for c in range(1, 8):                                       # grid_field.py:64-84
        d = ((c >> 2) & 1, (c >> 1) & 1, c & 1)
        nb = sub[d[0]:19 + d[0], d[1]:19 + d[1], d[2]:19 + d[2]] - 0.5
        for v0 in np.argwhere(base * nb < 0):
            segs.append([tuple(v0), tuple(v0 + np.array(d))])
    assert len(segs) > 100
    n_full, n_sel, r = run_seeded(engine, sub, 0.5, segs)
    assert n_sel == n_full


def test_select_keeps_the_vertex_id_base(engine):
    """A run with vert_id_base B numbers its vertices from B: the selection compacts in that range, so it gives the
    base-0 selection's mesh with every triangle id shifted by B."""
    from contourist_b200 import engine as E
    from contourist_b200 import tetrahedral
    n, B = 30, 1000
    x, y, z = np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing="ij")
    f = np.exp(-((x - 8) ** 2 + (y - 9) ** 2 + (z - 10) ** 2) / 12.0) + \
        np.exp(-((x - 21) ** 2 + (y - 20) ** 2 + (z - 19) ** 2) / 10.0)
    start = tetrahedral.initial_voxels(f, 0.5, [[(8, 9, 10), (8, 9, 0)]])
    flags = E.WANT_KEYS | E.WANT_NORMALS | E.GEOM_F64
    out = []
    for base in (0, B):
        full = engine.mt3d_run(f, 0.5, flags=flags, vert_id_base=base)
        nv, nt, _ = engine.mt3d_select_seeded(start)
        assert 0 < nt < int(full.n_tris)                        # the second blob is dropped
        out.append(engine.mt3d_fetch())
    a, b = out
    for k in ("verts", "normals", "keys", "lowmin"):
        assert np.array_equal(a[k], b[k])
    assert b["tris"].min() >= B
    assert np.array_equal(b["tris"], a["tris"] + B)


def test_facade_two_dots_seeded_is_the_reference_known_answer(engine):
    """test_tetrahedral.py:13-37 at the grid level: only the seeded dot comes back (minus the two leak triangles)."""
    from contourist_b200 import tetrahedral

    def two_dots(i, j, k):
        return 1 if (i == j == k == 0 or i == j == k == 4) else -1
    G = tetrahedral.Grid3DContour(8, 8, 8, two_dots, 0, [[(0, 0, 0), (0, 0, 8)]])
    pts, tris = G.get_points_and_triangles()
    world = [tuple(int(c) for c in (-8 + 2 * np.asarray(p))) for p in pts]
    got = set(frozenset(world[i] for i in t) for t in tris)
    assert got == {frozenset([(-7, -8, -8), (-7, -8, -7), (-7, -7, -7)]), frozenset([(-8, -8, -7), (-8, -7, -7), (-7, -7, -7)]),
                   frozenset([(-8, -8, -7), (-7, -8, -7), (-7, -7, -7)]), frozenset([(-8, -7, -8), (-7, -7, -8), (-7, -7, -7)]),
                   frozenset([(-7, -8, -8), (-7, -7, -8), (-7, -7, -7)]), frozenset([(-8, -7, -8), (-8, -7, -7), (-7, -7, -7)])}
    full = tetrahedral.Grid3DContour(8, 8, 8, two_dots, 0, None)
    assert len(full.get_points_and_triangles()[1]) > len(tris)
    # orientation after selection still works on the compacted mesh
    G.reference_orientation = True
    assert len(G.get_points_and_triangles()[1]) == len(tris)


def test_select_needs_a_full_volume_run(engine):
    from contourist_b200 import engine as E
    f = np.random.default_rng(0).standard_normal((12, 12, 12))
    engine.mt3d_run(f, 0.0, i_lo=0, i_hi=6)
    with pytest.raises(E.EngineError):
        engine.mt3d_select_seeded(np.zeros((1, 3), np.int32))


FILES2D = sorted(glob.glob(os.path.join(GOLDEN, "seeded2d_*.npz")))


@pytest.mark.parametrize("path", FILES2D, ids=[os.path.basename(f) for f in FILES2D])
def test_2d_reference_seeded_runs(engine, path):
    """Grid2DContour with explicit seeds returns the contours the reference's tracker finds (triangulated.py:307-338),
    not the full scan: same pairs as the reference run, same polylines as point sets."""
    from contourist_b200 import triangulated
    from oracle import mt2d
    g = np.load(path)
    field, z = g["field"], float(g["value"])
    seeds = [[tuple(a), tuple(b)] for a, b in g["seeds"].tolist()]
    G = triangulated.Grid2DContour(field.shape[0], field.shape[1], field, z, seeds)
    got = G.get_contour_sequences()
    want_keys = mt2d.seeded_keys(field, z, g["seeds"])
    assert np.array_equal(np.unique(G.segments["keys"]), want_keys)
    assert sorted(len(p) for _, p in got) == sorted(g["length"].tolist())
    assert sorted(bool(c) for c, _ in got) == sorted(bool(c) for c in g["closed"])
    mine = sorted(map(tuple, np.round(np.concatenate([p for _, p in got]), 9).tolist()))
    ref = sorted(map(tuple, np.round(g["pts"], 9).tolist()))
    assert mine == ref
    full = triangulated.Grid2DContour(field.shape[0], field.shape[1], field, z, None).get_contour_sequences()
    assert len(full) > len(got)


def test_2d_world_seeds_through_the_driver(engine):
    """DxDy2DContour with world-coordinate seeds (triangulated.py:92-118): only the dot the seed points at.  (With
    the dots of test_triangulated.py:44-68 the tracker hops from one to the other: they share the low point (1,1).)"""
    from contourist_b200 import triangulated

    def two_dots(x, y):
        return 1 if (x == y == -4 or x == y == 2) else -1
    C = triangulated.DxDy2DContour(-4, -4, 4, 4, 2, 2, two_dots, 0, [[(2, 2), (4, 2)]])
    contours = C.get_contour_sequences()
    assert len(contours) == 1 and contours[0][0]
    pts = sorted((int(round(x * 10)), int(round(y * 10))) for x, y in contours[0][1])
    assert pts == sorted([(20, 30), (30, 30), (30, 20), (20, 10), (10, 10), (10, 20)])
    assert len(triangulated.DxDy2DContour(-4, -4, 4, 4, 2, 2, two_dots, 0).get_contour_sequences()) == 2
    # the reference's own two dots share a low point: its tracker returns both from one seed
    def near_dots(x, y):
        return 1 if (x == y == -4 or x == y == 0) else -1
    assert len(triangulated.DxDy2DContour(-4, -4, 4, 4, 2, 2, near_dots, 0, [[(0, 0), (4, 0)]]).get_contour_sequences()) == 2
