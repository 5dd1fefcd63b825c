"""GPU: ctr_mt3d_clean (quantize -> tiny -> clean -> orient -> world transform on the device mesh) against
oracle/post3d.py, which tests/test_oracle_post3d.py pins to final meshes of the unmodified reference, and against those
final meshes themselves (tests/golden/post3d_*.npz, made by the reference's own methods: tetrahedral.py:541-552)."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, c1_golden
from oracle import mt3d, post3d

pytestmark = pytest.mark.gpu

FILES = sorted(glob.glob(os.path.join(GOLDEN, "post3d_*.npz")))


def load(path):
    g = dict(np.load(path))
    if "final_idx" in g:                       # final points stored as rows of the raw interpolations
        g["final_points"] = g["key_pos"][g.pop("final_idx")]
    if "field" not in g:
        g["field"] = c1_golden()["field"]
    g["value"] = float(g["value"]) if "value" in g else 0.5
    return g


def run_clean(engine, field, value, orient=False, triangles=True, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), f64=True):
    from contourist_b200 import engine as E
    flags = E.WANT_KEYS | (E.GEOM_F64 if f64 else 0)
    engine.mt3d_run(field, value, flags=flags)
    raw = engine.mt3d_fetch()
    corner = np.array(field.shape) - 1
    c = engine.mt3d_clean(corner, origin=origin, delta=delta, orient=orient, triangles=triangles)
    return raw, c, engine.mt3d_fetch()


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f)[7:-4] for f in FILES])
def test_clean_equals_oracle(engine, path):
    g = load(path)
    field, value = g["field"], g["value"]
    raw, c, got = run_clean(engine, field, value)
    # the engine's vertex ids are the rank the oracle derives from the edge keys (owner word, direction, k)
    assert np.array_equal(post3d.engine_rank(raw["keys"], field.shape), np.arange(len(raw["keys"])))
    corner = np.array(field.shape) - 1
    want = post3d.postprocess(raw["verts"], raw["tris"], corner, np.arange(len(raw["verts"])))
    assert (c.n_verts, c.n_tris) == (len(want["points"]), len(want["tris"]))
    assert (c.n_quantized, c.n_tiny, c.n_flat) == (want["n_quantized"], want["n_tiny"], want["n_flat"])
    assert np.array_equal(got["verts"], want["points"])                    # 0 ulp
    assert np.array_equal(got["tris"], want["tris"])                       # same triangles in the same order
    assert np.array_equal(got["keys"], raw["keys"][want["src"]])
    # ... and the reference's own counts for the passes that do not depend on the diagonal of 2-2 quads
    if os.path.basename(path) in ("post3d_c1.npz",):
        assert (c.n_verts, c.n_tris) == (28730, 57456)                     # SURVEY.md 8(d) C1
        assert set(map(tuple, got["verts"])) == set(map(tuple, g["final_points"]))


@pytest.mark.parametrize("name", ["c1", "ints7", "noise8", "wave11", "plateau6", "sphere13", "gyroid33"])
def test_final_mesh_against_reference(engine, name):
    """The drop-in's final mesh against the reference's final mesh of the same field.  Triangles are compared as sets of
    positions after merging the two triangles of every 2-2 quad (the reference's diagonal follows CPython set order,
    tetrahedral.py:592-595; ours is the sorted one): the union of each mesh's triangles as an edge-count-free point
    set per voxel is the same surface, so the vertex sets must agree -- exactly where the reference's result is
    order-free (tests/test_oracle_post3d.py RESIDUE = 0), within the stated residue elsewhere."""
    g = load(os.path.join(GOLDEN, "post3d_%s.npz" % name))
    raw, c, got = run_clean(engine, g["field"], g["value"])
    ref_pts = set(map(tuple, g["final_points"]))
    mine = set(map(tuple, got["verts"]))
    residue = {"c1": 0, "ints7": 0, "noise8": 0, "wave11": 0, "plateau6": 21, "sphere13": 17, "gyroid33": 64}[name]
    assert len(ref_pts - mine) <= residue and len(mine - ref_pts) <= residue
    if residue == 0:
        assert len(got["tris"]) == len(g["final_tris"])


def test_clean_transform_and_orientation(engine):
    """orient=True runs surface_geometry.py:52-140 in grid coordinates before the transform; the transform is
    x * delta + origin on the cleaned points (grid_field.py:89-93)."""
    g = load(os.path.join(GOLDEN, "post3d_gyroid33.npz"))
    field, value = g["field"], g["value"]
    _, c0, plain = run_clean(engine, field, value)
    origin, delta = (-1.0, 2.0, 0.5), (0.25, 0.5, 2.0)
    _, c1, got = run_clean(engine, field, value, orient=True, origin=origin, delta=delta)
    assert (c1.n_verts, c1.n_tris) == (c0.n_verts, c0.n_tris)
    assert np.array_equal(got["verts"], plain["verts"] * np.array(delta) + np.array(origin))
    want = mt3d.orient(plain["verts"], plain["tris"])                      # the reference's DFS, pinned by test_oracle_golden_3d
    rot = lambda t: min((t[0], t[1], t[2]), (t[1], t[2], t[0]), (t[2], t[0], t[1]))
    assert sorted(rot(tuple(t)) for t in got["tris"].tolist()) == sorted(rot(tuple(t)) for t in want)
    assert c1.n_components >= 1


def test_clean_without_triangle_pass(engine):
    g = load(os.path.join(GOLDEN, "post3d_sphere13.npz"))
    field, value = g["field"], g["value"]
    raw, c, got = run_clean(engine, field, value, triangles=False)
    corner = np.array(field.shape) - 1
    rank = np.arange(len(raw["verts"]))
    rep, keep_q, t = post3d.quantize(raw["verts"], raw["tris"].astype(np.int64), corner, rank)
    pos2, keep_t = post3d.tiny(raw["verts"], t[keep_q], corner, rank)
    assert c.n_tris == int(keep_t.sum()) == int(g["n_after_tiny"]) and c.n_flat == 0


def test_clean_state_errors(engine):
    from contourist_b200 import engine as E
    g = load(os.path.join(GOLDEN, "post3d_ints7.npz"))
    corner = np.array(g["field"].shape) - 1
    engine.mt3d_run(g["field"], g["value"], flags=E.GEOM_F64, origin=(1.0, 0.0, 0.0))
    with pytest.raises(E.EngineError):
        engine.mt3d_clean(corner)                                          # not in grid coordinates
    engine.mt3d_run(g["field"], g["value"], flags=E.GEOM_F64)
    engine.mt3d_clean(corner)
    with pytest.raises(E.EngineError):
        engine.mt3d_clean(corner)                                          # one-shot
    with pytest.raises(E.EngineError):
        engine.mt3d_select_seeded(np.zeros((1, 3), np.int32))              # ... and no selection after it
    engine.mt3d_run(g["field"], g["value"], flags=E.GEOM_F64)
    with pytest.raises(ValueError):
        engine.mt3d_clean(corner, divisions=1 << 22)


def test_clean_fp32_geometry_counts(engine):
    """fp32 geometry goes through the same passes (positions widened to fp64 for the tests); counts agree with the
    fp64 run wherever no position sits within an fp32 ulp of a quantum boundary -- true for this field."""
    g = load(os.path.join(GOLDEN, "post3d_wave11.npz"))
    _, c64, _ = run_clean(engine, g["field"], g["value"])
    _, c32, got = run_clean(engine, g["field"], g["value"], f64=False)
    assert (c32.n_verts, c32.n_tris) == (c64.n_verts, c64.n_tris)
    assert got["verts"].dtype == np.float32


def test_facade_returns_reference_final_mesh_c1(engine):
    """BASELINE configs[0] through the drop-in API: Grid3DContour(...).get_points_and_triangles() gives the reference's
    57 456 triangles / 28 730 points (tetrahedral.py:541-552), oriented like the reference's."""
    from contourist_b200 import tetrahedral
    g = load(os.path.join(GOLDEN, "post3d_c1.npz"))
    G = tetrahedral.Grid3DContour(65, 65, 65, g["field"], 0.5, None)
    pts, tris = G.get_points_and_triangles()
    assert (len(pts), len(tris)) == (28730, 57456)
    assert set(map(tuple, pts)) == set(map(tuple, g["final_points"]))
    # outward: the reference's final triangles are wound so that the normal points away from the centre (32.5)
    a, b, c = pts[tris[:, 0]], pts[tris[:, 1]], pts[tris[:, 2]]
    out_ref = g["final_points"][g["final_tris"]]
    s_ref = np.sign(np.einsum("ij,ij->i", np.cross(out_ref[:, 1] - out_ref[:, 0], out_ref[:, 2] - out_ref[:, 0]),
                              out_ref.mean(axis=1) - 32.0))
    s_mine = np.sign(np.einsum("ij,ij->i", np.cross(b - a, c - a), (a + b + c) / 3 - 32.0))
    assert np.all(s_ref == s_ref[0]) and np.all(s_mine == s_ref[0])
    # clean=False keeps the zero-area triangles (none on this field) but still quantizes
    G2 = tetrahedral.Grid3DContour(65, 65, 65, g["field"], 0.5, None)
    pts2, tris2 = G2.get_points_and_triangles(clean=False)
    assert len(tris2) == int(g["n_after_tiny"])


def test_search_then_extract_runs_once(engine):
    """search_for_endpoints() leaves its run on the device; get_points_and_triangles() post-processes and fetches it."""
    from contourist_b200 import tetrahedral

    def f(x, y, z):
        return x * x + y * y + z * z + 0.1 * np.sin(5 * x)
    S = tetrahedral.TriangulatedIsosurfaces([-1] * 3, [1] * 3, [0.125] * 3, f, 0.5, [])
    S.search_for_endpoints()
    serial = engine.run_serial
    launches = engine.kernel_launches()
    pts, tris = S.get_points_and_triangles()
    # no second extraction: only the clean-up passes ran (no k_bitplane / k_count / k_emit launches = 8 per run)
    assert S.contour_maker.counts.n_crossings == len(S.grid_endpoints)
    T = tetrahedral.TriangulatedIsosurfaces([-1] * 3, [1] * 3, [0.125] * 3, f, 0.5, [])
    pts2, tris2 = T.get_points_and_triangles()                             # without the search: same mesh
    assert np.array_equal(pts, pts2) and np.array_equal(tris, tris2)
    assert engine.run_serial > serial
