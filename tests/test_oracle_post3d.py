"""CPU: oracle/post3d.py (quantize -> tiny -> clean, made deterministic) against final meshes produced by the unmodified
reference's own quantize_interpolations / remove_tiny_simplices / extract_points_and_triangles on the same raw state
(tests/golden/make_golden.py post -> tests/golden/post3d_*.npz; tetrahedral.py:541-552).

The reference's result depends on CPython dict / set iteration order in three places (which interpolation of a quantum
survives, which point a collapsed simplex merges to, clean_triangles' vertex_map).  What is order-free is compared
exactly; the rest is compared in quantum-cell space (positions truncated to the quantize grid, where the choice of a
quantum's survivor is invisible) and the per-fixture residue is stated below.
"""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, c1_golden
from oracle import post3d
from test_oracle_golden_3d import golden_keys

FILES = sorted(glob.glob(os.path.join(GOLDEN, "post3d_*.npz")))

# fixture -> (triangles that differ as exact position triples, triangles that differ in quantum-cell space);
# both counted on the reference's side.  0 / 0 = identical geometric sets.
RESIDUE = {
    "c1": (0, 0),              # BASELINE configs[0]: 57 456 triangles / 28 730 points, identical
    "ints7": (0, 0),
    "noise8": (0, 0),
    "wave11": (0, 0),
    "plateau6": (126, 0),      # 49 simplices merged by quantize: the survivor of a quantum differs, cells do not
    "sphere13": (152, 92),     # 12 collapsed tiny simplices: the merge point is `points[0]` of a frozenset
    "gyroid33": (372, 180),    # 96 collapsed tiny simplices sharing vertices: sequential overwrite vs cluster merge
}


def load(path):
    g = dict(np.load(path))
    if "final_idx" in g:                       # final points stored as rows of the raw interpolations
        g["final_points"] = g["key_pos"][g.pop("final_idx")]
    if "field" not in g:
        g["field"] = c1_golden()["field"]
    for k in ("key_low", "key_high", "tris", "final_tris"):
        g[k] = g[k].astype(np.int64)
    return g


def tri_set(points, tris):
    return set(tuple(sorted(tuple(points[i]) for i in t)) for t in tris)


def run(g):
    shape = g["field"].shape
    keys, _ = golden_keys(g)
    rank = post3d.engine_rank(keys, shape)
    corner = np.array(shape) - 1
    return corner, post3d.postprocess(g["key_pos"], g["tris"], corner, rank)


def test_have_fixtures():
    assert len(FILES) >= 7


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f)[7:-4] for f in FILES])
def test_postprocess_matches_reference(path):
    name = os.path.basename(path)[7:-4]
    g = load(path)
    corner, r = run(g)
    n_raw = len(g["tris"])
    # the passes remove the same number of simplices as the reference's (order-free quantities)
    assert n_raw - r["n_quantized"] == int(g["n_after_quantize"])
    assert n_raw - r["n_quantized"] - r["n_tiny"] == int(g["n_after_tiny"])
    assert r["n_tiny"] == int(g["collapsed"])
    exact_res, cell_res = RESIDUE[name]
    ours, ref = tri_set(r["points"], r["tris"]), tri_set(g["final_points"], g["final_tris"])
    assert len(ref - ours) <= exact_res
    expander = (10000.0 / corner).astype(np.int64)
    qa, qb = (r["points"] * expander).astype(np.int64), (g["final_points"] * expander).astype(np.int64)
    ours_q, ref_q = tri_set(qa, r["tris"]), tri_set(qb, g["final_tris"])
    assert len(ref_q - ours_q) <= cell_res
    if exact_res == 0:
        assert ours == ref and len(r["tris"]) == len(g["final_tris"])
        assert set(map(tuple, r["points"])) == set(map(tuple, g["final_points"]))
        assert len(r["points"]) == len(g["final_points"])
    if cell_res == 0:
        assert ours_q == ref_q and len(r["tris"]) == len(g["final_tris"])
    # every final point is a raw interpolation (the passes move or drop vertices, never invent positions)
    raw = set(map(tuple, g["key_pos"]))
    assert set(map(tuple, r["points"])) <= raw


def test_c1_final_counts():
    """SURVEY.md 8(d) C1: the reference's final mesh of the 65^3 sphere."""
    g = load(os.path.join(GOLDEN, "post3d_c1.npz"))
    _, r = run(g)
    assert (len(r["points"]), len(r["tris"])) == (28730, 57456)


def test_engine_rank_is_word_direction_k():
    shape = (3, 2, 70)
    lin = np.array([5, 40, 33, 5, 69 + 70], dtype=np.uint64)
    d = np.array([3, 1, 1, 1, 2], dtype=np.uint64)
    keys = (lin << np.uint64(3)) | d
    # words (W = 3): 5 -> word 0, 40 / 33 -> word 1, 139 -> row 1, k 69 -> word 5
    assert post3d.engine_rank(keys, shape).tolist() == [1, 3, 2, 0, 4]


def test_transform_applied_last():
    g = load(os.path.join(GOLDEN, "post3d_ints7.npz"))
    shape = g["field"].shape
    keys, _ = golden_keys(g)
    rank = post3d.engine_rank(keys, shape)
    corner = np.array(shape) - 1
    a = post3d.postprocess(g["key_pos"], g["tris"], corner, rank)
    b = post3d.postprocess(g["key_pos"], g["tris"], corner, rank, mins=(-1.0, 2.0, 0.5), delta=(0.25, 0.5, 2.0))
    assert np.array_equal(a["tris"], b["tris"])
    assert np.array_equal(b["points"], a["points"] * np.array([0.25, 0.5, 2.0]) + np.array([-1.0, 2.0, 0.5]))
