"""Generate golden vectors by running the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

The reference is driven through its own public classes (Grid3DContour, GridContour4D,
Multiple2DContourGrid) with an array-backed callable; the raw state is captured after the
reference's own enumerate step and before its post-processing, then its post-processing is
run by calling the reference's own methods in the reference's own order
(tetrahedral.py:528-552, pentatopes.py:101-125).  See ref_harness.py for the py2->py3 shim.
"""
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as rh  # noqa: E402


def array_callable(arr):
    shape = arr.shape

    def f(*idx):
        ii = tuple(min(max(int(i), 0), n - 1) for i, n in zip(idx, shape))
        return float(arr[ii])
    return f


def strict_seeds(arr, value):
    """grid_field.py:64-84 restated vectorised ONLY to feed seeds to the reference engine
    (the reference's own scan needs a FunctionGrid; results are identical, see test)."""
    d = arr.ndim
    n = [s - 1 for s in arr.shape]
    base = arr[tuple(slice(0, k) for k in n)].astype(np.float64) - value
    seeds = []
    for c in range(1, 2 ** d):
        off = [(c >> (d - 1 - a)) & 1 for a in range(d)]
        nb = arr[tuple(slice(o, k + o) for o, k in zip(off, n))].astype(np.float64) - value
        idx = np.argwhere(base * nb < 0)
        for p in idx:
            seeds.append((tuple(int(x) for x in p), tuple(int(x) + o for x, o in zip(p, off))))
    return seeds


# ------------------------------------------------------------------ 3D
def fields3d():
    out = {}
    n = 13
    g = np.linspace(-1, 1, n)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    out["sphere13"] = (X * X + Y * Y + Z * Z, 0.5)
    out["wave11"] = (np.sin(3.1 * X[:11, :11, :11] + 0.3) * np.cos(2.3 * Y[:11, :11, :11]) + 0.7 * Z[:11, :11, :11] ** 2
                     + 0.25 * np.sin(5 * Z[:11, :11, :11] * X[:11, :11, :11]), 0.2)
    rng = np.random.default_rng(7)
    out["noise8"] = (rng.standard_normal((8, 7, 9)).astype(np.float32).astype(np.float64), 0.1)
    out["ints7"] = (rng.integers(-1, 2, size=(7, 7, 7)).astype(np.float64), 0.0)
    plate = 0.3 + 1e-7 * rng.standard_normal((6, 6, 6))
    plate[3:, :, :] += 0.4 * rng.standard_normal((3, 6, 6))
    out["plateau6"] = (plate, 0.3)
    return out


def run3d(arr, value):
    T = rh.load("tetrahedral")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    seeds = strict_seeds(arr, value)
    t0 = time.time()
    G = T.Grid3DContour(corner[0], corner[1], corner[2], f, value, seeds)
    # tetrahedral.py:535-540
    G.find_initial_voxels()
    while G.new_surface_voxels:
        G.expand_voxels()
    for triple in G.surface_voxels:
        G.enumerate_voxel_triangles(triple)
    corner_a = np.array(corner)
    vox = np.array(sorted(v for v in G.surface_voxels
                          if all(0 <= v[a] < corner[a] for a in range(3))), dtype=np.int64).reshape(-1, 3)
    n_leak = len(G.surface_voxels) - len(vox)
    pairs = list(G.interpolated_contour_pairs.keys())
    simplices = []
    for s in G.simplex_sets:
        pts = np.array([p for pair in s for p in pair])
        owner = pts.min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a):
            simplices.append(sorted(s))
    simplices = sorted(simplices)
    used = sorted(set(pair for s in simplices for pair in s))
    raw_low = np.array([p[0] for p in used], dtype=np.int64).reshape(-1, 3)
    raw_high = np.array([p[1] for p in used], dtype=np.int64).reshape(-1, 3)
    raw_pos = np.array([G.interpolated_contour_pairs[p] for p in used], dtype=np.float64).reshape(-1, 3)
    kidx = {p: i for i, p in enumerate(used)}
    raw_tris = np.array([[kidx[p] for p in s] for s in simplices], dtype=np.int64).reshape(-1, 3)
    # tetrahedral.py:541-552 (reference post-processing, its own code)
    G.quantize_interpolations()
    G.remove_tiny_simplices()
    pts, tris = G.extract_points_and_triangles(True)
    dt = time.time() - t0
    fin_pts = np.array(pts, dtype=np.float64).reshape(-1, 3)
    fin_tris = np.array(tris, dtype=np.int64).reshape(-1, 3)
    return dict(field=arr, value=np.float64(value), voxels=vox, n_leak=np.int64(n_leak),
                key_low=raw_low, key_high=raw_high, key_pos=raw_pos, tris=raw_tris,
                final_points=fin_pts, final_tris=fin_tris, n_seeds=np.int64(len(seeds)),
                seconds=np.float64(dt))


def c1_field():
    """BASELINE configs[0] (SURVEY.md 8(d) C1): f = x^2+y^2+z^2 on [-1,1]^3, delta 1/32 -> N = 65 voxels per axis read
    samples 0..65 (tetrahedral.py:465-469), value 0.5 -- the one config the full reference runs (about a minute)."""
    g = -1.0 + np.arange(66) / 32.0
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    return X * X + Y * Y + Z * Z, 0.5


def fields_seeded():
    """Multi-component fields with explicit seed segments (SURVEY.md 8(f3)): the reference's tracker must return only
    the components its seeds reach."""
    out = {}
    def two_dots(x, y, z):
        return 1.0 if (x == y == z == -8 or x == y == z == 0) else -1.0
    arr = np.array([[[two_dots(-8 + 2 * i, -8 + 2 * j, -8 + 2 * k) for k in range(10)] for j in range(10)] for i in range(10)])
    out["twodots"] = (arr, 0.0, [[(4, 4, 4), (4, 4, 9)]])               # from the dot at the origin (grid 4,4,4) outwards
    n = 18
    x, y, z = np.meshgrid(*(np.arange(n, dtype=np.float64),) * 3, indexing="ij")
    blobs = np.zeros((n, n, n))
    for c, r in (((4.3, 4.1, 4.6), 2.6), ((12.2, 5.1, 4.9), 2.2), ((5.2, 12.4, 11.8), 2.9), ((12.6, 12.3, 12.1), 2.4)):
        blobs += np.exp(-((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2) / (r * r))
    out["blobs_one"] = (blobs, 0.45, [[(4, 4, 4), (4, 4, 9)]])
    out["blobs_two"] = (blobs, 0.45, [[(12, 5, 5), (12, 9, 5)], [(16, 16, 16), (12, 12, 12)], [(12, 5, 5), (16, 5, 5)]])
    wave = np.sin(0.9 * x + 0.3) * np.cos(0.7 * y) + 0.05 * (z - 8)
    out["wave_sheet"] = (wave, 0.1, [[(0, 8, 8), (5, 8, 8)]])
    return out


def run_seeded(arr, value, seeds):
    T = rh.load("tetrahedral")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    G = T.Grid3DContour(corner[0], corner[1], corner[2], f, value, seeds)
    G.find_initial_voxels()                              # tetrahedral.py:396-441
    initial = sorted(G.new_surface_voxels)
    while G.new_surface_voxels:
        G.expand_voxels()                                # tetrahedral.py:443-463
    for triple in G.surface_voxels:
        G.enumerate_voxel_triangles(triple)
    inr = lambda v: all(0 <= v[a] < corner[a] for a in range(3))
    vox = np.array(sorted(v for v in G.surface_voxels if inr(v)), dtype=np.int64).reshape(-1, 3)
    corner_a = np.array(corner)
    simplices = []
    for s in G.simplex_sets:
        pts = np.array([p for pair in s for p in pair])
        owner = pts.min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a):
            simplices.append(sorted(s))
    used = sorted(set(pair for s in simplices for pair in s))
    return dict(field=arr, value=np.float64(value), seeds=np.array(seeds, dtype=np.int64).reshape(-1, 2, 3),
                initial=np.array(initial, dtype=np.int64).reshape(-1, 3), voxels=vox,
                n_leak=np.int64(len(G.surface_voxels) - len(vox)), n_keys=np.int64(len(used)), n_tris=np.int64(len(simplices)),
                key_low=np.array([p[0] for p in used], dtype=np.int64).reshape(-1, 3),
                key_high=np.array([p[1] for p in used], dtype=np.int64).reshape(-1, 3))


def run_clean(path):
    """surface_geometry.py:14-50 clean_triangles of the unmodified reference on the raw mesh of a 3D golden."""
    RS = rh.load("surface_geometry")
    g = np.load(path)
    geometry = RS.SurfaceGeometry([p for p in g["key_pos"]], [frozenset(int(i) for i in t) for t in g["tris"]])
    verts, tris = geometry.clean_triangles()
    full = sorted(tuple(sorted(t)) for t in tris if len(t) == 3)
    return dict(vertices=np.array(verts, dtype=np.float64).reshape(-1, 3), triangles=np.array(full, dtype=np.int32).reshape(-1, 3),
                n_degenerate=np.int64(sum(1 for t in tris if len(t) < 3)))


def run_post(arr, value, stages=False):
    """tetrahedral.py:541-552 of the unmodified reference -- quantize_interpolations, remove_tiny_simplices,
    extract_points_and_triangles (clean_triangles + orient_triangles) -- on the IN-RANGE raw state (the simplices owned
    by voxels with origin in [0, N-1], the parity domain of the engine: DESIGN.md section 2), by calling the reference's
    own methods in the reference's own order on its own object.  `raw_*` is that state in the numbering of the mt3d_*
    goldens (sorted pairs), so a restatement can start from exactly what the reference started from."""
    T = rh.load("tetrahedral")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    seeds = strict_seeds(arr, value)
    G = T.Grid3DContour(corner[0], corner[1], corner[2], f, value, seeds)
    G.find_initial_voxels()
    while G.new_surface_voxels:
        G.expand_voxels()
    for triple in G.surface_voxels:
        G.enumerate_voxel_triangles(triple)
    corner_a = np.array(corner)
    keep = set()
    for s in G.simplex_sets:
        owner = np.array([p for pair in s for p in pair]).min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a):
            keep.add(s)
    G.simplex_sets = keep
    used = sorted(set(pair for s in keep for pair in s))
    G.interpolated_contour_pairs = {pair: G.interpolated_contour_pairs[pair] for pair in used}
    kidx = {p: i for i, p in enumerate(used)}
    raw_low = np.array([p[0] for p in used], dtype=np.int64).reshape(-1, 3)
    raw_high = np.array([p[1] for p in used], dtype=np.int64).reshape(-1, 3)
    raw_pos = np.array([G.interpolated_contour_pairs[p] for p in used], dtype=np.float64).reshape(-1, 3)
    raw_tris = np.array(sorted(sorted(kidx[p] for p in s) for s in keep), dtype=np.int64).reshape(-1, 3)
    G.quantize_interpolations()
    n_after_q = len(G.simplex_sets)
    G.remove_tiny_simplices()
    n_after_t = len(G.simplex_sets)
    pts, tris = G.extract_points_and_triangles(True)
    return dict(field=arr, value=np.float64(value), key_low=raw_low, key_high=raw_high, key_pos=raw_pos, tris=raw_tris,
                final_points=np.array(pts, dtype=np.float64).reshape(-1, 3),
                final_tris=np.array(tris, dtype=np.int64).reshape(-1, 3),
                n_after_quantize=np.int64(n_after_q), n_after_tiny=np.int64(n_after_t),
                collapsed=np.int64(G.collapsed_simplices))


def main():
    which = sys.argv[1:] or ["3d"]
    if "clean" in which:
        for name in ("sphere13", "wave11", "noise8", "ints7", "plateau6"):
            g = run_clean(os.path.join(HERE, "mt3d_%s.npz" % name))
            np.savez_compressed(os.path.join(HERE, "clean3d_%s.npz" % name), **g)
            print(name, "vertices", len(g["vertices"]), "triangles", len(g["triangles"]), "two-vertex leftovers", int(g["n_degenerate"]))
    if "post" in which:
        todo = dict(fields3d())
        todo["c1"] = c1_field()
        g32 = np.linspace(-1.0, 1.0, 33)
        X, Y, Z = np.meshgrid(g32, g32, g32, indexing="ij")
        todo["gyroid33"] = (np.sin(4 * X) * np.cos(4 * Y) + np.sin(4 * Y) * np.cos(4 * Z) + np.sin(4 * Z) * np.cos(4 * X), 0.0)
        for name, (arr, value) in todo.items():
            g = run_post(arr, value)
            if name in ("c1",):
                g.pop("field")                         # conftest.c1_golden regenerates it from the formula
            for k in ("key_low", "key_high"):
                g[k] = g[k].astype(np.int16)
            g["tris"] = g["tris"].astype(np.int32)
            g["final_tris"] = g["final_tris"].astype(np.int32)
            # every final point is one of the raw interpolations: stored as its row in key_pos, which keeps the
            # files under 1 MB (the tests' load() maps the rows back to positions)
            first = {}
            for i, p in enumerate(map(tuple, g["key_pos"])):
                first.setdefault(p, i)
            final_points = g.pop("final_points")
            g["final_idx"] = np.array([first[tuple(p)] for p in final_points], dtype=np.int32)
            np.savez_compressed(os.path.join(HERE, "post3d_%s.npz" % name), **g)
            print(name, arr.shape, "raw", len(g["key_pos"]), len(g["tris"]), "after quantize", int(g["n_after_quantize"]),
                  "after tiny", int(g["n_after_tiny"]), "final", final_points.shape, g["final_tris"].shape)
    if "seeded" in which:
        for name, (arr, value, seeds) in fields_seeded().items():
            g = run_seeded(arr, value, seeds)
            np.savez_compressed(os.path.join(HERE, "seeded3d_%s.npz" % name), **g)
            print(name, arr.shape, "initial", g["initial"].tolist(), "voxels", len(g["voxels"]), "leak", int(g["n_leak"]),
                  "keys", int(g["n_keys"]), "tris", int(g["n_tris"]))
    if "c1" in which:
        arr, value = c1_field()
        g = run3d(arr, value)
        g.pop("field")                                 # regenerated by the tests from the formula above (conftest.c1_field)
        g["n_final_points"] = np.int64(len(g.pop("final_points")))
        g["n_final_tris"] = np.int64(len(g.pop("final_tris")))
        for k in ("voxels", "key_low", "key_high"):
            g[k] = g[k].astype(np.int16)
        g["tris"] = g["tris"].astype(np.int32)
        np.savez_compressed(os.path.join(HERE, "c1_sphere65.npz"), **g)
        print("c1", arr.shape, "voxels", len(g["voxels"]), "leak", int(g["n_leak"]), "keys", len(g["key_low"]),
              "tris", len(g["tris"]), "final", int(g["n_final_points"]), int(g["n_final_tris"]), "%.1fs" % g["seconds"])
    if "3d" in which:
        for name, (arr, value) in fields3d().items():
            g = run3d(arr, value)
            np.savez_compressed(os.path.join(HERE, "mt3d_%s.npz" % name), **g)
            print(name, arr.shape, "voxels", len(g["voxels"]), "leak", int(g["n_leak"]), "keys", len(g["key_low"]),
                  "tris", len(g["tris"]), "final", g["final_points"].shape, g["final_tris"].shape,
                  "%.1fs" % g["seconds"])


if __name__ == "__main__":
    main()


# ------------------------------------------------------------------ 2D
def fields2d():
    out = {}
    n = 21
    g = np.linspace(-2, 2, n)
    X, Y = np.meshgrid(g, g, indexing="ij")
    out["osc21"] = (np.sqrt(np.sin(3 * X + Y * Y) ** 2 + np.cos(4 * Y + X * X) ** 2), [0.3, 0.6, 0.9, 1.2])
    rng = np.random.default_rng(5)
    out["noise"] = (rng.standard_normal((12, 15)), [-0.5, 0.0, 0.7])
    out["ints"] = (rng.integers(0, 4, size=(9, 11)).astype(np.float64), [0.5, 1.0, 2.0])
    return out


def run2d(arr, levels):
    M = rh.load("multiple_2d_contour")
    T = rh.load("triangulated")
    G = rh.load("grid_field")
    n0, n1 = arr.shape

    def f(x, y):
        return float(arr[min(max(int(round(x)), 0), n0 - 1), min(max(int(round(y)), 0), n1 - 1)])
    grid = G.FunctionGrid((0, 0), (n0 - 1, n1 - 1), (1, 1), f)
    assert tuple(grid.grid_dimensions) == (n0, n1)
    C = M.Multiple2DContourGrid(grid, levels)
    t0 = time.time()
    # multiple_2d_contour.py:17-30, keeping each level's contour maker so its raw state can be read
    C.classify_endpoints()
    out = dict(field=arr, levels=np.array(sorted(levels), dtype=np.float64))
    for li, value in enumerate(sorted(C.value_to_endpoints)):
        endpoints = C.value_to_endpoints[value]
        try:
            cm = T.DxDy2DContourGrid(grid, value, endpoints)
            seqs = cm.get_contour_sequences()
        except AssertionError as e:
            print("   level", value, "reference assertion:", e)
            out["L%d_failed" % li] = np.int64(1)
            continue
        pairs = sorted(cm.contour_maker.interpolated_contour_pairs.keys())
        out["L%d_low" % li] = np.array([p[0] for p in pairs], dtype=np.int64).reshape(-1, 2)
        out["L%d_high" % li] = np.array([p[1] for p in pairs], dtype=np.int64).reshape(-1, 2)
        out["L%d_pos" % li] = np.array([cm.contour_maker.interpolated_contour_pairs[p] for p in pairs],
                                       dtype=np.float64).reshape(-1, 2)
        out["L%d_closed" % li] = np.array([c for c, _ in cm.grid_contours], dtype=np.int64)
        out["L%d_len" % li] = np.array([len(p) for _, p in cm.grid_contours], dtype=np.int64)
        out["L%d_pts" % li] = (np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 2) for _, p in cm.grid_contours])
                               if cm.grid_contours else np.zeros((0, 2)))
        trip = sorted(sorted(t) for t in cm.contour_maker.triangle_triples)
        out["L%d_triples" % li] = np.array(trip, dtype=np.int64).reshape(-1, 3, 2)
    out["seconds"] = np.float64(time.time() - t0)
    return out


def fields_seeded2d():
    """2D fields with several contours of one level and explicit seed segments: the reference's tracker
    (triangulated.py:307-338) must return only the contours its seeds reach."""
    n = 24
    x, y = np.meshgrid(np.arange(n, dtype=np.float64), np.arange(n, dtype=np.float64), indexing="ij")
    bumps = np.zeros((n, n))
    for c, r in (((5.3, 5.2), 3.1), ((17.4, 6.1), 2.7), ((6.2, 17.3), 3.4), ((17.6, 17.2), 2.9)):
        bumps += np.exp(-((x - c[0]) ** 2 + (y - c[1]) ** 2) / (r * r))
    out = {}
    out["bumps_one"] = (bumps, 0.5, [[(5, 5), (5, 11)]])
    out["bumps_two"] = (bumps, 0.5, [[(17, 6), (23, 6)], [(12, 12), (18, 17)]])
    ints = np.random.default_rng(3).integers(-2, 3, size=(14, 15)).astype(np.float64)
    ints[4:10, 4:11] = -2.0
    ints[6:8, 6:9] = 2.0
    out["ints_island"] = (ints, 0.0, [[(6, 6), (6, 4)]])
    return out


def run_seeded2d(arr, value, seeds):
    T = rh.load("triangulated")
    n0, n1 = arr.shape

    def f(i, j):
        return float(arr[min(max(int(i), 0), n0 - 1), min(max(int(j), 0), n1 - 1)])
    G = T.Grid2DContour(n0, n1, f, value, [[np.array(a), np.array(b)] for a, b in seeds])
    seqs = G.get_contour_sequences()                      # triangulated.py:221-293 (search, expand, chain)
    pairs = sorted(G.interpolated_contour_pairs.keys())
    return dict(field=arr, value=np.float64(value), seeds=np.array(seeds, dtype=np.int64).reshape(-1, 2, 2),
                low=np.array([p[0] for p in pairs], dtype=np.int64).reshape(-1, 2),
                high=np.array([p[1] for p in pairs], dtype=np.int64).reshape(-1, 2),
                closed=np.array([c for c, _ in seqs], dtype=np.int64), length=np.array([len(p) for _, p in seqs], dtype=np.int64),
                pts=(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 2) for _, p in seqs]) if seqs else np.zeros((0, 2))))


def main2d():
    for name, (arr, levels) in fields2d().items():
        g = run2d(arr, levels)
        np.savez_compressed(os.path.join(HERE, "mt2d_%s.npz" % name), **g)
        print(name, arr.shape, [(k, g[k].shape) for k in sorted(g) if k.endswith("_low")], "%.1fs" % g["seconds"])


def main_seeded2d():
    for name, (arr, value, seeds) in fields_seeded2d().items():
        g = run_seeded2d(arr, value, seeds)
        np.savez_compressed(os.path.join(HERE, "seeded2d_%s.npz" % name), **g)
        print(name, arr.shape, "pairs", len(g["low"]), "contours", len(g["closed"]), g["closed"].tolist(), g["length"].tolist())


if __name__ == "__main__" and "2d" in sys.argv[1:]:
    main2d()
if __name__ == "__main__" and "seeded2d" in sys.argv[1:]:
    main_seeded2d()


# ------------------------------------------------------------------ 4D
def fields4d():
    out = {}
    n, nt = 7, 4
    g = np.linspace(-2, 2, n)
    t = np.linspace(0, 1, nt)
    X, Y, Z, T_ = np.meshgrid(g, g, g, t, indexing="ij")
    bar = 3 * np.sqrt(X * X + Z * Z)
    g2 = 3 * np.sqrt((1 - np.sqrt(X * X + Y * Y)) ** 2 + Z * Z)
    out["morph7"] = (T_ * bar + (1 - T_) * g2, 1.2)
    rng = np.random.default_rng(13)
    out["noise4"] = (rng.standard_normal((4, 3, 4, 3)), 0.2)
    out["ints4"] = (rng.integers(-1, 2, size=(3, 4, 3, 4)).astype(np.float64), 0.0)
    return out


def run4d(arr, value):
    P = rh.load("pentatopes")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    seeds = strict_seeds(arr, value)
    t0 = time.time()
    G = P.GridContour4D(corner, f, value, seeds)
    # pentatopes.py:101-106
    G.find_initial_voxels()
    while G.new_surface_voxels:
        G.expand_voxels()
    for quad in G.surface_voxels:
        G.enumerate_voxel_tetrahedra(quad)
    corner_a = np.array(corner)
    vox = np.array(sorted(v for v in G.surface_voxels if all(0 <= v[a] < corner[a] for a in range(4))),
                   dtype=np.int64).reshape(-1, 4)
    simplices = []
    for s in G.simplex_sets:
        pts = np.array([p for pair in s for p in pair])
        owner = pts.min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a):
            simplices.append(sorted(s))
    simplices = sorted(simplices)
    used = sorted(set(pair for s in simplices for pair in s))
    raw_low = np.array([p[0] for p in used], dtype=np.int64).reshape(-1, 4)
    raw_high = np.array([p[1] for p in used], dtype=np.int64).reshape(-1, 4)
    raw_pos = np.array([np.array(G.interpolated_contour_pairs[p]) for p in used], dtype=np.float64).reshape(-1, 4)
    kidx = {p: i for i, p in enumerate(used)}
    raw_tets = np.array([[kidx[p] for p in s] for s in simplices if len(s) == 4], dtype=np.int64).reshape(-1, 4)
    # restrict the reference's state to in-range simplices so its post-processing is comparable
    G.simplex_sets = set(frozenset(s) for s in simplices)
    G.interpolated_contour_pairs = {p: G.interpolated_contour_pairs[p] for p in used}
    # pentatopes.py:107-125 (not flatten, not smooth)
    import io
    import contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        G.bin_times()
        binned_pos = np.array([np.array(G.interpolated_contour_pairs[p]) for p in used], dtype=np.float64).reshape(-1, 4)
        G.drop_instant_tetrahedra()
        after_drop = sorted(sorted(kidx[p] for p in s) for s in G.simplex_sets)
        G.remove_tiny_simplices(epsilon=1e-3)
        after_tiny = sorted(sorted(kidx[p] for p in s) for s in G.simplex_sets)
        tiny_pos = np.array([np.array(G.interpolated_contour_pairs[p]) for p in used], dtype=np.float64).reshape(-1, 4)
        mt = G.collect_morph_triangles()
    # express the MorphTriangles in terms of the `used` key numbering
    order = list(G.interpolated_contour_pairs.keys())
    remap = np.array([kidx[p] for p in order], dtype=np.int64)
    segs = np.array([(remap[i], remap[j]) for (i, j) in mt.segment_point_indices], dtype=np.int64).reshape(-1, 2)
    tris = np.array([list(t) for t in mt.triangle_segment_indices], dtype=np.int64).reshape(-1, 3)
    dt = time.time() - t0
    return dict(field=arr, value=np.float64(value), voxels=vox, key_low=raw_low, key_high=raw_high, key_pos=raw_pos,
                tets=raw_tets, binned_pos=binned_pos, tets_after_drop=np.array(after_drop, dtype=np.int64).reshape(-1, 4),
                tets_after_tiny=np.array(after_tiny, dtype=np.int64).reshape(-1, 4), tiny_pos=tiny_pos,
                morph_points=np.array(mt.points4d)[np.argsort(remap)] if len(remap) else np.zeros((0, 4)),
                morph_segments=segs, morph_triangles=tris, n_seeds=np.int64(len(seeds)), seconds=np.float64(dt))


def main4d():
    for name, (arr, value) in fields4d().items():
        g = run4d(arr, value)
        np.savez_compressed(os.path.join(HERE, "mp4d_%s.npz" % name), **g)
        print(name, arr.shape, "voxels", len(g["voxels"]), "keys", len(g["key_low"]), "tets", len(g["tets"]),
              "after drop", len(g["tets_after_drop"]), "after tiny", len(g["tets_after_tiny"]),
              "morph", g["morph_segments"].shape, g["morph_triangles"].shape, "%.1fs" % g["seconds"])


def main_json4d():
    """morph_geometry.py:91-128: the unmodified reference's MorphTriangles.to_json on the morph arrays of a 4D golden."""
    import hashlib
    import json
    RM = rh.load("morph_geometry")
    out = {}
    for name in ("morph7",):
        g = np.load(os.path.join(HERE, "mp4d_%s.npz" % name))
        mt = RM.MorphTriangles([p for p in g["morph_points"]], [tuple(int(x) for x in s) for s in g["morph_segments"]],
                               [tuple(int(x) for x in t) for t in g["morph_triangles"]])
        text = mt.to_json()
        out[name] = {"sha256": hashlib.sha256(text.encode()).hexdigest(), "length": len(text), "head": text[:200]}
        print(name, out[name]["length"], out[name]["sha256"])
    with open(os.path.join(HERE, "mp4d_to_json.json"), "w") as f:
        json.dump(out, f, indent=1)
    # html_demo.py:133-161 emit_three_json of the unmodified reference on the final mesh of a 3D golden
    RH = rh.load("html_demo")

    class Holder(object):
        def __init__(self, p, t):
            self.p, self.t = p, t

        def get_points_and_triangles(self):
            return self.p, self.t
    out3 = {}
    for name in ("wave11", "sphere13"):
        g = np.load(os.path.join(HERE, "mt3d_%s.npz" % name))
        text = RH.emit_three_json(Holder([np.array(p) for p in g["final_points"]], [tuple(int(i) for i in t) for t in g["final_tris"]]))
        out3[name] = {"sha256": hashlib.sha256(text.encode()).hexdigest(), "length": len(text)}
        print(name, out3[name])
    with open(os.path.join(HERE, "mt3d_three_json.json"), "w") as f:
        json.dump(out3, f, indent=1)


if __name__ == "__main__" and "4d" in sys.argv[1:]:
    main4d()
if __name__ == "__main__" and "json4d" in sys.argv[1:]:
    main_json4d()


# ------------------------------------------------------------------ 4D seeded
def fields_seeded4d():
    """Two separate blobs in (x, y, z, t): explicit seeds reach one of them (SURVEY.md 8(f3) in 4D: pentatopes.py:92-106 with
    the 80-neighbourhood OFFSETS4D, pentatopes.py:32-39)."""
    n, nt = 9, 6
    x, y, z, t = np.meshgrid(np.arange(n, dtype=np.float64), np.arange(n, dtype=np.float64), np.arange(n, dtype=np.float64),
                             np.arange(nt, dtype=np.float64), indexing="ij")
    a = np.exp(-((x - 2.2) ** 2 + (y - 2.4) ** 2 + (z - 2.1) ** 2 + 0.6 * (t - 1.3) ** 2) / 2.5)
    b = np.exp(-((x - 6.1) ** 2 + (y - 5.8) ** 2 + (z - 6.3) ** 2 + 0.6 * (t - 3.6) ** 2) / 2.9)
    f = a + b
    return {"blobs_a": (f, 0.5, [[(2, 2, 2, 1), (2, 2, 7, 1)]]),
            "blobs_b": (f, 0.5, [[(6, 6, 6, 4), (0, 6, 6, 4)], [(6, 6, 6, 3), (6, 6, 0, 3)]]),
            "blobs_both": (f, 0.5, [[(2, 2, 2, 1), (2, 2, 7, 1)], [(6, 6, 6, 4), (0, 6, 6, 4)]])}


def run_seeded4d(arr, value, seeds):
    P = rh.load("pentatopes")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    G = P.GridContour4D(corner, f, value, seeds)
    G.find_initial_voxels()
    initial = sorted(G.new_surface_voxels)
    while G.new_surface_voxels:
        G.expand_voxels()
    for quad in G.surface_voxels:
        G.enumerate_voxel_tetrahedra(quad)
    inr = lambda v: all(0 <= v[a] < corner[a] for a in range(4))
    vox = np.array(sorted(v for v in G.surface_voxels if inr(v)), dtype=np.int64).reshape(-1, 4)
    corner_a = np.array(corner)
    simplices = []
    for s in G.simplex_sets:
        pts = np.array([p for pair in s for p in pair])
        owner = pts.min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a) and len(s) == 4:
            simplices.append(sorted(s))
    used = sorted(set(pair for s in simplices for pair in s))
    return dict(field=arr, value=np.float64(value), seeds=np.array(seeds, dtype=np.int64).reshape(-1, 2, 4),
                initial=np.array(initial, dtype=np.int64).reshape(-1, 4), voxels=vox,
                n_leak=np.int64(len(G.surface_voxels) - len(vox)), n_keys=np.int64(len(used)), n_tets=np.int64(len(simplices)),
                key_low=np.array([p[0] for p in used], dtype=np.int16).reshape(-1, 4),
                key_high=np.array([p[1] for p in used], dtype=np.int16).reshape(-1, 4))


if __name__ == "__main__" and "seeded4d" in sys.argv[1:]:
    for name, (arr, value, seeds) in fields_seeded4d().items():
        g = run_seeded4d(arr, value, seeds)
        np.savez_compressed(os.path.join(HERE, "seeded4d_%s.npz" % name), **g)
        print(name, arr.shape, "initial", g["initial"].tolist(), "voxels", len(g["voxels"]), "leak", int(g["n_leak"]),
              "keys", int(g["n_keys"]), "tets", int(g["n_tets"]))


# ------------------------------------------------------------------ 4D legacy "sequence of morphing triangularizations"
def run_seq4d(arr, value):
    """pentatopes.py:370-444 iterate_morph_geometry / json_data of the unmodified reference (the format misc/morph_sequence.js
    loads) on the in-range state of a 4D golden, after the reference's own find_tetrahedra post-processing."""
    import contextlib
    import io
    P = rh.load("pentatopes")
    f = array_callable(arr)
    corner = [s - 1 for s in arr.shape]
    G = P.GridContour4D(corner, f, value, strict_seeds(arr, value))
    G.find_initial_voxels()
    while G.new_surface_voxels:
        G.expand_voxels()
    for quad in G.surface_voxels:
        G.enumerate_voxel_tetrahedra(quad)
    corner_a = np.array(corner)
    simplices = []
    for s in G.simplex_sets:
        owner = np.array([p for pair in s for p in pair]).min(axis=0)
        if np.all(owner >= 0) and np.all(owner < corner_a):
            simplices.append(sorted(s))
    used = sorted(set(pair for s in simplices for pair in s))
    G.simplex_sets = set(frozenset(s) for s in simplices)
    G.interpolated_contour_pairs = {p: G.interpolated_contour_pairs[p] for p in used}
    with contextlib.redirect_stdout(io.StringIO()):
        G.bin_times()
        G.drop_instant_tetrahedra()
        G.remove_tiny_simplices(epsilon=1e-3)
        kidx = {p: i for i, p in enumerate(used)}
        pos = np.array([np.array(G.interpolated_contour_pairs[p]) for p in used], dtype=np.float64).reshape(-1, 4)
        tets = np.array(sorted(sorted(kidx[p] for p in s) for s in G.simplex_sets if len(s) == 4), dtype=np.int64).reshape(-1, 4)
        morphs = list(G.iterate_morph_geometry())
        data = [m.json_data(integral=True, lists_only=True) for m in morphs]
    out = dict(field=arr, value=np.float64(value), pos=pos, tets=tets,
               minmax=np.array([[d["min_value"], d["max_value"]] for d in data], dtype=np.float64).reshape(-1, 2),
               scale=np.array([d["scale"] for d in data], dtype=np.float64).reshape(-1, 3),
               shift=np.array([d["shift"] for d in data], dtype=np.float64).reshape(-1, 3),
               vert_off=np.cumsum([0] + [len(d["start_positions"]) for d in data]).astype(np.int64),
               tri_off=np.cumsum([0] + [len(d["triangles"]) for d in data]).astype(np.int64),
               start=np.concatenate([np.array(d["start_positions"], dtype=np.int32).reshape(-1, 3) for d in data]),
               end=np.concatenate([np.array(d["end_positions"], dtype=np.int32).reshape(-1, 3) for d in data]),
               tris=np.concatenate([np.array([list(t) for t in d["triangles"]], dtype=np.int32).reshape(-1, 3) for d in data]))
    return out


if __name__ == "__main__" and "seq4d" in sys.argv[1:]:
    for name in ("morph7",):
        arr, value = fields4d()[name]
        g = run_seq4d(arr, value)
        np.savez_compressed(os.path.join(HERE, "seq4d_%s.npz" % name), **g)
        print(name, "morphs", len(g["minmax"]), "vertices", int(g["vert_off"][-1]), "triangles", int(g["tri_off"][-1]))
