"""CPU: oracle/mt3d_section.py:section (the definition of ctr_mt3d_section) on hand-made meshes, on an analytic sphere
whose sections have known areas and lengths, and on a capped ball whose sections add up to its volume; the layout of
ctr_section_params / ctr_section_counts and the new C ABI symbols (no GPU here)."""
import ctypes

import numpy as np
import pytest

from oracle import mt3d, mt3d_cap, mt3d_components, mt3d_section
from test_oracle_cap_cpu import corner_ball, engine_mesh

TRI = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])


def test_one_triangle():
    r = mt3d_section.section(TRI, [[0, 1, 2]], (1.0, 0.0, 0.0), [0.5])
    assert r["plane"].tolist() == [0]
    # the walk 0 -> 1 -> 2 goes low -> high on {0, 1} (end) and high -> low on {1, 2} (start)
    assert r["edges"].tolist() == [[[1, 2], [0, 1]]]
    assert r["points"].tolist() == [[[0.5, 0.5, 0.0], [0.5, 0.0, 0.0]]]
    # along n x (0, 0, 1) = -y; the chain starts at the smaller end key {0, 1}, runs backwards, and is reversed
    (closed, consistent, pts, length, area), = r["polylines"][0]
    assert not closed and consistent
    assert pts.tolist() == [[0.5, 0.5, 0.0], [0.5, 0.0, 0.0]]
    assert length == 0.5 and area == 0.0
    assert r["start_keys"][0] == [(1 << 32) | 2] and not r["junction"].any()


def test_vertex_on_plane_is_high():
    r = mt3d_section.section(TRI, [[0, 1, 2]], (1.0, 0.0, 0.0), [1.0])
    # vertex 1 has s == 1.0: high, so both crossings have t = 1 and sit on it
    assert r["edges"].tolist() == [[[1, 2], [0, 1]]]
    assert r["points"].tolist() == [[TRI[1].tolist(), TRI[1].tolist()]]


def test_plane_that_misses():
    r = mt3d_section.section(TRI, [[0, 1, 2]], (0.0, 0.0, 1.0), [-1.0, 0.5])
    assert len(r["plane"]) == 0 and r["polylines"] == [[], []]


def strip(n, flip=False):
    "a strip of 2n triangles along +y in the plane z = 0, facing +z (or -z)"
    v = np.array([[x, j, 0.0] for j in range(n + 1) for x in (0.0, 1.0)])
    t = []
    for j in range(n):
        a, b, c, d = 2 * j, 2 * j + 1, 2 * j + 2, 2 * j + 3
        t += [[a, b, c], [b, d, c]]
    t = np.array(t)
    return v, (t[:, ::-1] if flip else t)


@pytest.mark.parametrize("flip", [False, True])
def test_open_strip_start_and_reversal(flip):
    v, t = strip(3, flip)
    r = mt3d_section.section(v, t, (1.0, 0.0, 0.0), [0.25, 0.75])
    assert r["plane"].tolist() == [0, 1] * 6
    for l, x in enumerate((0.25, 0.75)):
        (closed, consistent, pts, length, area), = r["polylines"][l]
        assert not closed and consistent and length == 3.0
        # along n x (face normal): -y facing +z, +y facing -z
        ys = pts[:, 1]
        assert np.allclose(pts[:, 0], x) and len(pts) == 7
        assert (ys[0], ys[-1]) == ((3.0, 0.0) if not flip else (0.0, 3.0))
        assert (np.diff(ys) < 0).all() if not flip else (np.diff(ys) > 0).all()
        # the start key is that of the first point: the chain's smaller end unless it was reversed
        sk = r["start_keys"][l][0]
        end_keys = {int(mt3d_section.edge_key(2 * j, 2 * j + 1)): j for j in (0, 3)}
        assert end_keys[sk] == int(round(ys[0]))


def test_wound_against_each_other_is_inconsistent():
    v = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 1.0, 0.0]])
    good = mt3d_section.section(v, [[0, 1, 2], [2, 1, 3]], (1.0, 0.0, 0.0), [0.5])
    bad = mt3d_section.section(v, [[0, 1, 2], [1, 2, 3]], (1.0, 0.0, 0.0), [0.5])
    (c0, k0, p0, _, _), = good["polylines"][0]
    (c1, k1, p1, _, _), = bad["polylines"][0]
    assert not c0 and k0 and len(p0) == 3
    assert not c1 and not k1 and len(p1) == 3
    assert np.array_equal(np.sort(p0, axis=0), np.sort(p1, axis=0))


def test_nonmanifold_edge_is_a_junction():
    v = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, -1.0, 0.0], [0.0, 0.0, 1.0], [3.0, 3.0, 0.0]])
    t = [[0, 1, 2], [1, 0, 3], [0, 1, 4], [1, 5, 2]]
    r = mt3d_section.section(v, t, (1.0, 0.0, 0.0), [0.5, 2.0])
    assert r["junction"].tolist() == [True, False]
    assert r["polylines"][0] is None and len(r["polylines"][1]) == 1
    assert r["plane"].tolist() == [0, 0, 0, 0, 1]          # the junction plane's segments are still returned


def sphere(n, r, bright):
    x = np.arange(n + 1, dtype=np.float64)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    f = (X - n / 2) ** 2 + (Y - n / 2) ** 2 + (Z - n / 2) ** 2 - r * r
    return -f if bright else f


@pytest.mark.parametrize("normal", [(0.0, 0.0, 1.0), (1.0, 2.0, 2.0)])
def test_sphere_sections(normal):
    n, rad = 32, 11.3                                                 # (no sample on the isovalue)
    mesh = engine_mesh(sphere(n, rad, bright=False), 0.0)            # inside low: the raw mesh faces outward
    u = np.asarray(normal) / np.linalg.norm(normal)
    c = float(np.dot(u, [n / 2] * 3)) * np.linalg.norm(normal)
    h = np.linspace(-0.8, 0.8, 9) * rad                               # heights along u
    offs = c + h * np.linalg.norm(normal)
    r = mt3d_section.section(mesh["verts"], mesh["tris"], normal, offs)
    assert not r["junction"].any()
    for l, z in enumerate(h):
        (closed, consistent, pts, length, area), = r["polylines"][l]
        assert closed and consistent
        rr = np.sqrt(rad * rad - z * z)
        assert abs(area / (np.pi * rr * rr) - 1) < 0.03
        assert abs(length / (2 * np.pi * rr) - 1) < 0.03
        assert np.allclose(pts @ u, z + np.dot(u, [n / 2] * 3), atol=1e-9)


def test_sign_follows_winding():
    n, rad = 24, 8.3
    mesh = engine_mesh(sphere(n, rad, bright=True), 0.0)             # a bright blob: the raw mesh faces inward
    offs = [n / 2 - 3.0, n / 2, n / 2 + 3.0]
    raw = mt3d_section.section(mesh["verts"], mesh["tris"], (0.0, 0.0, 1.0), offs)
    oriented = np.array(mt3d.orient(mesh["verts"], mesh["tris"]), np.int64)
    out = mt3d_section.section(mesh["verts"], oriented, (0.0, 0.0, 1.0), offs)
    for l in range(3):
        (_, k0, _, _, a0), = raw["polylines"][l]
        (_, k1, _, _, a1), = out["polylines"][l]
        assert k0 and k1 and a0 < 0 < a1 and np.isclose(a0, -a1, rtol=1e-12)


def test_capped_ball_sections_add_up_to_its_volume():
    field, value = corner_ball(14), 9.3 ** 2
    mesh = engine_mesh(field, value)
    capped, counts = mt3d_cap.cap(mesh, field, value, "low")          # the region f < value, closed by its caps
    assert counts["n_missing"] == 0
    _, tab = mt3d_components.components(capped["verts"], capped["tris"])
    assert len(tab) == 1 and tab[0]["n_boundary_edges"] == 0 and tab[0]["volume"] > 0
    offs = np.arange(9) + 0.5                                        # the ball reaches z = 9.3
    r = mt3d_section.section(capped["verts"], capped["tris"], (0.0, 0.0, 1.0), offs)
    total = 0.0
    for l in range(len(offs)):
        assert r["polylines"][l] and all(p[0] and p[1] for p in r["polylines"][l])
        total += sum(p[4] for p in r["polylines"][l])
    assert abs(total / tab[0]["volume"] - 1) < 0.01


def test_abi_layout():
    from contourist_b200 import engine as E
    assert ctypes.sizeof(E.SectionParams) == 40 and ctypes.sizeof(E.SectionCounts) == 32


def test_header_declares_section_api():
    from test_capi_symbols import declared_symbols
    syms = declared_symbols()
    for s in ("ctr_mt3d_section", "ctr_mt3d_section_segments_fetch", "ctr_mt3d_section_polylines_fetch"):
        assert s in syms
