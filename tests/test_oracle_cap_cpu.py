"""CPU: oracle/mt3d_cap.py:cap (the definition of ctr_mt3d_cap) against a naive per-face-triangle restatement, on
analytic fields whose capped regions have known volumes, and on fields whose capped meshes must be closed; the layout
of ctr_cap_params / ctr_cap_counts (no GPU here)."""
import ctypes

import numpy as np
import pytest

from oracle import mt3d, mt3d_cap


def engine_mesh(field, value, geom_dtype=np.float64, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), normals=True):
    """oracle/mt3d.extract's mesh as the engine's fetch gives it: every triangle wound towards the high side (the
    direction low -> high along its vertices' edges), positions in world coordinates, keys, lowmin, normals."""
    r = mt3d.extract(field, value, geom_dtype)
    t = r["tris"].astype(np.int64).copy()
    pmin, pmax = mt3d.key_points(r["keys"], field.shape)
    up = np.where(r["lowmin"][:, None] == 1, pmax - pmin, pmin - pmax).astype(np.float64)
    P = r["pos"].astype(np.float64)
    fn = np.cross(P[t[:, 1]] - P[t[:, 0]], P[t[:, 2]] - P[t[:, 0]])
    flip = (fn * (up[t[:, 0]] + up[t[:, 1]] + up[t[:, 2]])).sum(axis=1) < 0
    t[flip] = t[flip][:, ::-1]
    gd = np.dtype(geom_dtype)
    pos = np.empty_like(r["pos"])
    for a in range(3):
        pos[:, a] = r["pos"][:, a] * gd.type(delta[a]) + gd.type(origin[a])
    out = dict(verts=pos, tris=t.astype(np.int32), keys=r["keys"], lowmin=r["lowmin"], normals=None)
    if normals:
        out["normals"] = mt3d.normals(field, value, r["keys"], geom_dtype, delta)
    return out


def naive_cap(mesh, field, value, side, origin, delta, geom_dtype):
    """The definition restated one face triangle at a time, with a dict of keys and vertices made on first use."""
    side = mt3d_cap.SIDES[side]
    shape = field.shape
    gd = np.dtype(geom_dtype)
    n1, n2 = shape[1], shape[2]
    lin = lambda p: (p[0] * n1 + p[1]) * n2 + p[2]
    index = {int(k): i for i, k in enumerate(mesh["keys"])}
    low = lambda p: float(field[tuple(p)]) < value
    tris, used, missing = [], set(), 0
    for axis, hi, a, b in mt3d_cap.faces(shape):
        ea, eb = np.eye(3, dtype=np.int64)[a], np.eye(3, dtype=np.int64)[b]
        for u in range(shape[a] - 1):
            for w in range(shape[b] - 1):
                m = np.zeros(3, np.int64)
                m[axis], m[a], m[b] = (shape[axis] - 1 if hi else 0), u, w
                for t in range(2):
                    C = [m, m + (ea if t == 0 else eb), m + ea + eb]
                    on = [low(c) == (side == mt3d_cap.LOW) for c in C]
                    poly, ok = [], True
                    for i in range(3):
                        j = (i + 1) % 3
                        if on[i]:
                            poly.append(("p", lin(C[i])))
                        if on[i] != on[j]:
                            lo = np.minimum(C[i], C[j])
                            d = np.abs(C[j] - C[i])
                            k = lin(lo) * 8 + int(d[0] * 4 + d[1] * 2 + d[2])
                            ok = ok and k in index
                            poly.append(("v", index.get(k, -1)))
                    if not poly:
                        continue
                    if not ok:
                        missing += 1
                        continue
                    # the cap faces into the box for HIGH, out of it for LOW; T0 turns like e_a x e_b, T1 the other way
                    outward = 1 if hi else -1
                    want = -outward if side == mt3d_cap.HIGH else outward
                    nat = np.cross(C[1] - C[0], C[2] - C[0])[axis]
                    for k in range(1, len(poly) - 1):
                        tri = [poly[0], poly[k], poly[k + 1]]
                        if nat * want < 0:
                            tri = [tri[0], tri[2], tri[1]]
                        tris.append(tri)
                        used.update(x[1] for x in tri if x[0] == "p")
    pts = sorted(used)
    nV = len(mesh["keys"])
    ids = {p: nV + i for i, p in enumerate(pts)}
    T = np.array([[x[1] if x[0] == "v" else ids[x[1]] for x in tri] for tri in tris], np.int64).reshape(-1, 3)
    P = np.array([(p // (n1 * n2), (p // n2) % n1, p % n2) for p in pts], np.int64).reshape(-1, 3)
    pos = np.array([[gd.type(P[i, x]) * gd.type(delta[x]) + gd.type(origin[x]) for x in range(3)] for i in range(len(P))],
                   gd).reshape(-1, 3)
    nrm = np.zeros((len(P), 3))
    for i, p in enumerate(P):
        for axis, hi, a, b in mt3d_cap.faces(shape):
            if p[axis] == (shape[axis] - 1 if hi else 0):
                g = np.zeros(3)
                g[axis] = (1.0 if hi else -1.0) * (-1.0 if side == mt3d_cap.HIGH else 1.0)
                e = np.zeros(3)                         # two in-face vectors, in world coordinates
                e[a] = delta[a]
                f = np.zeros(3)
                f[b] = delta[b]
                wn = np.cross(e, f) * np.sign(np.cross(np.eye(3)[a], np.eye(3)[b])[axis] * g[axis])
                nrm[i] += wn / np.linalg.norm(wn)
    nrm = nrm / np.linalg.norm(nrm, axis=1)[:, None] if len(nrm) else nrm
    return dict(tris=T, pts=np.array(pts, np.int64), pos=pos, normals=nrm, lowmin=np.array([low(p) for p in P], np.uint8),
                n_missing=missing)


def directed_edges_closed(tris):
    """every directed edge of the mesh appears once and its reverse once: closed and consistently wound"""
    T = np.asarray(tris, np.int64)
    e = np.concatenate([T[:, [0, 1]], T[:, [1, 2]], T[:, [2, 0]]])
    code = e[:, 0] * (T.max() + 1) + e[:, 1]
    rev = e[:, 1] * (T.max() + 1) + e[:, 0]
    u, c = np.unique(code, return_counts=True)
    return bool((c == 1).all()) and np.array_equal(np.sort(code), np.sort(rev))


def signed_volume(verts, tris):
    P = np.asarray(verts, np.float64)
    T = np.asarray(tris, np.int64)
    a, b, c = P[T[:, 0]], P[T[:, 1]], P[T[:, 2]]
    return float((a * np.cross(b, c)).sum() / 6.0)


@pytest.mark.parametrize("geom_dtype", [np.float64, np.float32])
@pytest.mark.parametrize("side", ["high", "low"])
def test_oracle_matches_naive_restatement(geom_dtype, side):
    rng = np.random.default_rng(5 if side == "high" else 6)
    for shape, origin, delta in [((5, 6, 7), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
                                 ((4, 3, 6), (0.25, -1.5, 3.0), (0.5, -0.75, 2.0)),
                                 ((2, 5, 2), (1.0, 2.0, -3.0), (-1.0, 0.3, 0.7))]:
        field = rng.standard_normal(shape)
        value = 0.1
        mesh = engine_mesh(field, value, geom_dtype, origin, delta)
        got, cnt = mt3d_cap.cap(mesh, field, value, side, origin, delta, geom_dtype)
        want = naive_cap(mesh, field, value, side, origin, delta, geom_dtype)
        nV, nT = len(mesh["keys"]), len(mesh["tris"])
        assert cnt == dict(n_verts=nV + len(want["pts"]), n_tris=nT + len(want["tris"]), n_cap_verts=len(want["pts"]),
                           n_cap_tris=len(want["tris"]), n_missing=want["n_missing"])
        assert np.array_equal(got["tris"][:nT], mesh["tris"]) and np.array_equal(got["tris"][nT:], want["tris"])
        assert np.array_equal(got["keys"][nV:], (want["pts"] * 8).astype(np.uint64))
        assert np.array_equal(got["verts"][:nV], mesh["verts"]) and got["verts"].dtype == np.dtype(geom_dtype)
        assert got["verts"][nV:].tobytes() == want["pos"].tobytes()
        assert np.array_equal(got["lowmin"][nV:], want["lowmin"])
        assert np.array_equal(got["normals"][:nV], mesh["normals"])
        assert np.allclose(got["normals"][nV:], want["normals"], rtol=0, atol=1e-6)


def box_halfspace_volume(c, a, L):
    """volume of {a . x <= c} in the box [0, L]^3 for a > 0 (inclusion-exclusion over the box corners)"""
    tot = 0.0
    for v in np.ndindex(2, 2, 2):
        s = c - float(np.dot(a, np.array(v) * L))
        tot += (-1) ** sum(v) * max(s, 0.0) ** 3
    return tot / (6.0 * a[0] * a[1] * a[2])


def test_linear_field_volume():
    n = 11
    L = n - 1
    x = np.arange(n, dtype=np.float64)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    field = X + 0.3 * Y - 0.2 * Z
    value = 4.3141
    mesh = engine_mesh(field, value)
    hi, ch = mt3d_cap.cap(mesh, field, value, "high")
    lo, cl = mt3d_cap.cap(mesh, field, value, "low")
    assert ch["n_missing"] == cl["n_missing"] == 0
    assert directed_edges_closed(hi["tris"]) and directed_edges_closed(lo["tris"])
    # f >= v  <=>  x' + 0.3 y' + 0.2 z <= L + 0.3 L - v  with x' = L - x, y' = L - y
    v_high = box_halfspace_volume(1.3 * L - value, np.array([1.0, 0.3, 0.2]), L)
    assert abs(-signed_volume(hi["verts"], hi["tris"]) - v_high) <= 1e-12 * v_high
    assert abs(signed_volume(lo["verts"], lo["tris"]) - (L ** 3 - v_high)) <= 1e-12 * L ** 3


def test_all_high_field():
    shape = (4, 5, 7)
    field = np.full(shape, 2.0)
    mesh = engine_mesh(field, 1.0)
    assert len(mesh["tris"]) == 0
    hi, ch = mt3d_cap.cap(mesh, field, 1.0, "high")
    n0, n1, n2 = shape
    assert ch["n_cap_tris"] == 4 * ((n0 - 1) * (n1 - 1) + (n0 - 1) * (n2 - 1) + (n1 - 1) * (n2 - 1))
    assert ch["n_cap_verts"] == n0 * n1 * n2 - (n0 - 2) * (n1 - 2) * (n2 - 2)
    assert directed_edges_closed(hi["tris"])
    assert abs(-signed_volume(hi["verts"], hi["tris"]) - (n0 - 1) * (n1 - 1) * (n2 - 1)) < 1e-9
    assert (hi["lowmin"] == 0).all() and (hi["keys"] % 8 == 0).all()
    lo, cl = mt3d_cap.cap(mesh, field, 1.0, "low")
    assert cl == dict(n_verts=0, n_tris=0, n_cap_verts=0, n_cap_tris=0, n_missing=0)


def corner_ball(n):
    x = np.arange(n, dtype=np.float64)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return X * X + Y * Y + Z * Z


@pytest.mark.parametrize("case", ["corner_ball", "random"])
def test_closed_and_volume_identity(case):
    if case == "corner_ball":
        field, value = corner_ball(12), 7.3 ** 2
        origin, delta = (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)
    else:
        field = np.random.default_rng(9).standard_normal((7, 8, 9))
        value = 0.0123
        origin, delta = (-1.0, 0.5, 2.0), (0.5, 0.25, 1.5)
    assert np.abs(field - value).min() > 1e-4                 # no sample within allclose of the isovalue
    mesh = engine_mesh(field, value, origin=origin, delta=delta)
    hi, ch = mt3d_cap.cap(mesh, field, value, "high", origin, delta)
    lo, cl = mt3d_cap.cap(mesh, field, value, "low", origin, delta)
    assert ch["n_missing"] == cl["n_missing"] == 0 and ch["n_cap_tris"] > 0 and cl["n_cap_tris"] > 0
    assert directed_edges_closed(hi["tris"]) and directed_edges_closed(lo["tris"])
    box = float(np.prod((np.array(field.shape) - 1) * np.array(delta)))
    diff = signed_volume(lo["verts"], lo["tris"]) - signed_volume(hi["verts"], hi["tris"])
    assert abs(diff - box) <= 1e-9 * box


def test_skipped_tets_count_as_missing():
    rng = np.random.default_rng(2)
    field = rng.standard_normal((5, 6, 5))
    field[:2] = 0.5 + rng.choice([-1e-9, 1e-9], size=(2, 6, 5))     # the first voxel layer: every tet skipped by allclose
    mesh = engine_mesh(field, 0.5)
    for side in ("high", "low"):
        got, c = mt3d_cap.cap(mesh, field, 0.5, side)
        want = naive_cap(mesh, field, 0.5, side, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), np.float64)
        assert c["n_missing"] == want["n_missing"] > 0
        assert np.array_equal(got["tris"][len(mesh["tris"]):], want["tris"])


def test_abi_layout():
    from contourist_b200 import engine as E
    assert ctypes.sizeof(E.CapParams) == 8 and ctypes.sizeof(E.CapCounts) == 40
    assert E.CAP_SIDES == {"high": mt3d_cap.HIGH, "low": mt3d_cap.LOW}
