"""ORACLE (test infrastructure, not product code) -- caps that close the 3D isosurface at the faces of the volume.

An engine extension: the reference leaves a surface cut by the volume's box open, so `cap` below is the DEFINITION
that ctr_mt3d_cap is tested against (parity UNPINNED by the reference).  It works on the engine's own fetched mesh
(positions, normals, triangles, keys, lowmin), the run's field and isovalue.

With the Kuhn decomposition every box face is triangulated along the min -> max diagonal of each face square: the face
square with minimum corner m and in-face axes a < b has the face triangles T0 = (m, m + e_a, m + e_a + e_b) and
T1 = (m, m + e_b, m + e_a + e_b), each a face of exactly one tetrahedron.  The surface's rim on a box face is the
marching-triangles contour of the face samples on those triangles, and its rim vertices are the surface's own crossing
vertices, found by edge key.
"""
import numpy as np

HIGH, LOW = 0, 1
SIDES = {"high": HIGH, "low": LOW}


def faces(shape):
    """The six box faces in the engine's order: (axis, hi, a, b) for axis 0 lo, axis 0 hi, ..., axis 2 hi; a < b are
    the in-face axes."""
    out = []
    for axis in range(3):
        a, b = [x for x in range(3) if x != axis]
        out.append((axis, False, a, b))
        out.append((axis, True, a, b))
    return out


def _lin(P, shape):
    return (P[..., 0] * shape[1] + P[..., 1]) * shape[2] + P[..., 2]


def _edge_key(P, Q, shape):
    """edge key lin(min endpoint) * 8 + d of the grid edge P-Q (one endpoint is component-wise below the other)"""
    lo = np.minimum(P, Q)
    d = np.abs(Q - P)
    return _lin(lo, shape) * 8 + d[..., 0] * 4 + d[..., 1] * 2 + d[..., 2]


def polygon(s):
    """Vertex tokens of the piece of a face triangle (c0, c1, c2) on the chosen side, s = on-side flags of the three
    corners: walking i = 0, 1, 2, corner i if it is on the side, then the crossing of edge (i, i+1 mod 3) if exactly
    one of its ends is.  ('c', i) is a corner, ('x', i, j) a crossing.  The tokens keep the cyclic order of
    (c0, c1, c2)."""
    out = []
    for i in range(3):
        j = (i + 1) % 3
        if s[i]:
            out.append(("c", i))
        if s[i] != s[j]:
            out.append(("x", i, j))
    return out


def fan(n):
    """The pieces of an n-gon p0..p(n-1): the fan (p0, p_k, p_k+1), k = 1 .. n-2 (one triangle, or two for the quad)"""
    return [(0, k, k + 1) for k in range(1, n - 1)]


def cap_normal_sign(axis, hi, side):
    """+1 / -1: the cap triangles of this face point along +e_axis / -e_axis in grid coordinates.  HIGH caps face into
    the box, LOW caps out of it."""
    out = 1 if hi else -1
    return -out if side == HIGH else out


def natural_sign(axis, t):
    """+1 / -1: cross(c1 - c0, c2 - c0) of face triangle t (0 or 1) points along +e_axis / -e_axis"""
    sigma = (1, -1, 1)[axis]                      # e_a x e_b = sigma e_axis for a < b
    return sigma if t == 0 else -sigma


def cap(mesh, field, value, side, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), geom_dtype=np.float64):
    """(capped mesh dict, counts) -- ctr_mt3d_cap's definition.

    mesh: dict with verts [V, 3], tris [T, 3], keys [V] uint64, lowmin [V] uint8 and optionally normals [V, 3], as
    the engine's fetch returns them (ids in [0, V)).  side: "high" / "low" or HIGH (0) / LOW (1).

      * Side.  HIGH closes the region f >= value ("not low"), LOW the region f < value; "low" is the strict f < value
        of the extraction, compared in float64.
      * Faces in the order of faces(); each face square (u over axis a, w over axis b, row-major) has the face
        triangles T0 and T1 of the module docstring.
      * Piece of a face triangle: its part on the chosen side, the polygon of polygon().  0 corners on the side:
        nothing; 3: the whole triangle; 1: the corner and its two crossings; 2: a quad.  The polygon is split by the
        fan from its first vertex in the walk order (fan()): for a quad (p0, p1, p2, p3) the pieces are (p0, p1, p2)
        and (p0, p2, p3).
      * Crossing vertices are the mesh vertices whose key is the in-face edge's key lin(min endpoint) * 8 + d.  When a
        needed key is not in the mesh the face triangle contributes nothing and counts in n_missing (the surface
        itself has a gap there, e.g. a tetrahedron skipped by allclose).
      * Winding: the surface's triangles face the high side, so HIGH caps face into the box and LOW caps out of it
        (in grid coordinates): every rim edge is then crossed in opposite directions by its surface triangle and its
        cap triangle.  A piece whose polygon order has the other orientation is written reversed, (p0, p_k+1, p_k).
      * New vertices: one per box-surface grid point that is a corner of some cap triangle (also on box edges and
        corners, so the faces share it), appended after the existing vertices in ascending key order; key
        lin * 8 + 0 (d = 0 names the grid point itself), lowmin 1 if the point is low, position
        (G)grid * (G)delta + (G)origin rounded per operation in the geometry type G, normal (when the mesh has
        normals) the normalised sum, over the box faces the point lies on, of the unit world normal of those faces'
        cap triangles.  Existing vertices keep their rows.
      * New triangles are appended after the existing ones, ordered by face, face square, face triangle, piece.

    Known cases that are not watertight: a face sample exactly equal to `value` gives a crossing vertex at ratio 1
    that is not merged with the cap's grid vertex at the same position; a skipped tetrahedron leaves a gap in the
    surface.  Otherwise every edge of the capped mesh is used exactly twice.

    counts: dict(n_verts, n_tris, n_cap_verts, n_cap_tris, n_missing)."""
    side = SIDES[side] if isinstance(side, str) else int(side)
    assert side in (HIGH, LOW)
    field = np.asarray(field)
    shape = field.shape
    gd = np.dtype(geom_dtype)
    value = float(value)
    verts = np.asarray(mesh["verts"])
    tris = np.asarray(mesh["tris"], np.int64).reshape(-1, 3)
    keys = np.asarray(mesh["keys"], np.uint64).astype(np.int64)
    nV, nT = len(verts), len(tris)
    order = np.argsort(keys, kind="stable")
    skeys = keys[order]

    def lookup(k):
        pos = np.searchsorted(skeys, k)
        pos = np.minimum(pos, max(len(skeys) - 1, 0))
        hit = (skeys[pos] == k) if len(skeys) else np.zeros(k.shape, bool)
        return np.where(hit, order[pos] if len(skeys) else -1, -1)

    low = field.astype(np.float64) < value
    pieces = []                                                      # per face: refs [Q, 2, 2, 3], valid [Q, 2, 2]
    n_missing = 0
    for axis, hi, a, b in faces(shape):
        na, nb = shape[a], shape[b]
        u, w = np.meshgrid(np.arange(na - 1), np.arange(nb - 1), indexing="ij")
        u, w = u.reshape(-1), w.reshape(-1)
        Q = len(u)
        m = np.zeros((Q, 3), np.int64)
        m[:, axis] = shape[axis] - 1 if hi else 0
        m[:, a] = u
        m[:, b] = w
        ea = np.zeros(3, np.int64)
        ea[a] = 1
        eb = np.zeros(3, np.int64)
        eb[b] = 1
        refs = np.zeros((Q, 2, 2, 3), np.int64)
        valid = np.zeros((Q, 2, 2), bool)
        for t in range(2):
            C = np.stack([m, m + (ea if t == 0 else eb), m + ea + eb], axis=1)          # [Q, 3 corners, 3]
            lowc = low[C[..., 0], C[..., 1], C[..., 2]]
            s = lowc if side == LOW else ~lowc
            flip = natural_sign(axis, t) != cap_normal_sign(axis, hi, side)
            pat = s[:, 0] * 1 + s[:, 1] * 2 + s[:, 2] * 4
            for code in range(1, 8):
                rows = np.nonzero(pat == code)[0]
                if not len(rows):
                    continue
                toks = polygon([(code >> i) & 1 for i in range(3)])
                ids = np.zeros((len(rows), len(toks)), np.int64)
                ok = np.ones(len(rows), bool)
                for q, tok in enumerate(toks):
                    if tok[0] == "c":
                        ids[:, q] = -(_lin(C[rows, tok[1]], shape) + 1)      # a grid point, numbered below
                    else:
                        vid = lookup(_edge_key(C[rows, tok[1]], C[rows, tok[2]], shape))
                        ok &= vid >= 0
                        ids[:, q] = vid
                n_missing += int((~ok).sum())
                for pc, (i0, i1, i2) in enumerate(fan(len(toks))):
                    tri = (i0, i2, i1) if flip else (i0, i1, i2)
                    refs[rows, t, pc] = ids[:, list(tri)]
                    valid[rows, t, pc] = ok
        pieces.append(refs[valid])
    new_refs = np.concatenate(pieces) if pieces else np.zeros((0, 3), np.int64)
    pts = np.unique(-new_refs[new_refs < 0] - 1)                     # lin of the used grid points, ascending
    new_tris = new_refs.copy()
    cm = new_refs < 0
    new_tris[cm] = nV + np.searchsorted(pts, -new_refs[cm] - 1)
    n1, n2 = shape[1], shape[2]
    P = np.stack([pts // (n1 * n2), (pts // n2) % n1, pts % n2], axis=1)
    origin = np.asarray(origin, np.float64)
    delta = np.asarray(delta, np.float64)
    new_pos = np.empty((len(pts), 3), gd)
    for ax in range(3):
        new_pos[:, ax] = P[:, ax].astype(gd) * gd.type(delta[ax]) + gd.type(origin[ax])
    out = dict(mesh)
    out["verts"] = np.concatenate([verts, new_pos]).astype(verts.dtype if nV else gd)
    out["tris"] = np.concatenate([tris, new_tris]).astype(np.int32)
    out["keys"] = np.concatenate([np.asarray(mesh["keys"], np.uint64), (pts * 8).astype(np.uint64)])
    out["lowmin"] = np.concatenate([np.asarray(mesh["lowmin"], np.uint8),
                                    low[P[:, 0], P[:, 1], P[:, 2]].astype(np.uint8)])
    if mesh.get("normals") is not None:
        nrm = np.zeros((len(pts), 3), gd)
        dsgn = np.sign(delta)
        for axis, hi, a, b in faces(shape):
            on = P[:, axis] == (shape[axis] - 1 if hi else 0)
            nrm[on, axis] += gd.type(cap_normal_sign(axis, hi, side) * dsgn[a] * dsgn[b])
        ln = np.sqrt((nrm * nrm).sum(axis=1))
        out["normals"] = np.concatenate([np.asarray(mesh["normals"]), (nrm / ln[:, None]).astype(gd)])
    counts = dict(n_verts=nV + len(pts), n_tris=nT + len(new_tris), n_cap_verts=len(pts), n_cap_tris=len(new_tris),
                  n_missing=n_missing)
    return out, counts
