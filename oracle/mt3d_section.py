"""ORACLE (test infrastructure, not product code) -- sections of a 3D triangle mesh with a stack of parallel planes.

An engine extension with no counterpart in the reference (VTK's vtkCutter on polydata does the same job): `section`
below is the DEFINITION that ctr_mt3d_section is tested against, parity UNPINNED by the reference, like
oracle/mt3d_components.py.  It is a pure function of a mesh, a normal and the plane offsets.
"""
import numpy as np


def edge_key(a, b):
    "key of the undirected edge {a, b}: min << 32 | max"
    a = np.asarray(a, np.int64)
    b = np.asarray(b, np.int64)
    return ((np.minimum(a, b) << 32) | np.maximum(a, b)).astype(np.uint64)


def sides(verts, normal):
    "s_v = (n0 x + n1 y) + n2 z in fp64 on the widened positions, every operation rounded on its own"
    p = np.asarray(verts).astype(np.float64)
    n = np.asarray(normal, np.float64)
    return (n[0] * p[:, 0] + n[1] * p[:, 1]) + n[2] * p[:, 2]


def segments(verts, tris, normal, offsets, geom_dtype=None):
    """The segments (plane [S] int32, edges [S, 2, 2] int32, points [S, 2, 3] geometry type), by triangle, then plane.
    A vertex is high for plane l when s_v >= offsets[l].  A triangle whose corners are not all on one side gives one
    segment: from the crossing on the edge its corner walk takes from high to low (start edge) to the crossing on the
    edge it takes from low to high.  The crossing on {a, b}, a the low end: t = (d - s_a) / (s_b - s_a),
    p = p_a + t * (p_b - p_a) per axis (multiply, then add), fp64, rounded once to the geometry type."""
    verts = np.asarray(verts)
    gd = np.dtype(geom_dtype or verts.dtype)
    tris = np.asarray(tris, np.int64).reshape(-1, 3)
    off = np.asarray(offsets, np.float64)
    if len(tris) and (tris.min() < 0 or tris.max() >= len(verts)):
        raise ValueError("triangle ids outside [0, n_verts)")
    s = sides(verts, normal)
    p = verts.astype(np.float64)
    st = s[tris]                                              # [T, 3]
    lo = np.searchsorted(off, st.min(axis=1), side="right")   # crossed: smin < d <= smax
    hi = np.searchsorted(off, st.max(axis=1), side="right")
    cnt = hi - lo
    S = int(cnt.sum())
    t = np.repeat(np.arange(len(tris)), cnt)
    first = np.cumsum(cnt) - cnt
    plane = (np.repeat(lo, cnt) + np.arange(S) - np.repeat(first, cnt)).astype(np.int64)
    d = off[plane]
    V, sv = tris[t], st[t]
    h = sv >= d[:, None]
    hn = np.roll(h, -1, axis=1)                               # the corner after each corner
    ks = np.argmax(h & ~hn, axis=1)
    ke = np.argmax(~h & hn, axis=1)
    r = np.arange(S)
    ends = [(V[r, (ks + 1) % 3], V[r, ks], sv[r, (ks + 1) % 3], sv[r, ks]),      # start edge: low end, high end
            (V[r, ke], V[r, (ke + 1) % 3], sv[r, ke], sv[r, (ke + 1) % 3])]      # end edge
    edges = np.empty((S, 2, 2), np.int32)
    points = np.empty((S, 2, 3), gd)
    for q, (a, b, sa, sb) in enumerate(ends):
        edges[:, q, 0] = np.minimum(a, b)
        edges[:, q, 1] = np.maximum(a, b)
        tt = (d - sa) / (sb - sa)
        points[:, q] = (p[a] + tt[:, None] * (p[b] - p[a])).astype(gd)
    return plane.astype(np.int32), edges, points


def measures(points, closed, normal):
    """(length, area) in fp64 from the points widened: length sum |p_{i+1} - p_i| (the closing segment too when
    closed), area 1/2 sum ((p_i - p_0) x (p_{i+1} - p_0)) . n / |n| (also for open polylines, where it encloses
    nothing)."""
    p = np.asarray(points).astype(np.float64)
    n = np.asarray(normal, np.float64)
    u = n / np.sqrt((n * n).sum())
    q = np.concatenate([p, p[:1]]) if closed else p
    dp = q[1:] - q[:-1]
    length = float(np.sqrt((dp * dp).sum(axis=1)).sum())
    a, b = p[:-1] - p[0], p[1:] - p[0]
    c = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                  a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)
    return length, float(0.5 * (c @ u).sum())


def section(verts, tris, normal, offsets, geom_dtype=None):
    """Sections of the mesh (verts [V, 3], tris [T, 3], wound as the engine winds them) with the planes
    {x : normal . x == offsets[l]} (parity UNPINNED by the reference -- engine definition, ctr_mt3d_section).
    Returns dict(plane, edges, points: the segments (see `segments`); junction [nplanes] bool; polylines: one list per
    plane of (closed, consistent, points [k, 3], length, area), open ones first, then by start key, or None for a
    junction plane; start_keys: the same lists of start keys).
      - The vertices of a polyline are the pairs (plane, undirected edge).  A plane where some vertex lies on three or
        more segments (a non-manifold edge) is a junction plane: none of its segments is chained.  A segment whose two
        crossing edges are one edge (a triangle with a repeated vertex) is not chained either.
      - An open chain starts at its smaller end key, a closed one at its smallest key and runs towards the smaller
        neighbour (edge key min << 32 | max; both neighbours equal -- two segments between the same two vertices --:
        along the smaller dart 2s + q, dart 2s + q leaving end q of segment s).
      - If the first segment then runs from its point 1 to its point 0 the polyline is reversed: an open one starts at
        its other end, a closed one keeps its point 0 and lists the rest in reverse order.
      - consistent: every segment runs from point i to point i + 1, the closing one included; start key: the edge key
        of point 0."""
    off = np.asarray(offsets, np.float64)
    plane, edges, points = segments(verts, tris, normal, offsets, geom_dtype)
    S = len(plane)
    nplanes = len(off)
    key = edge_key(edges[:, :, 0], edges[:, :, 1]).astype(np.int64)      # [S, 2]; < 2^63
    live = key[:, 0] != key[:, 1]
    # vertices: (plane, key) of the live segment ends; incidences (segment, end) per vertex
    ls = np.nonzero(live)[0]
    vp = np.repeat(plane[ls].astype(np.int64), 2)
    vk = key[ls].reshape(-1)
    uv, inv, deg = np.unique(np.stack([vp, vk], axis=1), axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    junction = np.zeros(nplanes, bool)
    junction[uv[deg >= 3, 0]] = True
    vert_of = np.full((S, 2), -1, np.int64)
    vert_of[ls] = inv.reshape(-1, 2)
    inc = [[] for _ in range(len(uv))]
    for s, q in zip(np.repeat(ls, 2).tolist(), [0, 1] * len(ls)):
        inc[vert_of[s, q]].append((s, q))
    vert_of = vert_of.tolist()
    keyl = key.tolist()
    used = np.zeros(S, bool)
    used[~live] = True
    used[junction[plane]] = True
    used = used.tolist()
    per_plane = [[] for _ in range(nplanes)]

    def walk(v, s, q):
        "darts (s, q) from vertex v along segment s until an end or back at the start"
        darts = []
        while True:
            used[s] = True
            darts.append((s, q))
            w = vert_of[s][1 - q]
            nxt = [(t, r) for (t, r) in inc[w] if t != s or r != 1 - q]
            if not nxt or used[nxt[0][0]]:
                return darts
            s, q = nxt[0]

    order = np.lexsort((uv[:, 1], uv[:, 0], deg != 1)).tolist()     # open ends first, in (plane, key) order
    for v in order:
        if junction[uv[v, 0]] or all(used[s] for s, _ in inc[v]):
            continue
        if deg[v] == 1:
            darts = walk(v, *inc[v][0])
            closed = False
        else:
            (s1, q1), (s2, q2) = inc[v]
            k1, k2 = keyl[s1][1 - q1], keyl[s2][1 - q2]
            first = (s1, q1) if (k1, 2 * s1 + q1) < (k2, 2 * s2 + q2) else (s2, q2)
            darts = walk(v, *first)
            closed = True
        idx = [darts[0][0] * 2 + darts[0][1]] + [s * 2 + 1 - q for s, q in (darts[:-1] if closed else darts)]
        pk = [keyl[i >> 1][i & 1] for i in idx]
        if darts[0][1] == 1:                                          # the first segment runs backwards
            idx = idx[::-1] if not closed else idx[:1] + idx[:0:-1]
            pk = pk[::-1] if not closed else pk[:1] + pk[:0:-1]
        consistent = all(q == darts[0][1] for _, q in darts)
        pts = points.reshape(-1, 3)[idx]
        length, area = measures(pts, closed, normal)
        per_plane[int(plane[darts[0][0]])].append((closed, consistent, pts, length, area, pk[0]))
    polylines, start_keys = [], []
    for l in range(nplanes):
        if junction[l]:
            polylines.append(None)
            start_keys.append(None)
            continue
        rows = sorted(per_plane[l], key=lambda r: (r[0], r[5]))
        polylines.append([r[:5] for r in rows])
        start_keys.append([r[5] for r in rows])
    return dict(plane=plane, edges=edges, points=points, junction=junction, polylines=polylines, start_keys=start_keys)
