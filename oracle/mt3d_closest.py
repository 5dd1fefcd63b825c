"""ORACLE (test infrastructure, not product code) -- closest points on a 3D triangle mesh to query points.

An engine extension with no counterpart in the reference: `closest` below is the DEFINITION that ctr_mt3d_closest is
tested against, parity UNPINNED by the reference, like oracle/mt3d_clip.py.  It is a pure function of a mesh (as the
engine's fetch returns it), the query points and a distance limit.  Every operation is one separately rounded fp64
operation in a fixed order, so the device result equals it bit for bit.
"""
import numpy as np


def _sub(x, y):
    return (x[0] - y[0], x[1] - y[1], x[2] - y[2])


def _dot(x, y):
    return (x[0] * y[0] + x[1] * y[1]) + x[2] * y[2]


def _axpy(u, t, w):
    "u + t * w per axis (multiply, then add)"
    return (u[0] + t * w[0], u[1] + t * w[1], u[2] + t * w[2])


def _where(m, x, y):
    return tuple(np.where(m, x[i], y[i]) for i in range(3))


def _segment(p, u, v):
    "closest point of segment (u, v): u + clamp(dot(p-u, w) / dot(w, w), 0, 1) * w with w = v-u; u where dot(w, w) == 0"
    w = _sub(v, u)
    ww = _dot(w, w)
    t = np.minimum(np.maximum(_dot(_sub(p, u), w) / np.where(ww == 0, 1.0, ww), 0.0), 1.0)
    return _where(ww == 0, u, _axpy(u, t, w))


def triangle_closest(p, a, b, c):
    """(q, d2): the closest point q (3 arrays) of triangle (a, b, c) to p, and d2 = dot(p-q, p-q).  p, a, b, c are
    triples of broadcastable fp64 arrays.  The region walk and the segment rule of the definition (see `closest`)."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        ab, ac, ap = _sub(b, a), _sub(c, a), _sub(p, a)
        d1, d2 = _dot(ab, ap), _dot(ac, ap)
        bp = _sub(p, b)
        d3, d4 = _dot(ab, bp), _dot(ac, bp)
        vc = d1 * d4 - d3 * d2
        cp = _sub(p, c)
        d5, d6 = _dot(ab, cp), _dot(ac, cp)
        vb = d5 * d2 - d1 * d6
        va = d3 * d6 - d5 * d4
        e, f = d4 - d3, d5 - d6
        s = (va + vb) + vc
        den3, den5, den6 = d1 - d3, d2 - d6, e + f
        v, w = vb / s, vc / s
        # the region of the walk: the first of steps 1..6 whose test holds, else 7
        tests = [(d1 <= 0) & (d2 <= 0), (d3 >= 0) & (d4 <= d3), (vc <= 0) & (d1 >= 0) & (d3 <= 0),
                 (d6 >= 0) & (d5 <= d6), (vb <= 0) & (d2 >= 0) & (d6 <= 0), (va <= 0) & (e >= 0) & (f >= 0)]
        shape = np.broadcast(*(list(p) + list(a) + list(b) + list(c))).shape
        region = np.full(shape, 7, np.int8)
        for r in range(6, 0, -1):
            region = np.where(tests[r - 1], r, region)
        seg = (((region == 3) & (den3 == 0)) | ((region == 5) & (den5 == 0)) | ((region == 6) & (den6 == 0)) |
               ((region == 7) & ~((s > 0) & (v >= 0) & (w >= 0) & (v + w <= 1))))
        q = _axpy(_axpy(a, v, ab), w, ac)                                  # 7: (a + v*ab) + w*ac
        q = _where(region == 6, _axpy(b, e / den6, _sub(c, b)), q)
        q = _where(region == 5, _axpy(a, d2 / den5, ac), q)
        q = _where(region == 4, c, q)
        q = _where(region == 3, _axpy(a, d1 / den3, ab), q)
        q = _where(region == 2, b, q)
        q = _where(region == 1, a, q)
        if seg.any():
            best = _segment(p, a, b)
            bd = _dot(_sub(p, best), _sub(p, best))
            for u, x in ((b, c), (c, a)):
                o = _segment(p, u, x)
                od = _dot(_sub(p, o), _sub(p, o))
                best, bd = _where(od < bd, o, best), np.where(od < bd, od, bd)
            q = _where(seg, best, q)
        q = tuple(np.broadcast_to(x, shape) for x in q)
        d = _sub(p, q)
        return q, _dot(d, d)


def _pairs(P, V, tris, pi, ti):
    "(q [n, 3], d2 [n]) of the (point, triangle) pairs pi, ti"
    p = tuple(P[pi, i] for i in range(3))
    a, b, c = (tuple(V[tris[ti, k], i] for i in range(3)) for k in range(3))
    q, d2 = triangle_closest(p, a, b, c)
    return np.stack(q, axis=-1), d2


def closest(verts, tris, points, max_distance=np.inf, prune=False, chunk=1 << 19):
    """(dict(distance [P] f64, triangle [P] int32, point [P, 3] f64), n_found) -- ctr_mt3d_closest's definition.

      * Positions (fp32 or fp64 geometry) and query points (fp32 or fp64) are widened to fp64; every operation below is
        one fp64 operation, rounded on its own (no fused multiply-add), and dot(x, y) = (x0*y0 + x1*y1) + x2*y2.
      * Closest point q of triangle t = (a, b, c), corners in stored order, to p: Ericson's region walk (Real-Time
        Collision Detection, 5.1.5) in this order:
          1. ab = b-a, ac = c-a, ap = p-a, d1 = dot(ab,ap), d2 = dot(ac,ap).  d1 <= 0 and d2 <= 0: q = a.
          2. bp = p-b, d3 = dot(ab,bp), d4 = dot(ac,bp).  d3 >= 0 and d4 <= d3: q = b.
          3. vc = d1*d4 - d3*d2.  vc <= 0 and d1 >= 0 and d3 <= 0: q = a + (d1/(d1-d3))*ab.
          4. cp = p-c, d5 = dot(ab,cp), d6 = dot(ac,cp).  d6 >= 0 and d5 <= d6: q = c.
          5. vb = d5*d2 - d1*d6.  vb <= 0 and d2 >= 0 and d6 <= 0: q = a + (d2/(d2-d6))*ac.
          6. va = d3*d6 - d5*d4, e = d4-d3, f = d5-d6.  va <= 0 and e >= 0 and f >= 0: q = b + (e/(e+f))*(c-b).
          7. Otherwise s = (va+vb)+vc, v = vb/s, w = vc/s.  s > 0 and v >= 0 and w >= 0 and v+w <= 1:
             q = (a + v*ab) + w*ac, per axis.
        The segment rule replaces steps 3, 5 and 6 when their denominator is 0, and step 7 when its test fails: these
        are the degenerate and nearly degenerate triangles (marching tetrahedra emits zero-area ones), where the
        barycentric weights are rounding noise.  For each edge (a,b), (b,c), (c,a) in this order it takes
        u + clamp(dot(p-u, w)/dot(w, w), 0, 1)*w with w = v-u (u itself when dot(w, w) == 0), and keeps the edge with
        the smallest d2, the first on a tie.  So every weight is in [0, 1] and q is within a few rounding errors of
        the triangle: a search that prunes by boxes padded by much more than that finds what brute force finds.
      * d2 = dot(p-q, p-q); distance = sqrt(d2), correctly rounded.
      * The winner of a point is the triangle with the smallest d2, the smallest triangle index on a tie.  The point
        is found when that d2 <= max_distance * max_distance (the product in fp64; +inf finds every point).  A point
        not found, and every point on a mesh without triangles, gets distance +inf, triangle -1 and point NaN.
    n_found counts the found points.

    Brute force over every triangle, in chunks.  prune=True evaluates only the triangles that may win: r = the distance
    to the nearest vertex a triangle uses (scipy's cKDTree), which bounds the winner's distance; every triangle within
    r (or max_distance, when smaller) of p, with relative and absolute slack of 1e-7 far above the rounding errors of
    q and d2, has its centroid within that bound plus the largest centroid-to-corner distance of the mesh.  The
    result is the same (tests/test_oracle_closest_cpu.py checks it against brute force)."""
    V = np.asarray(verts).astype(np.float64).reshape(-1, 3)
    T = np.asarray(tris, np.int64).reshape(-1, 3)
    P = np.asarray(points).astype(np.float64).reshape(-1, 3)
    md = float(max_distance)
    if not (md >= 0):
        raise ValueError("max_distance must be >= 0")
    if not np.isfinite(P).all():
        raise ValueError("query points must be finite")
    if len(T) and (T.min() < 0 or T.max() >= len(V)):
        raise ValueError("triangle ids outside [0, n_verts)")
    nP, nT = len(P), len(T)
    best_d2 = np.full(nP, np.inf)
    best_t = np.full(nP, -1, np.int64)
    best_q = np.full((nP, 3), np.nan)
    if nP and nT:
        if prune:
            _pruned(V, T, P, md, best_d2, best_t, best_q, chunk)
        else:
            step_p = max(1, chunk // nT)
            step_t = min(nT, chunk)
            for p0 in range(0, nP, step_p):
                pi = np.arange(p0, min(nP, p0 + step_p))
                for t0 in range(0, nT, step_t):                          # ascending triangle order: < keeps the first
                    ti = np.arange(t0, min(nT, t0 + step_t))
                    PI, TI = np.repeat(pi, len(ti)), np.tile(ti, len(pi))
                    q, d2 = _pairs(P, V, T, PI, TI)
                    d2 = d2.reshape(len(pi), len(ti))
                    k = np.argmin(d2, axis=1)
                    m = d2[np.arange(len(pi)), k]
                    better = m < best_d2[pi]
                    sel = pi[better]
                    best_d2[sel] = m[better]
                    best_t[sel] = ti[k[better]]
                    best_q[sel] = q.reshape(len(pi), len(ti), 3)[np.arange(len(pi))[better], k[better]]
    found = (best_t >= 0) & (best_d2 <= md * md)
    distance = np.where(found, np.sqrt(np.where(found, best_d2, 0.0)), np.inf)
    point = np.where(found[:, None], best_q, np.nan)
    return dict(distance=distance, triangle=np.where(found, best_t, -1).astype(np.int32), point=point), int(found.sum())


def _pruned(V, T, P, md, best_d2, best_t, best_q, chunk):
    from scipy.spatial import cKDTree
    used = np.unique(T)
    r = cKDTree(V[used]).query(P)[0]
    scale = max(float(np.abs(V[used]).max()), float(np.abs(P).max()), 1.0)
    r = np.minimum(r, md)
    cen = V[T].mean(axis=1)
    rad = float(np.sqrt(((V[T] - cen[:, None, :]) ** 2).sum(axis=2)).max())
    reach = (r + rad) * (1 + 1e-7) + 1e-7 * scale
    tree = cKDTree(cen)
    lists = tree.query_ball_point(P, reach)
    counts = np.array([len(x) for x in lists], np.int64)
    if not counts.sum():
        return
    PI = np.repeat(np.arange(len(P)), counts)
    TI = np.concatenate([np.asarray(x, np.int64) for x in lists if len(x)])
    d2 = np.empty(len(PI))
    q = np.empty((len(PI), 3))
    for s0 in range(0, len(PI), chunk):
        sl = slice(s0, s0 + chunk)
        q[sl], d2[sl] = _pairs(P, V, T, PI[sl], TI[sl])
    o = np.lexsort((TI, d2, PI))                                         # by point, then d2, then triangle
    first = o[np.r_[True, PI[o][1:] != PI[o][:-1]]]
    pi = PI[first]
    best_d2[pi] = d2[first]
    best_t[pi] = TI[first]
    best_q[pi] = q[first]
