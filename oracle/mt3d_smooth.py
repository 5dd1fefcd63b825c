"""ORACLE (test infrastructure, not product code) -- Taubin lambda|mu smoothing of a 3D triangle mesh.

An engine extension, like oracle/mt3d_components.py: the reference's smooth_interpolations (tetrahedral.py:329-351) is
not available to pin, so `smooth` below is the DEFINITION that ctr_mt3d_smooth is tested against (parity UNPINNED by
the reference).  Positions are deterministic and the engine reproduces them bit for bit; `normals` is the definition of
the recomputed normals, which the engine sums in an unspecified order (equal within rounding).
"""
import numpy as np


def edges(tris):
    """(keys, uses) of the distinct undirected edges {a, b}, a != b: every edge slot (a, b) of every triangle is one
    use (the use count of oracle/mt3d_components.py without self-edges); key = max << 32 | min, ascending."""
    tris = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    a = tris[:, [0, 1, 2]].reshape(-1)
    b = tris[:, [1, 2, 0]].reshape(-1)
    real = a != b
    a, b = a[real], b[real]
    return np.unique((np.maximum(a, b) << 32) | np.minimum(a, b), return_counts=True)


def neighbours(n_verts, tris):
    """(off [V + 1], nbr, fixed [V] bool, n_edges): the CSR lists of the free vertices' distinct edge neighbours in
    ascending id order (fixed ones included); fixed vertices -- on an edge with uses != 2, or on no edge -- have none."""
    keys, uses = edges(tris)
    lo, hi = keys & 0xffffffff, keys >> 32
    fixed = np.ones(n_verts, bool)
    fixed[lo] = False
    fixed[hi] = False
    bad = uses != 2
    fixed[lo[bad]] = True
    fixed[hi[bad]] = True
    src = np.concatenate([lo, hi])
    dst = np.concatenate([hi, lo])
    keep = ~fixed[src]
    src, dst = src[keep], dst[keep]
    order = np.lexsort((dst, src))
    src, dst = src[order], dst[order]
    off = np.zeros(n_verts + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(src, minlength=n_verts))
    return off, dst, fixed, len(keys)


def smooth(verts, tris, iterations, lam, mu):
    """(verts, counts) after `iterations` lambda|mu pairs of Taubin smoothing (parity UNPINNED by the reference --
    engine definition, ctr_mt3d_smooth):
      - an edge is {a, b}, a != b, of some triangle; its uses are the triangle edge slots on it.  A vertex on an edge
        with uses != 2 (boundary or non-manifold) or on no edge is FIXED: it never moves and comes back bit for bit;
      - a free vertex averages all its distinct edge neighbours, fixed ones included: s = x[n0], s = s + x[n1], ... in
        ascending id order, avg = s / deg, x' = x + w * (avg - x) (multiply rounded, then add: no fused multiply-add);
      - all arithmetic in float64 on a copy widened from the geometry type; one step is a Jacobi step (every free vertex
        reads its neighbours as they were before the step); one iteration is a step with w = lam, then one with w = mu
        (skipped when mu == 0: plain Laplacian smoothing);
      - the result is rounded to the geometry type once, at the end.
    counts: dict(n_edges = distinct undirected edges without self-edges, n_fixed_verts)."""
    verts = np.asarray(verts)
    off, nbr, fixed, n_edges = neighbours(len(verts), tris)
    counts = dict(n_edges=int(n_edges), n_fixed_verts=int(fixed.sum()))
    if iterations == 0:
        return verts.copy(), counts
    free = np.flatnonzero(~fixed)
    deg = (off[1:] - off[:-1])[free]
    start = off[:-1][free]
    weights = [float(lam)] + ([float(mu)] if mu != 0 else [])
    x = verts.astype(np.float64)
    for _ in range(int(iterations)):
        for w in weights:
            s = x[nbr[start]].copy()
            for k in range(1, int(deg.max()) if len(deg) else 0):
                more = deg > k
                s[more] = s[more] + x[nbr[start[more] + k]]
            avg = s / deg[:, None].astype(np.float64)
            xn = x.copy()
            xn[free] = x[free] + w * (avg - x[free])
            x = xn
    return x.astype(verts.dtype), counts


def normals(verts, tris, old_normals):
    """Normals of the smoothed mesh (engine definition, ctr_mt3d_smooth with CTR_WANT_NORMALS): per vertex the sum of
    cross(b - a, c - a) of the triangles it is a corner of, positions widened to float64 from `verts` (the smoothed
    geometry-type array); a non-zero sum divided by its length, its sign flipped where its dot product with the old
    (gradient) normal is negative; a zero sum keeps the old normal.  Returned in the geometry type."""
    verts = np.asarray(verts)
    old = np.asarray(old_normals)
    t = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    p = verts.astype(np.float64)
    fn = np.cross(p[t[:, 1]] - p[t[:, 0]], p[t[:, 2]] - p[t[:, 0]])
    s = np.zeros((len(verts), 3), np.float64)
    for q in range(3):
        np.add.at(s, t[:, q], fn)
    nz = (s != 0).any(axis=1)
    length = np.sqrt((s * s).sum(axis=1))
    out = old.astype(np.float64).copy()
    n = s[nz] / length[nz, None]
    flip = (n * old[nz].astype(np.float64)).sum(axis=1) < 0
    n[flip] = -n[flip]
    out[nz] = n
    return out.astype(verts.dtype)


def face_normal_sums(verts, tris):
    """(|sum|, sum of |cross|) per vertex: how far the face normals around a vertex cancel (tests skip vertices whose
    sum is tiny against its parts, where the direction is decided by rounding)."""
    p = np.asarray(verts).astype(np.float64)
    t = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    fn = np.cross(p[t[:, 1]] - p[t[:, 0]], p[t[:, 2]] - p[t[:, 0]])
    s = np.zeros((len(p), 3))
    parts = np.zeros(len(p))
    ln = np.sqrt((fn * fn).sum(axis=1))
    for q in range(3):
        np.add.at(s, t[:, q], fn)
        np.add.at(parts, t[:, q], ln)
    return np.sqrt((s * s).sum(axis=1)), parts
