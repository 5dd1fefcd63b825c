"""ORACLE (test infrastructure, not product code) -- quadric vertex-clustering decimation of a 3D triangle mesh.

An engine extension, like oracle/mt3d_smooth.py: the reference's flatten (collapse_flat_segments, tetrahedral.py:217-327)
solves an LP per edge and is not reproduced, so `decimate` below is the DEFINITION that ctr_mt3d_decimate is tested
against (parity UNPINNED by the reference).  Lindstrom's quadric clustering (Out-of-core simplification of large
polygonal models, SIGGRAPH 2000), as in VTK's vtkQuadricClustering, with a regularised solve.  Counts, triangles and
the member of every output vertex are exact; the engine sums the quadrics in an unspecified order, so its positions
equal these within rounding.
"""
import numpy as np

QLIM = 1 << 20                                         # cell indices lie in [-2^20, 2^20)


def _cross(u, w):
    """cross(u, w) in the expression order of the engine's face normals (k_s_nsum)"""
    return np.stack([u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1],
                     u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2],
                     u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]], axis=1)


def cells(verts, cell, origin):
    """(q [V, 3] int64 cell indices, lo [V, 3] float64 cell corners) of every vertex: q = floor((p - origin) / cell)
    (subtract, then divide), lo = origin + q * cell (multiply, then add).  ValueError when an index leaves
    [-2^20, 2^20)."""
    p = np.asarray(verts).astype(np.float64).reshape(-1, 3)
    cell = np.broadcast_to(np.asarray(cell, np.float64), (3,))
    origin = np.broadcast_to(np.asarray(origin, np.float64), (3,))
    qf = np.floor((p - origin) / cell)
    if len(qf) and not ((qf >= -QLIM) & (qf < QLIM)).all():
        raise ValueError("a cell index (p - origin) / cell lies outside [-2^20, 2^20)")
    return qf.astype(np.int64), origin + qf * cell


def decimate(verts, tris, cell, origin=(0.0, 0.0, 0.0)):
    """(verts [V', 3] in the geometry type, tris [T', 3] int32, member [V'] int64, counts) after quadric clustering
    (parity UNPINNED by the reference -- engine definition, ctr_mt3d_decimate); all arithmetic in float64 on positions
    widened from the geometry type:
      1. cluster of a vertex: its cell q = floor((p - origin) / cell); cell corner lo = origin + q * cell;
      2. quadrics: every triangle (a, b, c), also one that collapses in 4, has n = cross(P_b - P_a, P_c - P_a); for each
         corner, with k its cluster and d = -(n . (P_a - lo_k)), A_k += n n^T and g_k += d n;
      3. position: m_k = mean of P - lo_k over the cluster's vertices, lam = 1e-3 * trace(A_k); x = m_k if lam == 0,
         else the solution of (A_k + lam I) x = lam m_k - g_k (by the adjugate); each axis of x clamped to
         [0, cell]; the position lo_k + x is rounded to the geometry type once;
      4. triangles through the clusters of their corners: fewer than three distinct clusters -> dropped (n_collapsed);
         of equal sets of three clusters (either winding) the first in triangle order stays (n_duplicate); kept
         triangles keep their order and corner order;
      5. every cluster a kept triangle uses becomes one vertex, in the order of its smallest member id; that member is
         `member` (keys / lowmin / old normals of the output are the member's rows).
    counts: dict(n_verts, n_tris, n_clusters = occupied cells, n_collapsed, n_duplicate)."""
    verts = np.asarray(verts)
    dtype = verts.dtype
    P = verts.astype(np.float64).reshape(-1, 3)
    T = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    cell = np.broadcast_to(np.asarray(cell, np.float64), (3,))
    q, lo = cells(P, cell, origin)
    nv = len(P)
    if nv == 0:
        return (np.zeros((0, 3), dtype), np.zeros((0, 3), np.int32), np.zeros(0, np.int64),
                dict(n_verts=0, n_tris=0, n_clusters=0, n_collapsed=0, n_duplicate=0))
    key = ((q[:, 0] + QLIM) << 42) | ((q[:, 1] + QLIM) << 21) | (q[:, 2] + QLIM)
    _, first, cid = np.unique(key, return_index=True, return_inverse=True)   # first: the smallest member of each
    cid = cid.reshape(-1)
    nc = len(first)
    rep = first[cid]                                    # every vertex's cluster, named by its smallest member
    # 2. quadrics, per cluster (indexed by cid)
    A = np.zeros((nc, 6))                               # xx xy xz yy yz zz
    g = np.zeros((nc, 3))

    def add(acc, idx, rows):
        for i in range(acc.shape[1]):
            acc[:, i] += np.bincount(idx, weights=rows[:, i], minlength=nc)
    if len(T):
        Pa, Pb, Pc = P[T[:, 0]], P[T[:, 1]], P[T[:, 2]]
        n = _cross(Pb - Pa, Pc - Pa)
        nn = np.stack([n[:, 0] * n[:, 0], n[:, 0] * n[:, 1], n[:, 0] * n[:, 2],
                       n[:, 1] * n[:, 1], n[:, 1] * n[:, 2], n[:, 2] * n[:, 2]], axis=1)
        for j in range(3):
            k = cid[T[:, j]]
            r = Pa - lo[T[:, j]]
            d = -((n[:, 0] * r[:, 0] + n[:, 1] * r[:, 1]) + n[:, 2] * r[:, 2])
            add(A, k, nn)
            add(g, k, d[:, None] * n)
    # 3. representative positions
    cnt = np.bincount(cid, minlength=nc).astype(np.float64)
    s = np.zeros((nc, 3))
    add(s, cid, P - lo)
    m = s / cnt[:, None]
    lam = 1e-3 * ((A[:, 0] + A[:, 3]) + A[:, 5])
    x = m.copy()
    z = lam != 0
    a00, a01, a02 = A[z, 0] + lam[z], A[z, 1], A[z, 2]
    a11, a12, a22 = A[z, 3] + lam[z], A[z, 4], A[z, 5] + lam[z]
    b = lam[z, None] * m[z] - g[z]
    c00 = a11 * a22 - a12 * a12
    c01 = a02 * a12 - a01 * a22
    c02 = a01 * a12 - a02 * a11
    c11 = a00 * a22 - a02 * a02
    c12 = a01 * a02 - a00 * a12
    c22 = a00 * a11 - a01 * a01
    det = (a00 * c00 + a01 * c01) + a02 * c02
    x[z, 0] = ((c00 * b[:, 0] + c01 * b[:, 1]) + c02 * b[:, 2]) / det
    x[z, 1] = ((c01 * b[:, 0] + c11 * b[:, 1]) + c12 * b[:, 2]) / det
    x[z, 2] = ((c02 * b[:, 0] + c12 * b[:, 1]) + c22 * b[:, 2]) / det
    x = np.minimum(np.maximum(x, 0.0), cell)
    clo = np.zeros((nc, 3))
    clo[cid] = lo
    pos = (clo + x).astype(dtype)
    # 4. triangles
    R = rep[T] if len(T) else np.zeros((0, 3), np.int64)
    distinct = (R[:, 0] != R[:, 1]) & (R[:, 0] != R[:, 2]) & (R[:, 1] != R[:, 2])
    keep = distinct.copy()
    if distinct.any():
        srt = np.sort(R[distinct], axis=1)
        order = np.lexsort((srt[:, 2], srt[:, 1], srt[:, 0]))   # stable: equal triples stay in triangle order
        s_ = srt[order]
        head = np.ones(len(s_), bool)
        head[1:] = (s_[1:] != s_[:-1]).any(axis=1)
        kd = np.zeros(len(s_), bool)
        kd[order[head]] = True
        keep[np.flatnonzero(distinct)] = kd
    kept = R[keep]
    # 5. vertices: the used clusters in the order of their smallest member
    member = np.unique(kept.reshape(-1))
    out_tris = np.searchsorted(member, kept).astype(np.int32).reshape(-1, 3)
    counts = dict(n_verts=len(member), n_tris=len(out_tris), n_clusters=nc, n_collapsed=int((~distinct).sum()),
                  n_duplicate=int(distinct.sum() - keep.sum()))
    return pos[cid[member]].reshape(-1, 3), out_tris, member.astype(np.int64), counts
