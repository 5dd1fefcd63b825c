"""ORACLE (test infrastructure, not product code) -- clipping of a 3D triangle mesh by a plane or by a vertex value.

An engine extension with no counterpart in the reference package (VTK's vtkClipPolyData does the same job; the
reference's constraints.py restricts a level set by half-spaces but nothing calls it): `clip` below is the DEFINITION
that ctr_mt3d_clip is tested against, parity UNPINNED by the reference, like oracle/mt3d_section.py.  It is a pure
function of a mesh (as the engine's fetch returns it), a side function and an offset.  Every output is a selection, a
copy or one fixed-order fp64 formula, so the device result equals it bit for bit.
"""
import numpy as np

from oracle.mt3d_cap import fan, polygon
from oracle.mt3d_section import edge_key, sides

HIGH, LOW = 0, 1
SIDES = {"high": HIGH, "low": LOW}


def clip(verts, tris, normals=None, keys=None, lowmin=None, values=None, *, normal=None, component=None, offset, side,
         geom_dtype):
    """(clipped mesh dict, counts) -- ctr_mt3d_clip's definition.

    Exactly one of `normal` (plane mode) and `component` (value mode, `values` [V] or [V, c] required) is given.
      * Side value of a vertex: plane mode s = (n0 x + n1 y) + n2 z on the positions widened to fp64, every operation
        rounded (oracle/mt3d_section.py:sides); value mode s = values[:, component] widened.  High when s >= offset,
        low otherwise; kept when on `side` ("high" / "low" or HIGH (0) / LOW (1)).  A NaN s raises ValueError.
      * Vertices: the kept ones in their order (also those no triangle uses), then one new vertex per distinct
        undirected edge {a, b} of some triangle whose ends are on different sides, in the order of first use (smallest
        triangle index, then the edge's position (v0,v1), (v1,v2), (v2,v0) in it).  With a the low end:
        t = (offset - s_a) / (s_b - s_a), position p_a + t * (p_b - p_a) per axis in fp64, rounded once to geom_dtype
        (the crossing point of oracle/mt3d_section.py:segments).  Normal: m = n_a + t * (n_b - n_a), then
        m / sqrt((mx*mx + my*my) + mz*mz) rounded once, or the kept end's normal where that length is 0.  key / lowmin:
        the kept end's.  Values: v_a + t * (v_b - v_a) per component, rounded once.
      * Triangles: each input triangle walks i = 0, 1, 2 and emits corner i if it is kept, then the crossing of edge
        (i, i+1 mod 3) if exactly one end of that edge is kept (oracle/mt3d_cap.py:polygon); 3 tokens are one triangle,
        4 the fan (p0, p1, p2), (p0, p2, p3) (fan), 0 drop it.  Output by input triangle, then piece: every piece keeps
        its source triangle's winding.
      * Every vertex kept: the mesh is returned unchanged, with n_new_verts = n_cut_tris = n_dropped_tris = 0.

    counts: dict(n_verts, n_tris, n_new_verts, n_cut_tris, n_dropped_tris)."""
    side = SIDES[side] if isinstance(side, str) else int(side)
    if side not in (HIGH, LOW):
        raise ValueError("side must be 'high' or 'low'")
    if (normal is None) == (component is None):
        raise ValueError("exactly one of normal and component")
    gd = np.dtype(geom_dtype)
    verts = np.asarray(verts)
    tris = np.asarray(tris, np.int64).reshape(-1, 3)
    nV, nT = len(verts), len(tris)
    if nT and (tris.min() < 0 or tris.max() >= nV):
        raise ValueError("triangle ids outside [0, n_verts)")
    offset = float(offset)
    if normal is not None:
        s = sides(verts, normal) if nV else np.zeros(0)
    else:
        if values is None:
            raise ValueError("value mode needs the vertex values")
        s = np.asarray(values).reshape(nV, -1)[:, int(component)].astype(np.float64)
    if np.isnan(s).any():
        raise ValueError("a side value is NaN")
    high = s >= offset
    kept = high if side == HIGH else ~high
    mesh = dict(verts=verts, tris=tris.astype(np.int32), normals=normals, keys=keys, lowmin=lowmin, values=values)
    if kept.all():
        return mesh, dict(n_verts=nV, n_tris=nT, n_new_verts=0, n_cut_tris=0, n_dropped_tris=0)

    kt = kept[tris]                                                  # [T, 3]
    cross = kt != np.roll(kt, -1, axis=1)                            # cross[:, i]: edge (v_i, v_i+1) is crossed
    cut = cross.any(axis=1)
    dropped = ~kt.any(axis=1)
    # crossed edges in (triangle, position) order; the first occurrence of every undirected edge numbers it
    ct, ci = np.nonzero(cross)
    ea, eb = tris[ct, ci], tris[ct, (ci + 1) % 3]
    ek = edge_key(ea, eb)
    uk, first, inv = np.unique(ek, return_index=True, return_inverse=True)
    rank = np.empty(len(uk), np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(len(uk))
    nk = int(kept.sum())
    xid = np.full((nT, 3), -1, np.int64)
    xid[ct, ci] = nk + rank[inv.reshape(-1)]
    # the new vertices
    fo = np.sort(first)
    a, b = ea[fo], eb[fo]
    lo = np.where(high[a], b, a)
    hi = np.where(high[a], a, b)
    ke = np.where(kept[a], a, b)
    t = (offset - s[lo]) / (s[hi] - s[lo])

    def lerp(x):
        x = np.asarray(x).reshape(nV, -1).astype(np.float64)
        return x[lo] + t[:, None] * (x[hi] - x[lo])

    out = {}
    out["verts"] = np.concatenate([verts[kept], lerp(verts).astype(gd)]).astype(gd)
    if normals is not None:
        normals = np.asarray(normals)
        m = lerp(normals)
        ln = np.sqrt((m[:, 0] * m[:, 0] + m[:, 1] * m[:, 1]) + m[:, 2] * m[:, 2])
        with np.errstate(divide="ignore", invalid="ignore"):
            nn = (m / ln[:, None]).astype(gd)
        nn[ln == 0] = normals[ke[ln == 0]]
        out["normals"] = np.concatenate([normals[kept], nn]).astype(gd)
    else:
        out["normals"] = None
    out["keys"] = None if keys is None else np.concatenate([np.asarray(keys)[kept], np.asarray(keys)[ke]])
    out["lowmin"] = None if lowmin is None else np.concatenate([np.asarray(lowmin)[kept], np.asarray(lowmin)[ke]])
    if values is not None:
        vals = np.asarray(values)
        nv_ = lerp(vals).astype(gd).reshape((len(lo),) + vals.shape[1:])
        out["values"] = np.concatenate([vals[kept], nv_]).astype(gd)
    else:
        out["values"] = None
    # the triangles: the corner walk of every input triangle, fanned
    vid = np.full(nV, -1, np.int64)
    vid[kept] = np.arange(nk)
    pieces = np.full((nT, 2, 3), -1, np.int64)
    valid = np.zeros((nT, 2), bool)
    code = kt[:, 0] * 1 + kt[:, 1] * 2 + kt[:, 2] * 4
    for c in range(1, 8):
        rows = np.nonzero(code == c)[0]
        if not len(rows):
            continue
        toks = polygon([(c >> i) & 1 for i in range(3)])
        ids = np.zeros((len(rows), len(toks)), np.int64)
        for q, tok in enumerate(toks):
            ids[:, q] = vid[tris[rows, tok[1]]] if tok[0] == "c" else xid[rows, tok[1]]
        for pc, tri in enumerate(fan(len(toks))):
            pieces[rows, pc] = ids[:, list(tri)]
            valid[rows, pc] = True
    out["tris"] = pieces[valid].astype(np.int32).reshape(-1, 3)
    counts = dict(n_verts=nk + len(fo), n_tris=len(out["tris"]), n_new_verts=len(fo), n_cut_tris=int(cut.sum()),
                  n_dropped_tris=int(dropped.sum()))
    return out, counts
