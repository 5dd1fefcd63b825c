"""ORACLE (test infrastructure, not product code) -- connected components of a 3D triangle mesh with their size and
topology.

An engine extension with no counterpart in the reference (its surface_geometry.py:52-140 orient_triangles finds the
same edge-connected components but keeps nothing of them): `components` below is the DEFINITION that
ctr_mt3d_components is tested against, parity UNPINNED by the reference, like oracle/mt3d_values.py.  It is a pure
function of a mesh.  The signed volume assumes the engine's winding (cross(b - a, c - a) towards the high side of the
field, or outward after orientation); oracle/mt3d.py:extract's `tris` are not wound.
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

# mirrors ctr_mt3d_component (include/contourist_b200.h), 112 bytes
COMPONENT_DTYPE = np.dtype([("n_tris", "<i8"), ("n_verts", "<i8"), ("n_edges", "<i8"), ("n_boundary_edges", "<i8"),
                            ("n_nonmanifold_edges", "<i8"), ("first_tri", "<i8"), ("area", "<f8"), ("volume", "<f8"),
                            ("lo", "<f8", (3,)), ("hi", "<f8", (3,))])


def _cross(u, w):
    return np.stack([u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1],
                     u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2],
                     u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]], axis=1)


def components(verts, tris):
    """(tri_component [T] int32, table [C] COMPONENT_DTYPE) of the mesh (parity UNPINNED by the reference -- engine
    definition, ctr_mt3d_components):
      - two triangles are in one component when they share an undirected vertex-id edge (not a lone vertex);
      - components are numbered in ascending order of their smallest triangle index (first_tri);
      - n_edges: distinct undirected edges, n_boundary_edges / n_nonmanifold_edges: those used once / three or more
        times (a use is one of a triangle's three edge slots); n_verts: distinct (component, vertex) pairs, so
        n_verts - n_edges + n_tris is the Euler characteristic;
      - lo / hi: the box of the component's vertices; area: sum of |cross(b - a, c - a)| / 2; volume: sum of
        (a - lo) . ((b - lo) x (c - lo)) / 6; positions widened to float64 first."""
    verts = np.asarray(verts)
    tris = np.asarray(tris, dtype=np.int64).reshape(-1, 3)
    nt = len(tris)
    if nt == 0:
        return np.zeros(0, np.int32), np.zeros(0, COMPONENT_DTYPE)
    if tris.min() < 0 or tris.max() >= len(verts):
        raise ValueError("triangle ids outside [0, n_verts)")
    # every edge slot of every triangle, as an undirected key
    a = tris[:, [0, 1, 2]].reshape(-1)
    b = tris[:, [1, 2, 0]].reshape(-1)
    ekey = (np.maximum(a, b) << 32) | np.minimum(a, b)
    uniq, inv, uses = np.unique(ekey, return_inverse=True, return_counts=True)
    ne = len(uniq)
    slot_tri = np.repeat(np.arange(nt), 3)
    g = coo_matrix((np.ones(3 * nt, np.int8), (slot_tri, nt + inv)), shape=(nt + ne, nt + ne)).tocsr()
    _, lab = connected_components(g, directed=False)
    lab = lab[:nt]
    raw, first = np.unique(lab, return_index=True)      # first triangle of each raw label
    order = np.argsort(first)
    remap = np.empty(len(first), np.int64)
    remap[raw[order]] = np.arange(len(first))
    label = remap[lab]
    nc = len(first)
    out = np.zeros(nc, COMPONENT_DTYPE)
    out["first_tri"] = first[order]
    out["n_tris"] = np.bincount(label, minlength=nc)
    edge_label = np.empty(ne, np.int64)
    edge_label[inv] = label[slot_tri]
    out["n_edges"] = np.bincount(edge_label, minlength=nc)
    out["n_boundary_edges"] = np.bincount(edge_label[uses == 1], minlength=nc)
    out["n_nonmanifold_edges"] = np.bincount(edge_label[uses >= 3], minlength=nc)
    pairs = np.unique((label[slot_tri] << 32) | tris.reshape(-1))
    out["n_verts"] = np.bincount(pairs >> 32, minlength=nc)
    p = verts.astype(np.float64)[tris]                   # [T, 3 corners, 3]
    out["area"] = np.bincount(label, weights=0.5 * np.sqrt((_cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]) ** 2).sum(axis=1)),
                              minlength=nc)
    srt = np.argsort(label, kind="stable")
    starts = np.searchsorted(label[srt], np.arange(nc))
    out["lo"] = np.minimum.reduceat(p.min(axis=1)[srt], starts, axis=0)
    out["hi"] = np.maximum.reduceat(p.max(axis=1)[srt], starts, axis=0)
    q = p - out["lo"][label][:, None, :]
    vol = (q[:, 0] * _cross(q[:, 1], q[:, 2])).sum(axis=1) / 6.0
    out["volume"] = np.bincount(label, weights=vol, minlength=nc)
    return label.astype(np.int32), out
