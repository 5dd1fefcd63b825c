"""ORACLE (test infrastructure, not product code) -- keeping or dropping connected components of a 3D triangle mesh.

An engine extension with no counterpart in the reference, like oracle/mt3d_components.py: `keep_components` below is
the DEFINITION that ctr_mt3d_keep_components is tested against.  It is a pure function of a mesh, its components
(oracle/mt3d_components.components or the engine's ctr_mt3d_components) and a keep mask.
"""
import numpy as np


def keep_components(tris, label, table, keep):
    """(tris [T', 3] int32, used [V'] int64, label [T'] int32, table [K]) after keeping the components c with keep[c]:
      - a triangle stays when its component is kept; kept triangles stay in their order;
      - a vertex stays when a kept triangle uses it (also one that a dropped component shares); `used` lists the kept
        old vertex ids in ascending order, so verts[used], normals[used], keys[used], lowmin[used] and values[used] are
        the compacted per-vertex arrays, and the ids in the triangles are the positions in `used`;
      - the kept components are renumbered 0..K-1 in their old order; their table rows are carried over as they are,
        except first_tri, which becomes the compacted index of the component's first triangle.
    keep: boolean (or 0 / non-zero) array of len(table) entries."""
    tris = np.asarray(tris).reshape(-1, 3)
    label = np.asarray(label, dtype=np.int64)
    keep = np.asarray(keep).astype(bool).reshape(-1)
    if len(keep) != len(table):
        raise ValueError("keep has %d entries for %d components" % (len(keep), len(table)))
    if len(label) != len(tris):
        raise ValueError("one label per triangle expected")
    keep_t = keep[label] if len(label) else np.zeros(0, bool)
    kept = tris[keep_t].astype(np.int64)
    used = np.unique(kept.reshape(-1))
    new_tris = np.searchsorted(used, kept).astype(np.int32).reshape(-1, 3)
    new_c = np.cumsum(keep) - 1                         # new number of every kept component
    tri_new = np.cumsum(keep_t) - 1                     # new index of every kept triangle
    new_label = new_c[label[keep_t]].astype(np.int32)
    new_table = np.array(table[keep], copy=True)
    if len(new_table):
        new_table["first_tri"] = tri_new[new_table["first_tri"]]
    return new_tris, used, new_label, new_table
