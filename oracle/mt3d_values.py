"""ORACLE (test infrastructure, not product code) -- values of other fields at the 3D vertices.

An engine extension with no counterpart in the reference (the reference's contour_pair_interpolation,
tetrahedral.py:471-487, interpolates positions only): `vertex_values` below is the DEFINITION that
ctr_mt3d_interpolate is tested against, parity UNPINNED by the reference, like oracle/mt3d.py:normals.  It reuses
the key decoding and the allclose tolerance of oracle/mt3d.py; in grid coordinates the field of grid coordinates
gives exactly mt3d.interpolate's positions (tests/test_oracle_attributes_cpu.py).
"""
import numpy as np

from .mt3d import ATOL, key_points


def vertex_values(field, value, keys, lowmin, attr, geom_dtype=np.float64):
    """Values of another field at the vertices (parity UNPINNED by the reference -- engine definition,
    ctr_mt3d_interpolate): a = a_low + ratio*(a_high - a_low), the same `ratio` as the position (mt3d.interpolate), the
    low end taken from the passed `lowmin` (at ratio 0.5 the two orientations round differently), attribute samples
    widened to geom_dtype first, no world transform.  attr [n0,n1,n2] or [n0,n1,n2,c] on the grid of `field`;
    keys / lowmin as the engine returns them (any order).  Returns [V] or [V, c] geom_dtype."""
    field = np.asarray(field)
    gd = np.dtype(geom_dtype)
    pmin, pmax = key_points(np.asarray(keys, dtype=np.uint64), field.shape)
    low = np.asarray(lowmin).astype(bool)
    fmin = field[pmin[:, 0], pmin[:, 1], pmin[:, 2]].astype(gd)
    fmax = field[pmax[:, 0], pmax[:, 1], pmax[:, 2]].astype(gd)
    flow = np.where(low, fmin, fmax)
    fhigh = np.where(low, fmax, fmin)
    den = fhigh - flow
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = (gd.type(value) - flow) / den
    ratio = np.where(np.abs(den.astype(np.float64)) <= ATOL, gd.type(0.5), ratio).astype(gd)
    a = np.asarray(attr)
    scalar = a.ndim == 3
    if scalar:
        a = a[..., None]
    amin = a[pmin[:, 0], pmin[:, 1], pmin[:, 2]].astype(gd)
    amax = a[pmax[:, 0], pmax[:, 1], pmax[:, 2]].astype(gd)
    alow = np.where(low[:, None], amin, amax)
    ahigh = np.where(low[:, None], amax, amin)
    out = (alow + ratio[:, None] * (ahigh - alow)).astype(gd)
    return out[:, 0] if scalar else out
