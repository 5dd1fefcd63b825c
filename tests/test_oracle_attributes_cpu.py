"""CPU: oracle/mt3d_values.py:vertex_values (the definition of ctr_mt3d_interpolate), the new C ABI symbols and the façade's
vertex_fields plumbing (no GPU here)."""
import ctypes
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import mt3d, mt3d_values

FILES = sorted(glob.glob(os.path.join(GOLDEN, "mt3d_*.npz")))


def coords(shape):
    return np.stack(np.indices(shape), -1)


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f) for f in FILES])
@pytest.mark.parametrize("gd", [np.float64, np.float32])
def test_coordinate_field_gives_positions(path, gd):
    g = np.load(path)
    field, value = g["field"], float(g["value"])
    r = mt3d.extract(field, value, gd)
    for attr in (coords(field.shape), coords(field.shape).astype(np.float32), coords(field.shape).astype(np.int16)):
        v = mt3d_values.vertex_values(field, value, r["keys"], r["lowmin"], attr, gd)
        assert v.dtype == np.dtype(gd) and np.array_equal(v, r["pos"])
    if gd is np.float64:
        # the reference's own positions (tests/golden/make_golden.py), in its key orientation
        n0, n1, n2 = field.shape
        klow, khigh = g["key_low"], g["key_high"]
        pmin = np.minimum(klow, khigh)
        d = np.maximum(klow, khigh) - pmin
        keys = ((((pmin[:, 0] * n1 + pmin[:, 1]) * n2 + pmin[:, 2]).astype(np.uint64) << np.uint64(3))
                | (d[:, 0] * 4 + d[:, 1] * 2 + d[:, 2]).astype(np.uint64))
        lowmin = (klow == pmin).all(axis=1).astype(np.uint8)
        v = mt3d_values.vertex_values(field, value, keys, lowmin, coords(field.shape), gd)
        assert np.array_equal(v, g["key_pos"])


def test_orientation_comes_from_lowmin():
    """At ratio 0.5 (a flat edge) a_low + 0.5*(a_high - a_low) depends on which end is low."""
    field = np.zeros((2, 2, 2))
    keys = np.array([1], np.uint64)                  # point (0,0,0) -> (0,0,1)
    attr = np.zeros((2, 2, 2))
    attr[0, 0, 0], attr[0, 0, 1] = 0.1, 0.7
    a = mt3d_values.vertex_values(field, 0.0, keys, np.array([1], np.uint8), attr)
    b = mt3d_values.vertex_values(field, 0.0, keys, np.array([0], np.uint8), attr)
    assert a[0] == 0.1 + 0.5 * (0.7 - 0.1) and b[0] == 0.7 + 0.5 * (0.1 - 0.7)
    assert a[0] != b[0]


def test_components_and_integer_samples():
    rng = np.random.default_rng(0)
    field = rng.standard_normal((6, 7, 9))
    r = mt3d.extract(field, 0.1)
    attr = rng.integers(0, 65536, size=(6, 7, 9, 3)).astype(np.uint16)
    v = mt3d_values.vertex_values(field, 0.1, r["keys"], r["lowmin"], attr)
    assert v.shape == (len(r["keys"]), 3)
    assert np.array_equal(v, mt3d_values.vertex_values(field, 0.1, r["keys"], r["lowmin"], attr.astype(np.float64)))
    for c in range(3):
        assert np.array_equal(v[:, c], mt3d_values.vertex_values(field, 0.1, r["keys"], r["lowmin"], attr[..., c]))


def test_new_symbols_declared_and_exported():
    from test_capi_symbols import declared_symbols
    from contourist_b200 import build, engine
    syms = declared_symbols()
    for s in ("ctr_mt3d_interpolate", "ctr_mt3d_interpolate_fetch", "ctr_mt3d_interpolate_device_ptr"):
        assert s in syms
    build.build()
    lib = engine.load_library()
    p = engine.AttrParams()
    assert lib.ctr_mt3d_interpolate(None, ctypes.byref(p), None) == -1       # null context, no CUDA touched
    assert lib.ctr_mt3d_interpolate_fetch(None, None) == -1
    assert ctypes.sizeof(engine.AttrParams) == 24


def test_facade_passes_vertex_fields_to_the_maker():
    from contourist_b200 import tetrahedral
    f = lambda x, y, z: x * x + y * y + z * z
    t = tetrahedral.TriangulatedIsosurfaces((-1, -1, -1), (1, 1, 1), (0.25, 0.25, 0.25), f, 0.5, [])
    t.vertex_fields = [lambda x, y, z: x + 0 * y + 0 * z]
    m = t._configure(t.contour_maker)
    assert m.vertex_fields is t.vertex_fields and m.field_grid is t.grid
    s = m._samples_of(t.vertex_fields[0], components=True)
    assert s.shape == t.grid.samples(1).shape and s[1, 0, 0] == -0.75
    assert tetrahedral.GridContour3d.vertex_fields is None and tetrahedral.GridContour3d.vertex_values is None
    grid_maker = tetrahedral.Grid3DContour(4, 4, 4, np.zeros((5, 5, 5)), 0.5, None)
    assert grid_maker._samples_of(lambda i, j, k: i + 0 * j + 0 * k)[3, 0, 0] == 3.0
    assert grid_maker._samples_of(np.zeros((5, 5, 5, 2)), components=True).shape == (5, 5, 5, 2)
    with pytest.raises(ValueError):
        grid_maker._samples_of(np.zeros((5, 5, 5, 2)))
    with pytest.raises(ValueError):
        grid_maker._samples_of(np.zeros((5, 5, 6)), components=True)
