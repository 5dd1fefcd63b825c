"""CPU: the sample-type map of the Python binding (no device needed)."""
import numpy as np
import pytest

from contourist_b200 import engine as E


def test_native_codes():
    assert E.dtype_code(np.float32) == E.F32 == 0
    assert E.dtype_code(np.float64) == E.F64 == 1
    assert E.dtype_code(np.uint8) == E.U8 == 2
    assert E.dtype_code(np.int16) == E.I16 == 3
    assert E.dtype_code(np.uint16) == E.U16 == 4
    assert E.dtype_code(None) == E.F64                       # np.dtype(None) is float64, as before


@pytest.mark.parametrize("dt", [np.int8, np.int32, np.uint32, np.int64, np.float16, np.bool_, ">u2", ">f4"])
def test_other_types_have_no_code(dt):
    assert E.dtype_code(dt) is None


def test_float_only_entry_points():
    assert E.dtype_code(np.float32, E.FLOAT_CODES) == E.F32
    for dt in (np.uint8, np.int16, np.uint16):
        assert E.dtype_code(dt, E.FLOAT_CODES) is None
        with pytest.raises(ValueError):
            E._device_code(dt, E.FLOAT_CODES)
    with pytest.raises(ValueError):
        E._device_code(np.int32, tuple(E.DTYPE_CODES.values()))


def test_host_fields():
    a = np.arange(27, dtype=np.uint16).reshape(3, 3, 3)
    assert E._host_field(a, 3, tuple(E.DTYPE_CODES.values())).dtype == np.uint16          # passed through
    assert E._host_field(a, 3, E.FLOAT_CODES).dtype == np.float64                          # 2D / 4D: widened
    assert E._host_field(a.astype(np.int32), 3, tuple(E.DTYPE_CODES.values())).dtype == np.float64
    assert E._host_field(a.astype(">u2"), 3, tuple(E.DTYPE_CODES.values())).dtype == np.float64
    with pytest.raises(ValueError):
        E._host_field(a, 2, E.FLOAT_CODES)
