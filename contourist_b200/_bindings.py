"""ctypes prototypes for the 2D / 4D / post-processing entry points, the closest-point query and the ray cast."""
import ctypes


class Mt2dParams(ctypes.Structure):
    _fields_ = [("field", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("n0", ctypes.c_int64), ("n1", ctypes.c_int64), ("levels", ctypes.POINTER(ctypes.c_double)),
                ("nlevels", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("origin", ctypes.c_double * 2), ("delta", ctypes.c_double * 2),
                ("i_lo", ctypes.c_int64), ("i_hi", ctypes.c_int64), ("row_offset", ctypes.c_int64)]


class Mt2dCounts(ctypes.Structure):
    _fields_ = [("n_segments", ctypes.c_int64), ("n_active_squares", ctypes.c_int64),
                ("fmin", ctypes.c_double), ("fmax", ctypes.c_double)]


class Mp4dParams(ctypes.Structure):
    _fields_ = [("field", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("n0", ctypes.c_int64), ("n1", ctypes.c_int64), ("n2", ctypes.c_int64), ("n3", ctypes.c_int64),
                ("isovalue", ctypes.c_double), ("origin", ctypes.c_double * 4), ("delta", ctypes.c_double * 4),
                ("nbins", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class Mp4dCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tets", ctypes.c_int64), ("n_active_cells", ctypes.c_int64),
                ("n_crossings", ctypes.c_int64), ("n_codes", ctypes.c_int64), ("n_morph_tris", ctypes.c_int64),
                ("fmin", ctypes.c_double), ("fmax", ctypes.c_double), ("t_min", ctypes.c_double), ("t_max", ctypes.c_double)]


class ClosestParams(ctypes.Structure):
    _fields_ = [("points", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("n_points", ctypes.c_int64), ("max_distance", ctypes.c_double)]


class ClosestCounts(ctypes.Structure):
    _fields_ = [("n_found", ctypes.c_int64), ("height", ctypes.c_int64)]


class RayParams(ctypes.Structure):
    _fields_ = [("origins", ctypes.c_void_p), ("directions", ctypes.c_void_p), ("dtype", ctypes.c_int32),
                ("flags", ctypes.c_uint32), ("n_rays", ctypes.c_int64), ("t_min", ctypes.c_double), ("t_max", ctypes.c_double)]


class RayCounts(ctypes.Structure):
    _fields_ = [("n_hit", ctypes.c_int64), ("height", ctypes.c_int64)]


def bind(lib):
    vp, i32 = ctypes.c_void_p, ctypes.c_int
    lib.ctr_mt2d_run.argtypes = [vp, ctypes.POINTER(Mt2dParams), ctypes.POINTER(Mt2dCounts)]
    lib.ctr_mt2d_run.restype = i32
    lib.ctr_mt2d_fetch.argtypes = [vp, vp, vp, vp]
    lib.ctr_mt2d_fetch.restype = i32
    lib.ctr_mp4d_run.argtypes = [vp, ctypes.POINTER(Mp4dParams), ctypes.POINTER(Mp4dCounts)]
    lib.ctr_mp4d_run.restype = i32
    lib.ctr_mp4d_fetch.argtypes = [vp] + [vp] * 9
    lib.ctr_mp4d_fetch.restype = i32
    lib.ctr_mt3d_closest.argtypes = [vp, ctypes.POINTER(ClosestParams), ctypes.POINTER(ClosestCounts)]
    lib.ctr_mt3d_closest.restype = i32
    lib.ctr_mt3d_closest_fetch.argtypes = [vp] * 4
    lib.ctr_mt3d_closest_fetch.restype = i32
    lib.ctr_mt3d_raycast.argtypes = [vp, ctypes.POINTER(RayParams), ctypes.POINTER(RayCounts)]
    lib.ctr_mt3d_raycast.restype = i32
    lib.ctr_mt3d_raycast_fetch.argtypes = [vp] * 6
    lib.ctr_mt3d_raycast_fetch.restype = i32
