"""ctypes binding of libcontourist_b200.so (include/contourist_b200.h).

This is the only way the Python package computes anything: there is NO CPU fallback.  If the
shared library is missing or no CUDA device is usable the import / constructor raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTR_LIB") or os.path.join(_HERE, "libcontourist_b200.so")   # CTR_LIB: experiment builds

F32, F64, U8, I16, U16 = 0, 1, 2, 3, 4
FIELD_ON_DEVICE = 1
GEOM_F64 = 2
WANT_NORMALS = 4
WANT_KEYS = 8
WANT_CODES = 16
NO_GEOMETRY = 32
WANT_MINMAX = 64
MORPH = 128


class EngineError(RuntimeError):
    pass


# sample type codes (ctr_dtype) of the native sample types; the 2D and 4D runs take the float types only
DTYPE_CODES = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.uint8): U8, np.dtype(np.int16): I16,
               np.dtype(np.uint16): U16}
FLOAT_CODES = (F32, F64)


def dtype_code(dtype, accepted=tuple(DTYPE_CODES.values())):
    """ctr_dtype code of a native sample type (None -> float64), or None when the entry point does not read it."""
    code = DTYPE_CODES.get(np.dtype(dtype))
    return code if code in accepted else None


def _host_field(field, ndim, accepted):
    """C-contiguous array of a type the entry point reads natively; any other type is widened to float64."""
    if dtype_code(field.dtype, accepted) is None:
        field = field.astype(np.float64)
    field = np.ascontiguousarray(field)
    if field.ndim != ndim:
        raise ValueError("%dD field expected" % ndim)
    return field


def _device_code(dtype, accepted):
    code = dtype_code(dtype, accepted)
    if code is None:
        raise ValueError("device field of dtype %s: this entry point reads %s" % (
            np.dtype(dtype), ", ".join(str(d) for d, c in DTYPE_CODES.items() if c in accepted)))
    return code


class Mt3dParams(ctypes.Structure):
    _fields_ = [("field", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("n0", ctypes.c_int64), ("n1", ctypes.c_int64), ("n2", ctypes.c_int64),
                ("isovalue", ctypes.c_double), ("origin", ctypes.c_double * 3), ("delta", ctypes.c_double * 3),
                ("i_lo", ctypes.c_int64), ("i_hi", ctypes.c_int64), ("plane_offset", ctypes.c_int64),
                ("vert_id_base", ctypes.c_int64)]


class AttrParams(ctypes.Structure):
    _fields_ = [("field", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("ncomp", ctypes.c_int32), ("reserved", ctypes.c_int32)]


# ctr_mt3d_component (include/contourist_b200.h), 112 bytes: one row of Engine.mt3d_components()'s table
COMPONENT_DTYPE = np.dtype([("n_tris", "<i8"), ("n_verts", "<i8"), ("n_edges", "<i8"), ("n_boundary_edges", "<i8"),
                            ("n_nonmanifold_edges", "<i8"), ("first_tri", "<i8"), ("area", "<f8"), ("volume", "<f8"),
                            ("lo", "<f8", (3,)), ("hi", "<f8", (3,))])


class CleanParams(ctypes.Structure):
    _fields_ = [("corner", ctypes.c_int64 * 3), ("divisions", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("epsilon", ctypes.c_double), ("origin", ctypes.c_double * 3), ("delta", ctypes.c_double * 3)]


class CleanCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tris", ctypes.c_int64), ("n_quantized", ctypes.c_int64),
                ("n_tiny", ctypes.c_int64), ("n_flat", ctypes.c_int64), ("n_components", ctypes.c_int64),
                ("n_flipped", ctypes.c_int64)]


class SmoothParams(ctypes.Structure):
    _fields_ = [("iterations", ctypes.c_int32), ("reserved", ctypes.c_uint32), ("lam", ctypes.c_double),
                ("mu", ctypes.c_double)]


class SmoothCounts(ctypes.Structure):
    _fields_ = [("n_edges", ctypes.c_int64), ("n_fixed_verts", ctypes.c_int64)]


class DecimateParams(ctypes.Structure):
    _fields_ = [("cell", ctypes.c_double * 3), ("origin", ctypes.c_double * 3)]


class DecimateCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tris", ctypes.c_int64), ("n_clusters", ctypes.c_int64),
                ("n_collapsed", ctypes.c_int64), ("n_duplicate", ctypes.c_int64)]


class CapParams(ctypes.Structure):
    _fields_ = [("side", ctypes.c_int32), ("reserved", ctypes.c_uint32)]


class CapCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tris", ctypes.c_int64), ("n_cap_verts", ctypes.c_int64),
                ("n_cap_tris", ctypes.c_int64), ("n_missing", ctypes.c_int64)]


CAP_SIDES = {"high": 0, "low": 1}


class SectionParams(ctypes.Structure):
    _fields_ = [("normal", ctypes.c_double * 3), ("offsets", ctypes.c_void_p), ("nplanes", ctypes.c_int32),
                ("reserved", ctypes.c_uint32)]


class SectionCounts(ctypes.Structure):
    _fields_ = [("n_segments", ctypes.c_int64), ("n_polylines", ctypes.c_int64), ("n_points", ctypes.c_int64),
                ("n_junction_planes", ctypes.c_int64)]


class ClipParams(ctypes.Structure):
    _fields_ = [("source", ctypes.c_int32), ("side", ctypes.c_int32), ("normal", ctypes.c_double * 3),
                ("offset", ctypes.c_double), ("component", ctypes.c_int32), ("reserved", ctypes.c_uint32)]


class ClipCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tris", ctypes.c_int64), ("n_new_verts", ctypes.c_int64),
                ("n_cut_tris", ctypes.c_int64), ("n_dropped_tris", ctypes.c_int64)]


CLIP_PLANE, CLIP_VALUE = 0, 1
CLIP_SIDES = {"high": 0, "low": 1}


class PolyCounts(ctypes.Structure):
    _fields_ = [("n_polylines", ctypes.c_int64), ("n_points", ctypes.c_int64), ("junction_levels", ctypes.c_uint64)]


class Mt3dCounts(ctypes.Structure):
    _fields_ = [("n_verts", ctypes.c_int64), ("n_tris", ctypes.c_int64), ("n_active_cells", ctypes.c_int64),
                ("n_crossings", ctypes.c_int64), ("n_codes", ctypes.c_int64),
                ("fmin", ctypes.c_double), ("fmax", ctypes.c_double)]


_lib = None


def load_library():
    """Load the CUDA shared library; raise (never fall back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineError(
            "contourist_b200: %s not found. Build it with `python -m contourist_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32
    lib.ctr_create.argtypes = [i32, ctypes.POINTER(vp)]
    lib.ctr_create.restype = i32
    lib.ctr_destroy.argtypes = [vp]
    lib.ctr_destroy.restype = None
    lib.ctr_last_error.argtypes = [vp]
    lib.ctr_last_error.restype = ctypes.c_char_p
    lib.ctr_set_stream.argtypes = [vp, vp]
    lib.ctr_set_stream.restype = i32
    lib.ctr_set_timing.argtypes = [vp, i32]
    lib.ctr_set_timing.restype = i32
    lib.ctr_stage_times.argtypes = [vp, ctypes.POINTER(ctypes.c_float), i32]
    lib.ctr_stage_times.restype = i32
    lib.ctr_kernel_launches.argtypes = [vp]
    lib.ctr_kernel_launches.restype = i64
    lib.ctr_mt3d_run.argtypes = [vp, ctypes.POINTER(Mt3dParams), ctypes.POINTER(Mt3dCounts)]
    lib.ctr_mt3d_run.restype = i32
    lib.ctr_mt3d_enqueue.argtypes = [vp, ctypes.POINTER(Mt3dParams)]
    lib.ctr_mt3d_enqueue.restype = i32
    lib.ctr_mt3d_finish.argtypes = [vp, ctypes.POINTER(Mt3dCounts)]
    lib.ctr_mt3d_finish.restype = i32
    lib.ctr_mt3d_offset_ids.argtypes = [vp, i64]
    lib.ctr_mt3d_offset_ids.restype = i32
    lib.ctr_mt3d_publish_counts.argtypes = [vp, vp]
    lib.ctr_mt3d_publish_counts.restype = i32
    lib.ctr_mt3d_fetch.argtypes = [vp] + [vp] * 7
    lib.ctr_mt3d_fetch.restype = i32
    lib.ctr_mt3d_device_ptrs.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp)]
    lib.ctr_mt3d_device_ptrs.restype = i32
    lib.ctr_mt3d_orient_reference.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.ctr_mt3d_orient_reference.restype = i32
    lib.ctr_mt3d_select_seeded.argtypes = [vp, vp, i64, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.ctr_mt3d_select_seeded.restype = i32
    lib.ctr_mt3d_clean.argtypes = [vp, ctypes.POINTER(CleanParams), ctypes.POINTER(CleanCounts)]
    lib.ctr_mt3d_clean.restype = i32
    lib.ctr_mt3d_components.argtypes = [vp, ctypes.POINTER(i64)]
    lib.ctr_mt3d_components.restype = i32
    lib.ctr_mt3d_components_fetch.argtypes = [vp, vp, vp]
    lib.ctr_mt3d_components_fetch.restype = i32
    lib.ctr_mt3d_keep_components.argtypes = [vp, vp, i64, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.ctr_mt3d_keep_components.restype = i32
    lib.ctr_mt3d_smooth.argtypes = [vp, ctypes.POINTER(SmoothParams), ctypes.POINTER(SmoothCounts)]
    lib.ctr_mt3d_smooth.restype = i32
    lib.ctr_mt3d_decimate.argtypes = [vp, ctypes.POINTER(DecimateParams), ctypes.POINTER(DecimateCounts)]
    lib.ctr_mt3d_decimate.restype = i32
    lib.ctr_mt3d_cap.argtypes = [vp, ctypes.POINTER(CapParams), ctypes.POINTER(CapCounts)]
    lib.ctr_mt3d_cap.restype = i32
    lib.ctr_mt3d_section.argtypes = [vp, ctypes.POINTER(SectionParams), ctypes.POINTER(SectionCounts)]
    lib.ctr_mt3d_section.restype = i32
    lib.ctr_mt3d_section_segments_fetch.argtypes = [vp] * 4
    lib.ctr_mt3d_section_segments_fetch.restype = i32
    lib.ctr_mt3d_section_polylines_fetch.argtypes = [vp] * 9
    lib.ctr_mt3d_section_polylines_fetch.restype = i32
    lib.ctr_mt3d_clip.argtypes = [vp, ctypes.POINTER(ClipParams), ctypes.POINTER(ClipCounts)]
    lib.ctr_mt3d_clip.restype = i32
    lib.ctr_mt3d_interpolate.argtypes = [vp, ctypes.POINTER(AttrParams), ctypes.POINTER(i64)]
    lib.ctr_mt3d_interpolate.restype = i32
    lib.ctr_mt3d_interpolate_fetch.argtypes = [vp, vp]
    lib.ctr_mt3d_interpolate_fetch.restype = i32
    lib.ctr_mt3d_interpolate_device_ptr.argtypes = [vp, ctypes.POINTER(vp)]
    lib.ctr_mt3d_interpolate_device_ptr.restype = i32
    lib.ctr_comm_unique_id.argtypes = [vp]
    lib.ctr_comm_unique_id.restype = i32
    lib.ctr_comm_init.argtypes = [vp, vp, i32, i32]
    lib.ctr_comm_init.restype = i32
    lib.ctr_comm_destroy.argtypes = [vp]
    lib.ctr_comm_destroy.restype = i32
    lib.ctr_allgather_offsets.argtypes = [vp, vp, vp, vp]
    lib.ctr_allgather_offsets.restype = i32
    lib.ctr_gather_mesh.argtypes = [vp, i32, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.ctr_gather_mesh.restype = i32
    lib.ctr_gathered_fetch.argtypes = [vp, vp, vp, vp]
    lib.ctr_gathered_fetch.restype = i32
    lib.ctr_mt2d_polylines.argtypes = [vp, ctypes.POINTER(PolyCounts)]
    lib.ctr_mt2d_polylines.restype = i32
    lib.ctr_mt2d_polylines_fetch.argtypes = [vp] + [vp] * 6
    lib.ctr_mt2d_polylines_fetch.restype = i32
    lib.ctr_host_alloc.argtypes = [vp, ctypes.c_uint64, ctypes.POINTER(vp)]
    lib.ctr_host_alloc.restype = i32
    lib.ctr_host_free.argtypes = [vp, vp]
    lib.ctr_host_free.restype = i32
    lib.ctr_stage_upload.argtypes = [vp, vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.POINTER(vp)]
    lib.ctr_stage_upload.restype = i32
    lib.ctr_wait_for.argtypes = [vp, vp]
    lib.ctr_wait_for.restype = i32
    _bind_optional(lib)
    _lib = lib
    return lib


def _bind_optional(lib):
    """2D / 4D / post-processing entry points (bound when present in this build)."""
    from . import _bindings
    _bindings.bind(lib)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Engine(object):
    """One context = one device + one stream.  Not thread-safe."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.ctr_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise EngineError("ctr_create(device=%d) failed (%d): %s" % (
                device, rc, self.lib.ctr_last_error(None).decode()))
        self.h = h
        self.device = device
        self.run_serial = 0           # bumped by every call that replaces or rewrites the device results

    def close(self):
        if getattr(self, "h", None):
            if self.__dict__.get("_xpool") is not None:
                self._xpool.shutdown(wait=True)
                self._xpool = None
            for name in ("_twin", "_uploader"):
                if self.__dict__.get(name) is not None:
                    self.__dict__[name].close()
                    self.__dict__[name] = None
            for ptr, _ in getattr(self, "_pinned", {}).values():
                self.lib.ctr_host_free(self.h, ptr)
            self._pinned = {}
            self.lib.ctr_destroy(self.h)
            self.h = None

    def pinned_empty(self, name, shape, dtype):
        """numpy array over page-locked host memory from a grow-only pool keyed by `name` (valid until the next
        request under the same name): device <-> host copies of it run at full PCIe rate."""
        pool = self.__dict__.setdefault("_pinned", {})
        dtype = np.dtype(dtype)
        need = int(np.prod(shape)) * dtype.itemsize
        ptr, cap = pool.get(name, (None, 0))
        if cap < max(need, 1):
            if ptr:
                self._check(self.lib.ctr_host_free(self.h, ptr), "ctr_host_free")
            cap = max(need + need // 4, 4096)
            p = ctypes.c_void_p()
            self._check(self.lib.ctr_host_alloc(self.h, cap, ctypes.byref(p)), "ctr_host_alloc")
            ptr = p.value
            pool[name] = (ptr, cap)
        buf = (ctypes.c_char * max(need, 1)).from_address(ptr)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.ctr_last_error(self.h).decode()
            if rc == -1:
                raise ValueError("%s: %s" % (what, msg))
            raise EngineError("%s failed (%d): %s" % (what, rc, msg))

    def set_stream(self, cuda_stream):
        self._check(self.lib.ctr_set_stream(self.h, ctypes.c_void_p(int(cuda_stream))), "ctr_set_stream")

    def set_timing(self, enabled=True):
        self._check(self.lib.ctr_set_timing(self.h, 1 if enabled else 0), "ctr_set_timing")

    def stage_times(self, n=8):
        buf = (ctypes.c_float * n)()
        self._check(self.lib.ctr_stage_times(self.h, buf, n), "ctr_stage_times")
        return [float(x) for x in buf]

    def kernel_launches(self):
        return int(self.lib.ctr_kernel_launches(self.h))

    def stage_upload(self, host, dst_offset, total_bytes):
        """Queue the copy of the C-contiguous array `host` to byte offset dst_offset of this context's staging buffer
        (grown to total_bytes first) and return the buffer's device address without waiting (ctr_stage_upload)."""
        base = ctypes.c_void_p()
        self._check(self.lib.ctr_stage_upload(self.h, ctypes.c_void_p(host.ctypes.data), int(dst_offset), int(host.nbytes),
                                              int(total_bytes), ctypes.byref(base)), "ctr_stage_upload")
        return int(base.value)

    def wait_for(self, other):
        """Work queued on this engine from now on starts when what `other` has queued so far is done (device-side)."""
        self._check(self.lib.ctr_wait_for(self.h, other.h), "ctr_wait_for")

    # ------------------------------------------------------------------ 3D
    def _mt3d_params(self, field, value, origin, delta, flags, i_lo, i_hi, plane_offset, shape, dtype, vert_id_base):
        p = Mt3dParams()
        if isinstance(field, np.ndarray):
            field = _host_field(field, 3, tuple(DTYPE_CODES.values()))
            self._keep = field
            p.field = field.ctypes.data
            p.dtype = dtype_code(field.dtype)
            shape = field.shape
            flags &= ~FIELD_ON_DEVICE
        else:
            p.field = int(field)
            p.dtype = _device_code(dtype, tuple(DTYPE_CODES.values()))
            flags |= FIELD_ON_DEVICE
        p.flags = flags
        p.n0, p.n1, p.n2 = (int(s) for s in shape)
        self._shape3 = (p.n0, p.n1, p.n2)                             # the array mt3d_interpolate's fields match
        p.isovalue = float(value)
        for a in range(3):
            p.origin[a] = float(origin[a])
            p.delta[a] = float(delta[a])
        p.i_lo = int(i_lo)
        p.i_hi = int(p.n0 if i_hi is None else i_hi)
        p.plane_offset = int(plane_offset)
        p.vert_id_base = int(vert_id_base)
        return p, flags

    def mt3d_run(self, field, value, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), flags=0,
                 i_lo=0, i_hi=None, plane_offset=0, shape=None, dtype=None, vert_id_base=0):
        """field: C-contiguous numpy array [n0,n1,n2], or an integer device pointer (then pass shape, dtype and
        FIELD_ON_DEVICE).  float32, float64, uint8, int16 and uint16 samples are read as they are (an integer field gives
        exactly the result of its float64 copy); host arrays of any other type are widened to float64, device fields
        of any other type raise ValueError.  Returns Mt3dCounts."""
        p, flags = self._mt3d_params(field, value, origin, delta, flags, i_lo, i_hi, plane_offset, shape, dtype, vert_id_base)
        c = Mt3dCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_run(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_run")
        self._last3 = (flags, c)
        return c

    def mt3d_enqueue(self, field, value, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), flags=0,
                     i_lo=0, i_hi=None, plane_offset=0, shape=None, dtype=None, vert_id_base=0):
        """Queue an extraction on the stream and return at once; mt3d_finish() waits for it and returns the counts."""
        p, flags = self._mt3d_params(field, value, origin, delta, flags, i_lo, i_hi, plane_offset, shape, dtype, vert_id_base)
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_enqueue(self.h, ctypes.byref(p)), "ctr_mt3d_enqueue")
        self._pending3 = flags

    def mt3d_publish_counts(self, device_ptr):
        """Every following 3D run also stores (n_verts, n_tris) as two int64 at this device address, on the engine's
        stream, behind its last kernel (None: off): a collective can send the counts without a host round trip."""
        self._check(self.lib.ctr_mt3d_publish_counts(self.h, ctypes.c_void_p(int(device_ptr)) if device_ptr else None),
                    "ctr_mt3d_publish_counts")

    # ------------------------------------------------------------------ multi-GPU (NCCL inside the library)
    @staticmethod
    def comm_unique_id():
        """128-byte NCCL id (rank 0 makes it, the host sends it to the other ranks by any means)."""
        lib = load_library()
        buf = ctypes.create_string_buffer(128)
        rc = lib.ctr_comm_unique_id(buf)
        if rc != 0:
            raise EngineError("ctr_comm_unique_id failed (%d): NCCL could not be loaded" % rc)
        return buf.raw

    def comm_init(self, unique_id, rank, nranks):
        self._comm = (int(rank), int(nranks))
        self._check(self.lib.ctr_comm_init(self.h, ctypes.c_char_p(bytes(unique_id)), int(rank), int(nranks)), "ctr_comm_init")

    def comm_destroy(self):
        self._check(self.lib.ctr_comm_destroy(self.h), "ctr_comm_destroy")

    def allgather_offsets(self):
        """NCCL all-gather of the last 3D run's device counts.  Returns (counts [nranks, 2], this rank's exclusive
        (vertex, triangle) offsets, totals)."""
        rank, nranks = self._comm
        counts = np.zeros((nranks, 2), dtype=np.int64)
        off = np.zeros(2, dtype=np.int64)
        tot = np.zeros(2, dtype=np.int64)
        self._check(self.lib.ctr_allgather_offsets(self.h, _ptr(counts), _ptr(off), _ptr(tot)), "ctr_allgather_offsets")
        return counts, off, tot

    def gather_mesh(self, root=0):
        """Collective: the ranks' meshes to `root` (ncclSend / ncclRecv of what each rank has).  On the root returns
        dict(verts, normals, tris) with global triangle ids; None elsewhere."""
        rank, nranks = self._comm
        tv, tt = ctypes.c_int64(), ctypes.c_int64()
        self._check(self.lib.ctr_gather_mesh(self.h, int(root), ctypes.byref(tv), ctypes.byref(tt)), "ctr_gather_mesh")
        if rank != root:
            return None
        flags, _ = self._last3
        gd = np.float64 if flags & GEOM_F64 else np.float32
        V, T = int(tv.value), int(tt.value)
        a_v = np.empty((V, 3), gd)
        a_n = np.empty((V, 3), gd) if flags & WANT_NORMALS else None
        a_t = np.empty((T, 3), np.int32)
        self._check(self.lib.ctr_gathered_fetch(self.h, _ptr(a_v), _ptr(a_n), _ptr(a_t)), "ctr_gathered_fetch")
        return dict(verts=a_v, normals=a_n, tris=a_t)

    def mt3d_finish(self):
        c = Mt3dCounts()
        self._check(self.lib.ctr_mt3d_finish(self.h, ctypes.byref(c)), "ctr_mt3d_finish")
        self._last3 = (self._pending3, c)
        return c

    def mt3d_orient_reference(self):
        """Rewind the last run's device triangles with the reference's outward rule (surface_geometry.py:52-140);
        returns (components, triangles reversed).  Fetch afterwards."""
        nc, nf = ctypes.c_int64(), ctypes.c_int64()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_orient_reference(self.h, ctypes.byref(nc), ctypes.byref(nf)), "ctr_mt3d_orient_reference")
        return int(nc.value), int(nf.value)

    def _mesh_edited(self, n_verts, n_tris):
        "a pass has dropped rows of the device mesh: the new counts, which mt3d_fetch sizes its arrays from"
        flags, c = self._last3
        c = type(c).from_buffer_copy(c)                                # the caller keeps the full scan's counts
        c.n_verts, c.n_tris = int(n_verts), int(n_tris)
        self._last3 = (flags, c)

    def mt3d_select_seeded(self, start_voxels):
        """Keep only what the reference's flood fill reaches from these voxel origins ([n, 3] ints, the output of
        find_initial_voxels): tetrahedral.py:443-469 on the device mesh of the last full-volume run.
        Returns (n_verts, n_tris, emitting voxels selected); fetch afterwards."""
        sv = np.ascontiguousarray(np.asarray(start_voxels, dtype=np.int32).reshape(-1, 3))
        nv, nt, nc = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_select_seeded(self.h, _ptr(sv) if len(sv) else None, len(sv), ctypes.byref(nv),
                                                    ctypes.byref(nt), ctypes.byref(nc)), "ctr_mt3d_select_seeded")
        self._mesh_edited(nv.value, nt.value)
        return int(nv.value), int(nt.value), int(nc.value)

    def mt3d_clean(self, corner, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), divisions=10000, epsilon=1e-4, orient=False,
                   triangles=True):
        """The reference's post-processing of the last run's device mesh (tetrahedral.py:541-552: quantize, tiny, clean,
        optionally the outward orientation, then grid -> world).  The run must have used origin 0 / delta 1; the
        transform is applied here, last.  triangles=False skips clean_triangles (the reference's clean=False).
        Returns CleanCounts; fetch afterwards."""
        p = CleanParams()
        for a in range(3):
            p.corner[a] = int(corner[a])
            p.origin[a] = float(origin[a])
            p.delta[a] = float(delta[a])
        p.divisions = int(divisions)
        p.epsilon = float(epsilon)
        p.flags = (1 if orient else 0) | (0 if triangles else 2)
        c = CleanCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_clean(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_clean")
        self._mesh_edited(c.n_verts, c.n_tris)
        return c

    def mt3d_components(self):
        """Edge-connected components of the last 3D run's mesh as it stands now (after a selection, clean-up or
        orientation too): (tri_component [T] int32, row for row with mt3d_fetch()'s triangles, and table [C]
        COMPONENT_DTYPE), numbered by smallest triangle index (ctr_mt3d_components).  Per component: triangle, vertex
        and edge counts (n_verts - n_edges + n_tris is the Euler characteristic), boundary and non-manifold edges, fp64
        area, signed enclosed volume (> 0 around a region below the isovalue on the raw mesh, >= 0 for closed
        components after orientation) and the box lo / hi.  Not updated by a later selection or clean-up
        (mt3d_keep_components updates them)."""
        n = ctypes.c_int64()
        self._comp_shape = None
        self._check(self.lib.ctr_mt3d_components(self.h, ctypes.byref(n)), "ctr_mt3d_components")
        self._comp_shape = (int(self._last3[1].n_tris), int(n.value))
        return self.mt3d_components_fetch()

    def mt3d_components_fetch(self):
        """The current (tri_component, table) of the last mt3d_components(), as a later mt3d_keep_components() left
        them, without measuring again (ctr_mt3d_components_fetch)."""
        T, C = getattr(self, "_comp_shape", None) or (0, 0)   # (no results: the library refuses the fetch)
        labels = np.empty(T, np.int32)
        table = np.empty(C, COMPONENT_DTYPE)
        self._check(self.lib.ctr_mt3d_components_fetch(self.h, _ptr(labels) if T else None, _ptr(table) if C else None),
                    "ctr_mt3d_components_fetch")
        return labels, table

    def mt3d_keep_components(self, keep):
        """Keep the components named by `keep` on the device mesh and drop the others (ctr_mt3d_keep_components):
        `keep` is a boolean mask with one entry per component of the last mt3d_components(), or an array of component
        indices.  Kept triangles and vertices stay in order, ids renumbered; normals, keys and the values of an
        mt3d_interpolate() made on this mesh are compacted with them, and the component results are renumbered
        0..K-1 (mt3d_components_fetch()).  Returns (n_verts, n_tris); fetch afterwards."""
        C = (getattr(self, "_comp_shape", None) or (0, -1))[1]
        k = np.asarray(keep)
        if k.dtype == np.bool_:
            if C >= 0 and k.shape != (C,):
                raise ValueError("keep mask of shape %r: the last mt3d_components() found %d components" % (k.shape, C))
            mask = k.astype(np.uint8)
        elif k.size == 0 or np.issubdtype(k.dtype, np.integer):
            idx = k.astype(np.int64).reshape(-1)
            if len(idx) and (idx.min() < 0 or idx.max() >= max(C, 0)):
                raise ValueError("component index outside [0, %d)" % max(C, 0))
            mask = np.zeros(max(C, 0), np.uint8)
            mask[idx] = 1
        else:
            raise TypeError("keep: a boolean mask or integer component indices, not %s" % k.dtype)
        mask = np.ascontiguousarray(mask)
        nv, nt = ctypes.c_int64(), ctypes.c_int64()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_keep_components(self.h, _ptr(mask) if len(mask) else None, len(mask), ctypes.byref(nv),
                                                      ctypes.byref(nt)), "ctr_mt3d_keep_components")
        self._mesh_edited(nv.value, nt.value)
        self._comp_shape = (int(nt.value), int(mask.astype(bool).sum()))
        return int(nv.value), int(nt.value)

    def mt3d_smooth(self, iterations=10, lam=0.5, mu=-0.53):
        """Taubin lambda|mu smoothing of the last 3D run's device mesh as it stands now, in place (ctr_mt3d_smooth;
        oracle/mt3d_smooth.py is the definition): each iteration moves every free vertex by lam, then by mu, towards
        the average of its edge neighbours (mu=0: plain Laplacian smoothing, which shrinks).  Vertices on boundary or
        non-manifold edges stay bit for bit; normals (WANT_NORMALS) are recomputed; triangles and keys do not change.
        Afterwards mt3d_components() must measure again before mt3d_keep_components(), and mt3d_select_seeded() /
        mt3d_clean() are refused.  Returns SmoothCounts (n_edges, n_fixed_verts); fetch afterwards."""
        p = SmoothParams()
        p.iterations = int(iterations)
        p.lam = float(lam)
        p.mu = float(mu)
        c = SmoothCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_smooth(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_smooth")
        return c

    def mt3d_decimate(self, cell, origin=(0.0, 0.0, 0.0)):
        """Quadric vertex-clustering decimation of the last 3D run's device mesh as it stands now, in place
        (ctr_mt3d_decimate; oracle/mt3d_decimate.py is the definition): the vertices in one cell of the grid of edge
        lengths `cell` (a number or 3 numbers, in the units of the current positions) with its corner at `origin`
        become one vertex, placed where the planes of the triangles around it meet best (a corner or ridge inside a
        cell survives) and clamped to the cell.  Triangles left with fewer than three cells, and repeats of an earlier
        triangle's three cells, are dropped; the rest keep their order.  Each output vertex carries the keys of its
        cell's smallest vertex id (mt3d_interpolate() then samples the field there); normals (WANT_NORMALS) are
        recomputed.  Afterwards mt3d_components() must measure again before mt3d_keep_components(), and
        mt3d_select_seeded() / mt3d_clean() are refused.  Returns DecimateCounts (n_verts, n_tris, n_clusters,
        n_collapsed, n_duplicate); fetch afterwards."""
        p = DecimateParams()
        cell = np.broadcast_to(np.asarray(cell, np.float64), (3,))
        origin = np.broadcast_to(np.asarray(origin, np.float64), (3,))
        for a in range(3):
            p.cell[a] = float(cell[a])
            p.origin[a] = float(origin[a])
        c = DecimateCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_decimate(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_decimate")
        self._mesh_edited(c.n_verts, c.n_tris)
        return c

    def mt3d_cap(self, side):
        """Close the last 3D run's device mesh at the faces of the volume's box (ctr_mt3d_cap; oracle/mt3d_cap.py is the
        definition): side "high" closes the region f >= value, "low" the region f < value.  On every box face the part
        of each face triangle of the tetrahedral grid on that side is appended; its rim vertices are the surface's own,
        and the box-surface grid points it uses become new vertices (key lin * 8 + 0), so the region's boundary is
        closed.  The run needs WANT_KEYS; accepted on the mesh as extracted or smoothed (smooth first for flat caps),
        refused after a selection, clean-up, component filter, decimation, orientation or an earlier cap.  Device
        pointers must be taken again afterwards.  Returns CapCounts (n_verts, n_tris, n_cap_verts, n_cap_tris,
        n_missing); fetch afterwards."""
        if side not in CAP_SIDES:
            raise ValueError("side must be 'high' or 'low', not %r" % (side,))
        p = CapParams()
        p.side = CAP_SIDES[side]
        c = CapCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_cap(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_cap")
        self._mesh_edited(c.n_verts, c.n_tris)
        return c

    def mt3d_section(self, normal, offsets):
        """Sections of the last 3D run's device mesh as it stands now with the planes {x : normal . x == offsets[l]}
        (ctr_mt3d_section; oracle/mt3d_section.py is the definition), `offsets` strictly increasing, in the units of
        the current positions.  The mesh is not edited.  Returns (segments, polylines):
          segments  = dict(plane [S] int32, edges [S, 2, 2] int32 (vertex-id pairs (min, max), start edge first),
                      points [S, 2, 3] in the geometry type), by triangle, then plane;
          polylines = one list per plane of (closed, consistent, points [k, 3], length, area), open ones first, then by
                      start key, or None for a junction plane (one that crosses a non-manifold edge: its segments are
                      not chained).  An outward-oriented closed surface gives counter-clockwise sections seen from
                      +normal, with area > 0 (the raw mesh is wound towards the high side)."""
        n = np.asarray(normal, np.float64).reshape(3)
        off = np.ascontiguousarray(np.asarray(offsets, np.float64).reshape(-1))
        p = SectionParams()
        for a in range(3):
            p.normal[a] = float(n[a])
        p.offsets = off.ctypes.data if len(off) else None
        p.nplanes = len(off)
        c = SectionCounts()
        self._check(self.lib.ctr_mt3d_section(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_section")
        flags, _ = self._last3
        gd = np.float64 if flags & GEOM_F64 else np.float32
        S, P, N = int(c.n_segments), int(c.n_polylines), int(c.n_points)
        seg = dict(plane=np.empty(S, np.int32), edges=np.empty((S, 2, 2), np.int32), points=np.empty((S, 2, 3), gd))
        self._check(self.lib.ctr_mt3d_section_segments_fetch(self.h, _ptr(seg["plane"]), _ptr(seg["edges"]),
                                                             _ptr(seg["points"])), "ctr_mt3d_section_segments_fetch")
        plane, fl, key = np.empty(P, np.int32), np.empty(P, np.uint8), np.empty(P, np.uint64)
        o, ln, meas = np.empty(P, np.uint32), np.empty(P, np.uint32), np.empty((P, 2), np.float64)
        pts, junction = np.empty((N, 3), gd), np.empty(len(off), np.uint8)
        self._check(self.lib.ctr_mt3d_section_polylines_fetch(self.h, _ptr(plane), _ptr(fl), _ptr(key), _ptr(o), _ptr(ln),
                                                              _ptr(meas), _ptr(pts), _ptr(junction)),
                    "ctr_mt3d_section_polylines_fetch")
        out = [None if junction[l] else [] for l in range(len(off))]
        for q in np.lexsort((key, fl & 1, plane)):
            out[int(plane[q])].append((bool(fl[q] & 1), bool(fl[q] & 2), pts[int(o[q]):int(o[q]) + int(ln[q])],
                                       float(meas[q, 0]), float(meas[q, 1])))
        return seg, out

    def mt3d_clip(self, normal=None, offset=0.0, keep="high", component=None):
        """Keep the part of the last 3D run's device mesh as it stands now on one side of a plane or of a vertex value,
        in place (ctr_mt3d_clip; oracle/mt3d_clip.py is the definition).  Give exactly one of `normal` (a plane:
        s = (n0 x + n1 y) + n2 z of each vertex, in the units of the current positions) and `component` (s = that
        component of the values of an mt3d_interpolate() made on the mesh as it stands).  keep="high" keeps
        s >= offset, "low" keeps s < offset.  Triangles across the cut are split at one new vertex per crossed edge
        (positions, normals and carried vertex values interpolated along the edge, keys from the kept end) and keep
        their winding; kept vertices stay in order, new ones follow.  Every vertex kept: nothing changes.  Accepted after
        every pass (six clips make a box); afterwards mt3d_select_seeded(), mt3d_clean() and mt3d_cap() are refused, and
        mt3d_components() must measure again before mt3d_keep_components().  Device pointers (mt3d_device_ptrs(),
        mt3d_interpolate_device_ptr()) must be taken again.  Returns ClipCounts (n_verts, n_tris, n_new_verts,
        n_cut_tris, n_dropped_tris); fetch afterwards."""
        if (normal is None) == (component is None):
            raise ValueError("give exactly one of normal (a plane clip) and component (a value clip)")
        if keep not in CLIP_SIDES:
            raise ValueError("keep must be 'high' or 'low', not %r" % (keep,))
        p = ClipParams()
        p.side = CLIP_SIDES[keep]
        p.offset = float(offset)
        if normal is not None:
            n = np.asarray(normal, np.float64).reshape(3)
            p.source = CLIP_PLANE
            for a in range(3):
                p.normal[a] = float(n[a])
        else:
            p.source = CLIP_VALUE
            p.component = int(component)
        c = ClipCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt3d_clip(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_clip")
        self._mesh_edited(c.n_verts, c.n_tris)
        return c

    def mt3d_closest(self, points, max_distance=np.inf, n=None, dtype=None):
        """Closest points of the last 3D run's device mesh as it stands now to query points (ctr_mt3d_closest;
        oracle/mt3d_closest.py is the definition).  points: numpy [P, 3] in the units of the current positions
        (float32 / float64 read as they are, other types widened to float64), or an integer device pointer with n and
        dtype (float32 or float64) -- e.g. another engine's vertices from mt3d_device_ptrs().  For each point: the
        closest point of the closest triangle (the smallest index on a tie), when it lies within max_distance.  The
        mesh is not edited; a tree over the triangles is built per call, so batch the points.  Returns
        (dict(distance [P] float64, triangle [P] int32, point [P, 3] float64), ClosestCounts (n_found, height)); a point
        not found has distance inf, triangle -1 and point NaN."""
        from ._bindings import ClosestCounts, ClosestParams
        p = ClosestParams()
        if isinstance(points, np.ndarray):
            if points.ndim != 2 or points.shape[1] != 3:
                raise ValueError("points of shape (P, 3) expected, not %r" % (points.shape,))
            if points.dtype not in (np.float32, np.float64):
                points = points.astype(np.float64)
            points = np.ascontiguousarray(points)
            p.points = points.ctypes.data if len(points) else None
            p.dtype = dtype_code(points.dtype)
            p.flags = 0
            P = len(points)
        else:
            if n is None or dtype is None:
                raise ValueError("device points need n and dtype")
            p.points = int(points)
            p.dtype = _device_code(dtype, FLOAT_CODES)
            p.flags = FIELD_ON_DEVICE
            P = int(n)
        p.n_points = P
        p.max_distance = float(max_distance)
        c = ClosestCounts()
        self._check(self.lib.ctr_mt3d_closest(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_closest")
        out = dict(distance=np.empty(P, np.float64), triangle=np.empty(P, np.int32), point=np.empty((P, 3), np.float64))
        self._check(self.lib.ctr_mt3d_closest_fetch(self.h, _ptr(out["distance"]), _ptr(out["triangle"]), _ptr(out["point"])),
                    "ctr_mt3d_closest_fetch")
        return out, c

    def mt3d_raycast(self, origins, directions, t_min=0.0, t_max=np.inf, n=None, dtype=None):
        """First hits of rays on the last 3D run's device mesh as it stands now (ctr_mt3d_raycast;
        oracle/mt3d_raycast.py is the definition).  origins, directions: numpy [R, 3] in the units of the current
        positions (one dtype for both: float32 / float64 read as they are, other types widened to float64), or two
        integer device pointers with n and dtype (float32 or float64) -- e.g. this engine's own vertices and normals
        from mt3d_device_ptrs() for wall thickness.  Directions need not be unit length: t is in units of |d|.  For
        each ray: the hit with the smallest t in [t_min, t_max] (the smallest triangle index on a tie), by the
        watertight test.  The mesh is not edited; a tree over the triangles is built per call, so batch the rays.
        Returns (dict(t [R] float64, triangle [R] int32, weights [R, 3] float64 (of the triangle's corners a, b, c),
        point [R, 3] float64, side [R] int8 (+1: the ray arrives from the side the triangle faces, -1: from behind)),
        RayCounts (n_hit, height)); a ray without a hit has t inf, triangle -1, weights and point NaN and side 0."""
        from ._bindings import RayCounts, RayParams
        p = RayParams()
        if isinstance(origins, np.ndarray) or isinstance(directions, np.ndarray):
            O, D = np.asarray(origins), np.asarray(directions)
            if O.ndim != 2 or O.shape[1] != 3 or D.shape != O.shape:
                raise ValueError("origins and directions of one shape (R, 3) expected, not %r and %r" % (O.shape, D.shape))
            if O.dtype != D.dtype or O.dtype not in (np.float32, np.float64):
                O, D = O.astype(np.float64), D.astype(np.float64)
            O, D = np.ascontiguousarray(O), np.ascontiguousarray(D)
            p.origins = O.ctypes.data if len(O) else None
            p.directions = D.ctypes.data if len(D) else None
            p.dtype = dtype_code(O.dtype)
            p.flags = 0
            R = len(O)
        else:
            if n is None or dtype is None:
                raise ValueError("device rays need n and dtype")
            p.origins, p.directions = int(origins), int(directions)
            p.dtype = _device_code(dtype, FLOAT_CODES)
            p.flags = FIELD_ON_DEVICE
            R = int(n)
        p.n_rays = R
        p.t_min, p.t_max = float(t_min), float(t_max)
        c = RayCounts()
        self._check(self.lib.ctr_mt3d_raycast(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt3d_raycast")
        out = dict(t=np.empty(R, np.float64), triangle=np.empty(R, np.int32), weights=np.empty((R, 3), np.float64),
                   point=np.empty((R, 3), np.float64), side=np.empty(R, np.int8))
        self._check(self.lib.ctr_mt3d_raycast_fetch(self.h, _ptr(out["t"]), _ptr(out["triangle"]), _ptr(out["weights"]),
                                                    _ptr(out["point"]), _ptr(out["side"])), "ctr_mt3d_raycast_fetch")
        return out, c

    def mt3d_interpolate(self, field, shape=None, dtype=None):
        """Values of another field at the vertices of the last 3D run's mesh as it stands now (after a selection or
        clean-up too), row for row with mt3d_fetch()'s vertices: a_low + ratio * (a_high - a_low) along each vertex's
        edge, with the ratio of its position (ctr_mt3d_interpolate; the run needs WANT_KEYS).  field: numpy array of
        the run's array shape [n0, n1, n2] or [n0, n1, n2, c] (c = 1..4), or an integer device pointer with shape and
        dtype.  Host arrays of float32 / float64 / uint8 / int16 / uint16 are read as they are, other types are widened
        to float64.  Returns [V] (or [V, c]) in the run's geometry type.  Values are not compacted by a later selection
        or clean-up: interpolate after the last one (mt3d_keep_components does compact them)."""
        p = AttrParams()
        codes = tuple(DTYPE_CODES.values())
        if isinstance(field, np.ndarray):
            if field.ndim not in (3, 4):
                raise ValueError("field of shape (n0, n1, n2) or (n0, n1, n2, c) expected")
            field = _host_field(field, field.ndim, codes)
            p.field = field.ctypes.data
            p.dtype = dtype_code(field.dtype)
            shape = field.shape
            p.flags = 0
        else:
            if shape is None or dtype is None:
                raise ValueError("a device field needs shape and dtype")
            p.field = int(field)
            p.dtype = _device_code(dtype, codes)
            p.flags = FIELD_ON_DEVICE
        shape = tuple(int(s) for s in shape)
        if len(shape) not in (3, 4) or shape[:3] != getattr(self, "_shape3", None):
            raise ValueError("field of shape %r: the last 3D run's array is %r" % (shape, getattr(self, "_shape3", None)))
        p.ncomp = shape[3] if len(shape) == 4 else 1
        n = ctypes.c_int64()
        self._check(self.lib.ctr_mt3d_interpolate(self.h, ctypes.byref(p), ctypes.byref(n)), "ctr_mt3d_interpolate")
        flags, _ = self._last3
        out = np.empty((int(n.value), int(p.ncomp)), np.float64 if flags & GEOM_F64 else np.float32)
        self._check(self.lib.ctr_mt3d_interpolate_fetch(self.h, _ptr(out)), "ctr_mt3d_interpolate_fetch")
        return out if len(shape) == 4 else out[:, 0]

    def mt3d_interpolate_device_ptr(self):
        """Device address of the last mt3d_interpolate()'s values (valid until the next run or interpolation)."""
        v = ctypes.c_void_p()
        self._check(self.lib.ctr_mt3d_interpolate_device_ptr(self.h, ctypes.byref(v)), "ctr_mt3d_interpolate_device_ptr")
        return v.value

    def mt3d_fetch(self, verts=True, normals=None, tris=True, keys=None, codes=None, pinned=False):
        """Copy the last run's outputs to host arrays.  pinned=True: the arrays live in the engine's page-locked pool
        (fast copies) and are overwritten by the next pinned fetch."""
        flags, c = self._last3
        empty = (lambda n, shape, dt: self.pinned_empty("mt3d_" + n, shape, dt)) if pinned else (lambda n, shape, dt: np.empty(shape, dtype=dt))
        gd = np.float64 if flags & GEOM_F64 else np.float32
        geom = not (flags & NO_GEOMETRY)
        out = {}
        if normals is None:
            normals = bool(flags & WANT_NORMALS)
        if keys is None:
            keys = bool(flags & WANT_KEYS)
        if codes is None:
            codes = bool(flags & WANT_CODES)
        V, T, C = int(c.n_verts), int(c.n_tris), int(c.n_codes)
        a_v = empty("v", (V, 3), gd) if (verts and geom) else None
        a_n = empty("n", (V, 3), gd) if (normals and geom) else None
        a_t = empty("t", (T, 3), np.int32) if (tris and geom) else None
        a_k = empty("k", (V,), np.uint64) if (keys and geom) else None
        a_l = empty("l", (V,), np.uint8) if (keys and geom) else None
        a_c = empty("c", (C,), np.int64) if codes else None
        a_d = empty("d", (C,), np.uint32) if codes else None
        self._check(self.lib.ctr_mt3d_fetch(self.h, _ptr(a_v), _ptr(a_n), _ptr(a_t), _ptr(a_k), _ptr(a_l),
                                            _ptr(a_c), _ptr(a_d)), "ctr_mt3d_fetch")
        out.update(verts=a_v, normals=a_n, tris=a_t, keys=a_k, lowmin=a_l, cells=a_c, codes=a_d)
        return out

    def mt3d_extract_host(self, field, value, origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0), flags=0, nslabs=8, own=None,
                          plane_offset=0):
        """Host array in, host mesh out, with the PCIe traffic of the two directions overlapped.

        The volume is cut into `nslabs` z-slabs (sharding.slab_with_halo, the multi-GPU decomposition).  An upload
        context sends the planes to the device ONCE, in slab order, on its own stream (ctr_stage_upload: a slab's halo
        planes are already there from its neighbour, so the host sends n0 planes, not n0 + 3 per slab); slab s is
        extracted from the staged planes on one of two alternating contexts as soon as its last plane has arrived
        (ctr_wait_for), while a worker thread downloads the mesh of slab s-1 from the other (PCIe is full duplex; ctypes
        releases the GIL), and slab s+1 is already queued (`ctr_mt3d_enqueue`) when the host waits for slab s, so the
        upload engine never idles.  Triangle ids are global: the vertex count of the slabs before a slab is added on
        the device (`ctr_mt3d_offset_ids`) before its download.  own=(A, B) restricts the call to owner planes
        [A, B) of the array (a rank's slab with its halo planes around it) and plane_offset is the global index of
        the array's first plane, as in ctr_mt3d_params.  `field` should be page-locked
        (Engine.pinned_empty) for full transfer rate.  Returns (totals dict, arrays dict); the arrays live in the
        engine's page-locked pool and are overwritten by the next call."""
        from concurrent.futures import ThreadPoolExecutor
        from . import sharding
        if not (isinstance(field, np.ndarray) and field.ndim == 3 and field.flags["C_CONTIGUOUS"]):
            raise ValueError("mt3d_extract_host needs a C-contiguous 3D numpy array")
        if dtype_code(field.dtype) is None:
            raise ValueError("float32 / float64 / uint8 / int16 / uint16 samples expected")
        flags &= ~(FIELD_ON_DEVICE | WANT_CODES | NO_GEOMETRY)
        n0 = field.shape[0]
        own_a, own_b = (0, n0) if own is None else (int(own[0]), int(own[1]))
        nslabs = max(1, min(int(nslabs), own_b - own_a - 1))
        twin = self.__dict__.get("_twin")
        if twin is None or twin.h is None:
            twin = self._twin = Engine(self.device)
        engines = (self, twin)
        up = self.__dict__.get("_uploader")
        if up is None or up.h is None:
            up = self._uploader = Engine(self.device)
        plane_bytes = field.shape[1] * field.shape[2] * field.itemsize
        pool = self.__dict__.setdefault("_xpool", ThreadPoolExecutor(max_workers=1))
        gd = np.float64 if flags & GEOM_F64 else np.float32
        gsz = np.dtype(gd).itemsize
        want_n, want_k = bool(flags & WANT_NORMALS), bool(flags & WANT_KEYS)
        cap_v, cap_t = self.__dict__.get("_xcap", (0, 0))
        bufs = {}

        def alloc(cv, ct):
            bufs["verts"] = self.pinned_empty("x_v", (cv, 3), gd)
            bufs["normals"] = self.pinned_empty("x_n", (cv, 3), gd) if want_n else None
            bufs["tris"] = self.pinned_empty("x_t", (ct, 3), np.int32)
            bufs["keys"] = self.pinned_empty("x_k", (cv,), np.uint64) if want_k else None
            bufs["lowmin"] = self.pinned_empty("x_l", (cv,), np.uint8) if want_k else None

        def fetch(eng, voff, toff, nv, nt):
            def at(a, off, item):
                return None if a is None else ctypes.c_void_p(a.ctypes.data + off * item)
            eng._check(eng.lib.ctr_mt3d_fetch(eng.h, at(bufs["verts"], voff, 3 * gsz), at(bufs["normals"], voff, 3 * gsz),
                                              at(bufs["tris"], toff, 12), at(bufs["keys"], voff, 8),
                                              at(bufs["lowmin"], voff, 1), None, None), "ctr_mt3d_fetch")

        for attempt in range(2):
            if cap_v and cap_t:
                alloc(cap_v, cap_t)
            pending = [None, None]
            vsum = tsum = 0
            totals = dict(n_active_cells=0, n_crossings=0)
            sizes = []
            overflow = False
            slabs = []
            for (a, b) in sharding.slab_bounds(own_b - own_a, nslabs):
                if b > a:
                    lo, hi, kw = sharding.slab_with_halo(a + own_a, b + own_a, n0)
                    kw["plane_offset"] += int(plane_offset)
                    slabs.append((lo, hi, kw))

            first = slabs[0][0] if slabs else 0              # planes [first, last) of the array are staged at offset 0
            last = slabs[-1][1] if slabs else 0
            sent = [first]

            def enqueue(k):
                # queued, not waited for: the planes slab k still lacks go up on the upload stream while the kernels of
                # slab k-1 run.  Its vertex ids start at 0; the base (vertices of the slabs before it) is added on the
                # device once it is known.
                lo, hi, kw = slabs[k]
                if pending[k & 1] is not None:
                    pending[k & 1].result()                   # the context's previous slab has been downloaded
                    pending[k & 1] = None
                base = up.stage_upload(field[sent[0]:max(hi, sent[0])], (sent[0] - first) * plane_bytes, (last - first) * plane_bytes)
                sent[0] = max(hi, sent[0])
                engines[k & 1].wait_for(up)
                engines[k & 1].mt3d_enqueue(base + (lo - first) * plane_bytes, value, origin=origin, delta=delta, flags=flags,
                                            shape=(hi - lo,) + tuple(field.shape[1:]), dtype=field.dtype, **kw)

            enqueue(0)
            for k in range(len(slabs)):
                if k + 1 < len(slabs):
                    enqueue(k + 1)
                eng = engines[k & 1]
                c = eng.mt3d_finish()
                nv, nt = int(c.n_verts), int(c.n_tris)
                sizes.append((nv, nt))
                totals["n_active_cells"] += int(c.n_active_cells)
                totals["n_crossings"] += int(c.n_crossings)
                if vsum:
                    eng._check(eng.lib.ctr_mt3d_offset_ids(eng.h, vsum), "ctr_mt3d_offset_ids")
                if not overflow and vsum + nv <= cap_v and tsum + nt <= cap_t:
                    if nv or nt:                              # (an empty slab has nothing to download; on a context's
                        pending[k & 1] = pool.submit(fetch, eng, vsum, tsum, nv, nt)   # first call there are no buffers yet)
                else:
                    overflow = True                           # first call (sizes unknown) or a larger mesh than before
                vsum += nv
                tsum += nt
            for f in pending:
                if f is not None:
                    f.result()
            cap_v = max(cap_v, vsum + vsum // 4 + 1024)
            cap_t = max(cap_t, tsum + tsum // 4 + 1024)
            self._xcap = (cap_v, cap_t)
            if not overflow:
                break
        totals.update(n_verts=vsum, n_tris=tsum, slabs=sizes)
        out = dict(verts=bufs["verts"][:vsum], normals=None if bufs["normals"] is None else bufs["normals"][:vsum],
                   tris=bufs["tris"][:tsum], keys=None if bufs["keys"] is None else bufs["keys"][:vsum],
                   lowmin=None if bufs["lowmin"] is None else bufs["lowmin"][:vsum], cells=None, codes=None)
        return totals, out

    # ------------------------------------------------------------------ 2D
    def mt2d_run(self, field, levels, origin=(0.0, 0.0), delta=(1.0, 1.0), flags=0, i_lo=0, i_hi=None,
                 row_offset=0, shape=None, dtype=None):
        """field: numpy [n0,n1] float32/float64 or device pointer (+shape, dtype); levels: strictly increasing."""
        from ._bindings import Mt2dParams, Mt2dCounts
        p = Mt2dParams()
        if isinstance(field, np.ndarray):
            field = _host_field(field, 2, FLOAT_CODES)
            self._keep = field
            p.field = field.ctypes.data
            p.dtype = dtype_code(field.dtype)
            shape = field.shape
            flags &= ~FIELD_ON_DEVICE
        else:
            p.field = int(field)
            p.dtype = _device_code(dtype, FLOAT_CODES)
            flags |= FIELD_ON_DEVICE
        lv = np.ascontiguousarray(np.asarray(levels, dtype=np.float64))
        self._keep_levels = lv
        p.flags = flags
        p.n0, p.n1 = (int(s) for s in shape)
        p.levels = lv.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        p.nlevels = int(lv.shape[0])
        for a in range(2):
            p.origin[a] = float(origin[a])
            p.delta[a] = float(delta[a])
        p.i_lo = int(i_lo)
        p.i_hi = int(p.n0 if i_hi is None else i_hi)
        p.row_offset = int(row_offset)
        c = Mt2dCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mt2d_run(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mt2d_run")
        self._last2 = (flags, c)
        return c

    def mt2d_fetch(self):
        flags, c = self._last2
        gd = np.float64 if flags & GEOM_F64 else np.float32
        S = int(c.n_segments)
        lvl = np.empty((S,), dtype=np.uint8)
        keys = np.empty((S, 2), dtype=np.uint64)
        pos = np.empty((S, 2, 2), dtype=gd)
        self._check(self.lib.ctr_mt2d_fetch(self.h, _ptr(lvl), _ptr(keys), _ptr(pos)), "ctr_mt2d_fetch")
        return dict(level=lvl, keys=keys, pos=pos)

    def mt2d_polylines(self):
        """Polylines of the last 2D run, chained on the device (ctr_mt2d_polylines).  Returns None when some level has a
        key on more than two segments (the caller chains such runs with triangulated.chain_segments), else a list per
        level index of (closed, points[k, 2]) in the canonical order: open contours first, by start key."""
        flags, c = self._last2
        pc = PolyCounts()
        self._check(self.lib.ctr_mt2d_polylines(self.h, ctypes.byref(pc)), "ctr_mt2d_polylines")
        if pc.junction_levels:
            return None
        P, N = int(pc.n_polylines), int(pc.n_points)
        gd = np.float64 if flags & GEOM_F64 else np.float32
        lvl = np.empty(P, np.int32)
        closed = np.empty(P, np.uint8)
        key = np.empty(P, np.uint64)
        off = np.empty(P, np.uint32)
        length = np.empty(P, np.uint32)
        pts = np.empty((N, 2), gd)
        if P:
            self._check(self.lib.ctr_mt2d_polylines_fetch(self.h, _ptr(lvl), _ptr(closed), _ptr(key), _ptr(off), _ptr(length),
                                                          _ptr(pts)), "ctr_mt2d_polylines_fetch")
        nlev = len(self._keep_levels)
        out = [[] for _ in range(nlev)]
        for q in np.lexsort((key, closed & 1, lvl)):
            out[int(lvl[q])].append((bool(closed[q]), pts[int(off[q]):int(off[q]) + int(length[q])]))
        return out

    # ------------------------------------------------------------------ 4D
    def mp4d_run(self, field, value, origin=(0.0,) * 4, delta=(1.0,) * 4, flags=0, nbins=100, shape=None, dtype=None):
        """field: numpy [n0,n1,n2,n3] float32/float64 (last axis = time) or device pointer (+shape, dtype)."""
        from ._bindings import Mp4dParams, Mp4dCounts
        p = Mp4dParams()
        if isinstance(field, np.ndarray):
            field = _host_field(field, 4, FLOAT_CODES)
            self._keep = field
            p.field = field.ctypes.data
            p.dtype = dtype_code(field.dtype)
            shape = field.shape
            flags &= ~FIELD_ON_DEVICE
        else:
            p.field = int(field)
            p.dtype = _device_code(dtype, FLOAT_CODES)
            flags |= FIELD_ON_DEVICE
        p.flags = flags
        p.n0, p.n1, p.n2, p.n3 = (int(s) for s in shape)
        p.isovalue = float(value)
        for a in range(4):
            p.origin[a] = float(origin[a])
            p.delta[a] = float(delta[a])
        p.nbins = int(nbins)
        c = Mp4dCounts()
        self.run_serial += 1
        self._check(self.lib.ctr_mp4d_run(self.h, ctypes.byref(p), ctypes.byref(c)), "ctr_mp4d_run")
        self._last4 = (flags, c, tuple(int(s) for s in shape))
        return c

    def mp4d_fetch(self, verts=True, tets=True, morph=None):
        flags, c, shape = self._last4
        gd = np.float64 if flags & GEOM_F64 else np.float32
        V, T, C, M = int(c.n_verts), int(c.n_tets), int(c.n_codes), int(c.n_morph_tris)
        keys = bool(flags & WANT_KEYS)
        codes = bool(flags & WANT_CODES)
        if morph is None:
            morph = bool(flags & MORPH)
        a_v = np.empty((V, 4), dtype=gd) if verts else None
        a_t = np.empty((T, 4), dtype=np.int32) if tets else None
        a_k = np.empty((V,), dtype=np.uint64) if keys else None
        a_l = np.empty((V,), dtype=np.uint8) if keys else None
        a_c = np.empty((C, 24), dtype=np.uint8) if codes else None
        a_i = np.empty((C,), dtype=np.int64) if codes else None
        a_mv = np.empty((V, 4), dtype=np.float64) if morph else None
        a_kp = np.empty((T,), dtype=np.uint8) if morph else None
        a_mt = np.empty((M, 3, 2), dtype=np.int32) if morph else None
        self._check(self.lib.ctr_mp4d_fetch(self.h, _ptr(a_v), _ptr(a_t), _ptr(a_k), _ptr(a_l), _ptr(a_c), _ptr(a_i),
                                            _ptr(a_mv), _ptr(a_kp), _ptr(a_mt)), "ctr_mp4d_fetch")
        cells = None
        if codes:
            # packed (word << 22 | bit << 17 | ...) -> linear hypervoxel index over the (n-1)^4 cell grid
            n0, n1, n2, n3 = shape
            W = (n3 + 31) // 32
            gw = (a_i.astype(np.uint64) >> np.uint64(22)).astype(np.int64)
            bit = ((a_i.astype(np.uint64) >> np.uint64(17)) & np.uint64(31)).astype(np.int64)
            row, w = gw // W, gw % W
            l = w * 32 + bit
            k = row % n2
            j = (row // n2) % n1
            i = row // (n2 * n1)
            cells = ((i * (n1 - 1) + j) * (n2 - 1) + k) * (n3 - 1) + l
        return dict(verts=a_v, tets=a_t, keys=a_k, lowmin=a_l, codes=a_c, cells=cells, morph_verts=a_mv, keep=a_kp,
                    morph_tris=a_mt)

    def mt3d_device_ptrs(self):
        v, n, t = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        self._check(self.lib.ctr_mt3d_device_ptrs(self.h, ctypes.byref(v), ctypes.byref(n), ctypes.byref(t)),
                    "ctr_mt3d_device_ptrs")
        return v.value, n.value, t.value


def canonical_mesh(out):
    """Key-sorted copy of an mt3d_fetch() result (needs WANT_KEYS).

    Vertex ids are an engine choice (deterministic, word-major; in this build they are the rank of the edge key).
    Parity checks must not depend on that choice: they sort here -- vertices / normals / keys / lowmin reordered
    by key, triangle ids remapped, triangle order kept."""
    keys = out["keys"]
    perm = np.argsort(keys, kind="stable")
    inv = np.empty(len(perm), dtype=np.int64)
    inv[perm] = np.arange(len(perm), dtype=np.int64)
    res = dict(out)
    for name in ("verts", "normals", "keys", "lowmin"):
        if out.get(name) is not None:
            res[name] = out[name][perm]
    if out.get("tris") is not None:
        t = out["tris"].astype(np.int64)
        local = t < len(perm)                      # ids >= n_verts belong to the next shard (sharded runs)
        res["tris"] = np.where(local, inv[np.minimum(t, len(perm) - 1)] if len(perm) else t, t).astype(out["tris"].dtype)
    return res


_default = {}


def default_engine(device=0):
    """Process-wide engine per device (contexts are cheap to keep, expensive to warm)."""
    e = _default.get(device)
    if e is None or e.h is None:
        e = _default[device] = Engine(device)
    return e
