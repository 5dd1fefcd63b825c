"""3D isosurfaces by marching tetrahedra -- drop-in for contourist/tetrahedral.py on the CUDA engine.

Same public names and signatures as the reference (tetrahedral.py:50-107,514-621): TriangulatedIsosurfaces,
Delta3DContour, Grid3DContour / GridContour3d with search_for_endpoints(), get_points_and_triangles(),
extract_surface_geometry().  Differences, all documented in DESIGN.md section 2:
  * `function` may be a numpy array of samples (N+1 per axis for N = grid_dimensions) besides a callable;
  * extraction is a FULL SCAN on the GPU.  Seeds from search_for_endpoints() (every crossing segment) keep it that
    way; explicit segment_endpoints at the grid level (Grid3DContour / GridContour3d) restrict the result to what
    the reference's tracker reaches from them: the start voxels are found on the host as in find_initial_voxels
    (tetrahedral.py:396-441, a few samples per seed) and the engine keeps the 26-connected components of border
    voxels that contain one (`ctr_mt3d_select_seeded`; expand_voxels, tetrahedral.py:443-469).  Start voxels outside
    the array (the reference's out-of-range "leak" voxels, which it can only evaluate through a callable) are
    ignored;
  * linear_interpolate=False (the callable evaluated off-grid) is not available: NotImplementedError;
  * points / triangles come back as numpy arrays (iterate / index them like the reference's lists);
  * get_points_and_triangles() returns what the reference returns (tetrahedral.py:541-552): the raw mesh after
    quantize_interpolations, remove_tiny_simplices, clean_triangles (when `clean`) and orient_triangles, all on the
    device (`ctr_mt3d_clean`), in the deterministic form of those passes ("smallest vertex id survives" wherever
    the reference depends on CPython dict / set order; oracle/post3d.py).  `post_process = False` on the maker
    gives the engine's raw indexed mesh instead, wound towards the high side (`reference_orientation=True` adds the
    reference's per-component outward flip to it);
  * search_for_endpoints() already runs the extraction (the crossing scan is its first two stages);
    get_points_and_triangles() then only post-processes and fetches that run.
"""
import numbers

import numpy as np

from . import engine as E
from . import grid_field
from . import surface_geometry

A = (0, 0, 0)
B = (0, 0, 1)
C = (0, 1, 0)
D = (0, 1, 1)
E_ = (1, 0, 0)
F = (1, 0, 1)
G = (1, 1, 0)
H = (1, 1, 1)
CUBE = np.array([A, B, C, D, E_, F, G, H], dtype=int)
TETRAHEDRA = np.array([[A, H, B, D], [A, H, D, C], [A, H, C, G], [A, H, G, E_], [A, H, E_, F], [A, H, F, B]], dtype=int)
OFFSETS = np.array([(i, j, k) for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1) if i != 0 or j != 0 or k != 0], dtype=int)


def initial_voxels(samples, value, end_points):
    """Start voxels of the reference's tracker for seed segments (tetrahedral.py:396-441 find_initial_voxels), on an
    array of samples: order low / high by value, integer bisection until the two points are adjacent, then each of
    them -- or the first of its 26 neighbours in OFFSETS order -- that is a border voxel (tetrahedral.py:383-394),
    with the reference's `visited` bookkeeping.  Voxels whose 8 samples are not all inside the array are not border
    voxels here.  Returns an int32 [n, 3] array of voxel origins."""
    samples = np.asarray(samples)
    top = np.array(samples.shape) - 2                     # last voxel origin per axis

    def f(p):
        if np.any(np.asarray(p) < 0) or np.any(np.asarray(p) > top + 1):
            raise ValueError("seed point %r outside the sample array of shape %r" % (tuple(int(x) for x in p), samples.shape))
        return float(samples[tuple(int(x) for x in p)])

    def border(p):
        p = np.asarray(p)
        if np.any(p < 0) or np.any(p > top):
            return False
        v = samples[p[0]:p[0] + 2, p[1]:p[1] + 2, p[2]:p[2] + 2].astype(np.float64).reshape(-1)
        if np.allclose(value, v):
            return False
        return v.min() <= value and v.max() >= value

    visited, found = set(), []
    for (low_point, high_point) in np.array(end_points, dtype=int).reshape(-1, 2, 3):
        low_value, high_value = f(low_point), f(high_point)
        if low_value > value or high_value < value:
            (low_point, low_value, high_point, high_value) = (high_point, high_value, low_point, low_value)
        assert low_value <= value and high_value >= value, \
            "Bad end points " + repr((tuple(low_point), low_value, tuple(high_point), high_value, value))
        while np.any(np.abs(low_point - high_point) > 1):
            mid_point = (low_point + high_point) // 2
            if f(mid_point) < value:
                low_point = mid_point
            else:
                high_point = mid_point
        for point in (low_point, high_point):
            tpoint = tuple(int(x) for x in point)
            if tpoint in visited:
                continue
            visited.add(tpoint)
            if border(point):
                found.append(tpoint)
                continue
            for offset_point in OFFSETS + point.reshape(1, 3):
                toffset = tuple(int(x) for x in offset_point)
                if toffset in visited:
                    continue
                visited.add(toffset)
                if border(offset_point):
                    found.append(toffset)
                    break
    return np.array(sorted(set(found)), dtype=np.int32).reshape(-1, 3)


def components_to_keep(table, rule):
    """What GridContour3d.keep_components asks for, on a component table (engine.COMPONENT_DTYPE): an int k names the k
    components with the most triangles (ties: the smaller component number; triangle counts are exact, so the choice
    is deterministic), a callable is called with the table and returns a boolean mask or component indices."""
    if isinstance(rule, numbers.Integral) and not isinstance(rule, bool):
        if rule < 0:
            raise ValueError("keep_components = %d: a number of components >= 0" % rule)
        return np.argsort(-table["n_tris"], kind="stable")[:int(rule)]
    if callable(rule):
        return rule(table)
    raise TypeError("keep_components: None, an int or a callable, not %r" % (rule,))


class GridContour3d(object):
    """Grid-coordinate engine front end (reference: GridContour + GridContour3d, tetrahedral.py:109-621).

    `function` may be an array of samples; uint8 / int16 / uint16 arrays reach the engine as they are (the result is
    that of their float64 copy), other non-float types are widened to float64."""

    flatten = False
    smooth = None
    minimum_ratio = 0.05
    minimum_extent = None
    geometry_dtype = np.float64
    reference_orientation = False
    want_normals = False
    full_scan = False                                  # set by search_for_endpoints(): the seeds are every crossing
    post_process = True                                # quantize / tiny / clean / orient like the reference
    quantize_divisions = 10000                         # tetrahedral.py:190
    tiny_epsilon = 1e-4                                # tetrahedral.py:353
    prefetched = None                                  # (engine, run_serial, flags, counts) of a run search_for_endpoints() made
    # vertex_fields: an array or callable, or a list of them, sampled on the field's grid (arrays may carry a trailing
    # axis of up to 4 components); get_points_and_triangles() then leaves their values at the returned points in
    # vertex_values (one array, or a list for a list), row for row (ctr_mt3d_interpolate)
    vertex_fields = None
    vertex_values = None
    field_grid = None                                  # world drivers: the FunctionGrid that callables are sampled on
    # measure_components: get_points_and_triangles() then leaves the edge-connected components of the returned mesh in
    # triangle_components ([T] int32, row for row with the returned triangles) and component_table (engine.COMPONENT_DTYPE:
    # counts, area, signed volume, box per component; ctr_mt3d_components)
    measure_components = False
    triangle_components = None
    component_table = None
    # keep_components: None (everything), an int k (the k components with the most triangles) or a callable
    # table -> boolean mask or component indices; get_points_and_triangles() then returns only those components
    # (ctr_mt3d_keep_components), and vertex_values / triangle_components / component_table describe that mesh
    keep_components = None
    # smooth_iterations > 0: get_points_and_triangles() smooths the mesh on the device (Taubin lambda|mu,
    # ctr_mt3d_smooth) after the component filter and before vertex_fields / measure_components, which then describe
    # the smoothed mesh; vertices on boundary or non-manifold edges stay put.  `smooth` (the reference's
    # smooth_interpolations) is a different algorithm and still raises.
    smooth_iterations = 0
    smooth_lambda = 0.5
    smooth_mu = -0.53
    # decimate_cell (a number or 3 numbers, in voxels): get_points_and_triangles() reduces the mesh on the device by
    # quadric vertex clustering (ctr_mt3d_decimate) on cells of decimate_cell * |delta| aligned with the voxel grid,
    # after the component filter and smoothing and before vertex_fields / measure_components, which then describe the
    # decimated mesh.  `flatten` (the reference's LP-based collapse_flat_segments) is a different algorithm and still
    # raises.
    decimate_cell = None
    # cap = "high" / "low" (with post_process = False, on a full scan): get_points_and_triangles() closes the surface at
    # the faces of the volume's box on the device (ctr_mt3d_cap), right after the run and before the reference
    # orientation, the component filter, smoothing, decimation, vertex_fields and measure_components: the region
    # f >= value ("high") or f < value ("low") then has a closed boundary, and its components are enclosed volumes.
    # Smoothing after the cap rounds the box edges (the cap's rim vertices are no longer fixed); Engine users who want
    # flat caps smooth first, then cap.
    cap = None

    def __init__(self, corner, function, value, segment_endpoints, linear_interpolate=True, callback=None,
                 origin=(0.0, 0.0, 0.0), delta=(1.0, 1.0, 1.0)):
        self.corner = np.array(corner, dtype=int)
        (self.dimension,) = self.corner.shape
        self.sanity_check()
        if not linear_interpolate:
            raise NotImplementedError("linear_interpolate=False evaluates the callable off-grid "
                                      "(tetrahedral.py:488-505); the array engine cannot")
        self.linear_interpolate = linear_interpolate
        self.end_points = segment_endpoints
        self.f = function
        self.value = value
        self.callback = callback
        self.origin = origin
        self.delta = delta
        self.normals = None
        self.counts = None

    def sanity_check(self):
        assert self.dimension == 3

    def _field(self):
        return self._samples_of(self.f)

    def _samples_of(self, f, components=False):
        """Samples of `f` on the grid of the isosurface's field: an array as it is (components=True: a trailing axis of
        components allowed), a callable sampled at the grid points (on field_grid for the world-coordinate drivers)."""
        want = tuple(int(c) + 1 for c in self.corner)
        if isinstance(f, np.ndarray):
            if tuple(f.shape) != want and not (components and f.ndim == 4 and tuple(f.shape[:3]) == want):
                raise ValueError("sample array has shape %r, corner %r needs %r" % (f.shape, tuple(self.corner), want))
            return f
        if self.field_grid is not None:
            g = self.field_grid
            return grid_field.FunctionGrid(g.mins, g.maxes, g.delta, f).samples(1)
        g = grid_field.FunctionGrid([0, 0, 0], [c for c in self.corner], [1, 1, 1], f)
        assert tuple(g.grid_dimensions) == want, (tuple(g.grid_dimensions), want)
        return g.samples(0)

    def get_points_and_triangles(self, clean=True):
        if self.flatten or self.smooth:
            # the reference's flatten solves an LP per edge, serially, and smooth is its own smoothing: the engine's
            # smoothing and decimation are other algorithms behind their own options (smooth_iterations,
            # decimate_cell), so these keep raising rather than silently giving a different mesh
            raise NotImplementedError("flatten / smooth (LP-based decimation, tetrahedral.py:217-351) are out of scope")
        eng = E.default_engine()
        flags = (E.GEOM_F64 if np.dtype(self.geometry_dtype) == np.float64 else 0) | (E.WANT_NORMALS if self.want_normals else 0)
        if self.vertex_fields is not None or self.cap is not None:
            flags |= E.WANT_KEYS                          # the values are interpolated, the rim found, along the keys
        seeded = not self.full_scan and self.end_points is not None
        if self.cap is not None:
            if self.cap not in E.CAP_SIDES:
                raise ValueError("cap must be None, 'high' or 'low', not %r" % (self.cap,))
            if self.post_process:
                raise ValueError("cap needs post_process = False: the reference's post-processing would merge and rewind "
                                 "the capped mesh")
            if seeded:
                raise ValueError("cap needs a full scan: a seeded selection keeps part of the surface, whose rim the caps "
                                 "would not meet")
        field = self._field()
        identity = tuple(float(x) for x in self.origin) == (0.0, 0.0, 0.0) and tuple(float(x) for x in self.delta) == (1.0, 1.0, 1.0)
        # with post-processing the run is made in grid coordinates and ctr_mt3d_clean applies the transform last, like
        # the reference (tetrahedral.py:86-90)
        run_origin, run_delta = ((0.0, 0.0, 0.0), (1.0, 1.0, 1.0)) if self.post_process else (self.origin, self.delta)
        pre = self.prefetched
        self.prefetched = None
        if (pre is not None and pre[0] is eng and pre[1] == eng.run_serial and (pre[2] & flags) == flags and
                (pre[2] & E.GEOM_F64) == (flags & E.GEOM_F64) and (self.post_process or identity)):
            self.counts = pre[3]                          # search_for_endpoints() made this very run: nothing to redo
        else:
            self.counts = eng.mt3d_run(field, self.value, origin=run_origin, delta=run_delta, flags=flags)
        if seeded:
            # seeded tracking: only what the flood fill reaches from the seeds' start voxels (no seeds: nothing)
            self.start_voxels = initial_voxels(field, self.value, self.end_points) if len(self.end_points) else \
                np.zeros((0, 3), np.int32)
            self.selected = eng.mt3d_select_seeded(self.start_voxels)
        if self.cap is not None:
            # on the mesh as extracted: the field still tells where its rim is and which way it faces
            self.capped = eng.mt3d_cap(self.cap)
        if self.post_process:
            # tetrahedral.py:541-552 on the device mesh: quantize, tiny, clean (if asked), orient, grid -> world
            self.cleaned = eng.mt3d_clean(self.corner, origin=self.origin, delta=self.delta, divisions=self.quantize_divisions,
                                          epsilon=self.tiny_epsilon, orient=True, triangles=bool(clean))
            self.components, self.flipped = int(self.cleaned.n_components), int(self.cleaned.n_flipped)
        elif self.reference_orientation:
            # surface_geometry.py:52-140 on the device mesh: one keep / reverse decision per edge-connected component
            self.components, self.flipped = eng.mt3d_orient_reference()
        if self.keep_components is not None:
            # after every pass that edits the mesh, before the values and the measurement below
            _, table = eng.mt3d_components()
            eng.mt3d_keep_components(components_to_keep(table, self.keep_components))
        smoothed = self.smooth_iterations > 0
        if smoothed:
            # after the filter (its components are measured on the unsmoothed mesh), before the values and the
            # measurement below
            eng.mt3d_smooth(self.smooth_iterations, self.smooth_lambda, self.smooth_mu)
        decimated = self.decimate_cell is not None
        if decimated:
            # after the filter and smoothing, before the values and the measurement below; cells of decimate_cell
            # voxels in the world coordinates the mesh has by now, aligned with the voxel grid
            cell = np.asarray(self.decimate_cell, np.float64) * np.abs(np.asarray(self.delta, np.float64))
            eng.mt3d_decimate(cell, origin=tuple(float(x) for x in self.origin))
        if self.vertex_fields is not None:
            # after every pass that edits the mesh: the values line up with the points fetched below
            many = isinstance(self.vertex_fields, (list, tuple))
            vals = [eng.mt3d_interpolate(self._samples_of(f, components=True))
                    for f in (self.vertex_fields if many else [self.vertex_fields])]
            self.vertex_values = vals if many else vals[0]
        if self.measure_components:
            # after every pass that edits the mesh, like the values above; the filter has already measured this mesh,
            # unless smoothing or decimation has changed it since
            self.triangle_components, self.component_table = \
                eng.mt3d_components_fetch() if self.keep_components is not None and not (smoothed or decimated) \
                else eng.mt3d_components()
        out = eng.mt3d_fetch()
        self.normals = out["normals"]
        points, triangles = out["verts"], out["tris"]
        if self.callback:
            self.callback(self)
        return (points, triangles)

    def extract_surface_geometry(self, clean=True):
        points, triangles = self.get_points_and_triangles(clean)
        geometry = surface_geometry.SurfaceGeometry(points, triangles)
        if not self.post_process:
            if clean:
                geometry.clean_triangles()
            geometry.orient_triangles()
        return geometry


def Grid3DContour(horizontal_n, vertical_m, forward_l, function, value, segment_endpoints,
                  linear_interpolate=True, callback=None):
    return GridContour3d((horizontal_n, vertical_m, forward_l), function, value, segment_endpoints, linear_interpolate,
                         callback)


class Delta3DContour(object):
    """World-coordinate driver (reference: triangulated.ContourGrid + tetrahedral.Delta3DContour)."""

    linear_interpolate = True
    flatten = False
    minimum_ratio = None
    minimum_extent = None
    smooth = None

    def __init__(self, function_grid, value, segment_endpoints=None, linear_interpolate=True):
        self.linear_interpolate = linear_interpolate
        self.grid = function_grid
        self.value = value
        self.segment_endpoints = segment_endpoints
        self.grid_endpoints = None
        self.contour_maker = self.get_contour_maker(None)

    def get_contour_maker(self, grid_endpoints):
        grid = self.grid
        self.grid_endpoints = grid_endpoints
        maker = GridContour3d(tuple(int(n) for n in grid.grid_dimensions), grid.samples(1), self.value, grid_endpoints,
                              linear_interpolate=self.linear_interpolate, origin=tuple(grid.mins), delta=tuple(grid.delta))
        maker.flatten = self.flatten
        maker.smooth = self.smooth
        maker.full_scan = True      # this facade only ever passes the complete seed set (triangulated.py:96 at HEAD)
        maker.prefetched = getattr(grid_endpoints, "engine_run", None)
        return self._configure(maker)

    def _configure(self, maker):
        "options set on this driver (before or after the maker was built) reach the maker"
        for name in ("post_process", "geometry_dtype", "want_normals", "reference_orientation", "quantize_divisions",
                     "tiny_epsilon", "vertex_fields", "measure_components", "keep_components", "smooth_iterations",
                     "smooth_lambda", "smooth_mu", "decimate_cell", "cap"):
            if hasattr(self, name):
                setattr(maker, name, getattr(self, name))
        maker.field_grid = self.grid
        return maker

    def search_for_endpoints(self, skip=1):
        (maxf, minf, grid_endpoints) = self.grid.find_contour_crossing_grid_segments(self.value, skip)
        self.grid_endpoints = grid_endpoints
        self.contour_maker = self.get_contour_maker(grid_endpoints)

    def get_points_and_triangles(self):
        # the engine applies grid_field.from_grid_coordinates (x*delta + mins) on the device
        maker = self._configure(self.contour_maker)
        result = maker.get_points_and_triangles()
        self.vertex_values = maker.vertex_values       # values of vertex_fields (when set) at the returned points
        self.triangle_components = maker.triangle_components   # with measure_components: aligned with the triangles
        self.component_table = maker.component_table
        return result


class TriangulatedIsosurfaces(Delta3DContour):

    def __init__(self, mins, maxes, delta, function, value, segment_endpoints,
                 linear_interpolate=True, flatten=False, minimum_ratio=None, minimum_extent=None, smooth=None):
        self.flatten = flatten
        self.smooth = smooth
        if minimum_ratio is not None:
            self.minimum_ratio = minimum_ratio
        if minimum_extent is not None:
            self.minimum_extent = minimum_extent
        grid = grid_field.FunctionGrid(mins, maxes, delta, function)
        Delta3DContour.__init__(self, grid, value, segment_endpoints, linear_interpolate=linear_interpolate)
