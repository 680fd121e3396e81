"""Python mirror of ftk::critical_point_tracker_{2d,3d}_regular over the C ABI (libftkb200.so).

Method names, argument meaning and call order follow the reference classes
(ref: include/ftk/filters/critical_point_tracker_2d_regular.hh, critical_point_tracker_3d_regular.hh,
regular_tracker.hh:24-30, critical_point_tracker.hh:64-69,105,126-132); all work happens in the CUDA
library -- there is no CPU path here.

Arrays are passed in *memory order*: the reference's ndarray is dim-0-fastest, so a scalar layer
(W,H[,D]) is a C-contiguous numpy array of shape ([D,]H,W), a vector layer (n,W,H[,D]) has shape
([D,]H,W,n) and a Jacobian layer (n,n,W,H[,D]) has shape ([D,]H,W,n,n).
"""
import ctypes as C

import numpy as np

from . import _lib as L

SOURCE_NONE, SOURCE_GIVEN, SOURCE_DERIVED = L.SOURCE_NONE, L.SOURCE_GIVEN, L.SOURCE_DERIVED

# ref: include/ftk/numeric/critical_point_type.hh:10-36, 95-118
CRITICAL_POINT_2D_DEGENERATE, CRITICAL_POINT_2D_MINIMUM, CRITICAL_POINT_2D_SADDLE, CRITICAL_POINT_2D_MAXIMUM = 1, 2, 4, 8


def critical_point_type_to_string(cpdims, ctype, scalar):
    """ref: critical_point_type.hh:95-118"""
    if cpdims == 2:
        if scalar:
            return {0x1: "degenerate", 0x2: "min", 0x4: "saddle", 0x8: "max"}.get(ctype, "unknown")
        return {0x1: "degenerate", 0x8: "attracting", 0x2: "repelling", 0x4: "saddle", 0x10: "attracting_focus",
                0x20: "repelling_focus", 0x40: "center"}.get(ctype, "unknown")
    if cpdims == 3:
        if scalar:
            return {0x1: "degenerate", 0x2: "min", 0x4: "saddle", 0x8: "max"}.get(ctype, "unknown")
        return "unknown"
    return "unknown"


class Lattice:
    """ftk::lattice(starts, sizes) (ref: include/ftk/mesh/lattice.hh:16-69)"""

    def __init__(self, starts, sizes):
        self.starts = [int(s) for s in starts]
        self.sizes = [int(s) for s in sizes]

    def lower_bounds(self):
        return list(self.starts)

    def upper_bounds(self):
        return [s + n - 1 for s, n in zip(self.starts, self.sizes)]


def _dev_ptr(a):
    """device pointer of a torch CUDA tensor / anything with __cuda_array_interface__, else None"""
    if hasattr(a, "__cuda_array_interface__"):
        return int(a.__cuda_array_interface__["data"][0])
    if hasattr(a, "data_ptr") and getattr(a, "is_cuda", False):
        return int(a.data_ptr())
    return None


class _RegularTracker:
    ND = 0

    def __init__(self, comm=None, device=0):
        self._device = int(device)
        self._h = None
        self._domain = None
        self._array_domain = None
        self._scalar_source = SOURCE_NONE
        self._vector_source = SOURCE_NONE
        self._jacobian_source = SOURCE_NONE
        self._symmetric = False
        self._robust = True
        self._degrees = False
        self._type_filter = None
        self._start_timestep = 0
        self._resolution_init = 0.0
        self._streaming = False
        self._coords = None
        self._point_capacity = 0
        self._keep = []   # borrowed device arrays stay referenced while resident

    # ---- configuration (same names as the reference) ------------------------------------------
    def set_domain(self, lattice):
        self._domain = lattice

    def set_array_domain(self, lattice):
        self._array_domain = lattice

    def set_scalar_field_source(self, s):
        self._scalar_source = int(s)

    def set_vector_field_source(self, s):
        self._vector_source = int(s)

    def set_jacobian_field_source(self, s):
        self._jacobian_source = int(s)

    def set_jacobian_symmetric(self, b):
        self._symmetric = bool(b)

    def set_enable_robust_detection(self, b):
        self._robust = bool(b)

    def set_enable_computing_degrees(self, b):
        self._degrees = bool(b)

    def set_type_filter(self, f):
        self._type_filter = int(f)

    # physical coordinates (ref: regular_tracker.hh:38-40); applied at initialize()
    def set_coords_bounds(self, bounds):
        self._coords = (L.COORDS_BOUNDS, np.ascontiguousarray(bounds, np.float64).ravel())

    def set_coords_rectilinear(self, arrays):
        self._coords = (L.COORDS_RECTILINEAR, np.concatenate([np.ascontiguousarray(a, np.float64).ravel() for a in arrays]))

    def set_coords_explicit(self, coords):
        """coords in memory order: shape (H, W, ncomp)"""
        self._coords = (L.COORDS_EXPLICIT, np.ascontiguousarray(coords, np.float64).ravel())

    def set_enable_streaming_trajectories(self, b):
        """ref: critical_point_tracker.hh:38 -- trajectories grown after every interval sweep (hh:522-641)"""
        self._streaming = bool(b)

    def set_start_timestep(self, t):
        self._start_timestep = int(t)

    def set_current_timestep(self, t):
        self._start_timestep = int(t)

    def set_initial_resolution(self, r):
        """running min non-zero |v| inherited from earlier time slabs (multi-GPU time sharding)"""
        self._resolution_init = float(r)

    def set_number_of_threads(self, n):
        pass   # the sweep runs on the GPU

    def use_accelerator(self, name):
        if str(name).lower() not in ("cuda", "b200", "ftkb200"):
            raise ValueError("ftk_b200 only runs on CUDA (sm_100a); there is no CPU or other back end")

    def set_device_ids(self, ids):
        self._device = int(ids[0])

    def initialize(self):
        if self._array_domain is None:
            raise RuntimeError("set_array_domain() must be called before initialize()")
        dims = self._array_domain.sizes
        nd = self.ND
        if len(dims) != nd:
            raise ValueError("array domain dimensionality mismatch")
        dom = self._domain or Lattice([0] * nd, dims)
        cfg = L.Config()
        cfg.abi_version = L.ABI_VERSION
        cfg.nd = nd
        lb, ub = dom.lower_bounds(), dom.upper_bounds()
        for i in range(3):
            cfg.dims[i] = dims[i] if i < nd else 1
            cfg.lb[i] = lb[i] - self._array_domain.starts[i] if i < nd else 0
            cfg.ub[i] = ub[i] - self._array_domain.starts[i] if i < nd else 0
        cfg.scalar_source, cfg.vector_source, cfg.jacobian_source = self._scalar_source, self._vector_source, self._jacobian_source
        cfg.jacobian_symmetric = int(self._symmetric)
        cfg.robust_detection = int(self._robust)
        cfg.compute_degrees = int(self._degrees)
        cfg.use_type_filter = int(self._type_filter is not None)
        cfg.type_filter = int(self._type_filter or 0)
        cfg.start_timestep = self._start_timestep
        cfg.device = self._device
        cfg.resolution_init = self._resolution_init
        cfg.point_capacity = int(self._point_capacity)
        h = C.c_void_p()
        rc = L.lib().ftkb_create(C.byref(cfg), C.byref(h))
        if rc:
            raise L.FTKBError(rc, L.lib().ftkb_last_error(None).decode())
        self._h = h
        self._dims = list(dims)
        if self._streaming:
            self._check(L.lib().ftkb_set_streaming_trajectories(self._h, 1))
        if self._coords is not None:
            mode, data = self._coords
            self._check(L.lib().ftkb_set_coords(self._h, mode, data.ctypes.data, data.size))

    def reset(self):
        self.close()

    def close(self):
        if self._h:
            L.lib().ftkb_destroy(self._h)
            self._h = None
        self._keep = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise L.FTKBError(rc, L.lib().ftkb_last_error(self._h).decode())

    # ---- data ----------------------------------------------------------------------------------
    def _shape(self, trailing):
        return tuple(reversed(self._dims)) + tuple(trailing)

    def push_field_data_snapshot(self, scalar=None, vector=None, jacobian=None, borrow=False):
        """ref: critical_point_tracker.hh:202-213.  Host numpy arrays are copied; CUDA tensors are
        copied device-to-device, or used in place with borrow=True."""
        n = self.ND
        given = [a for a in (scalar, vector, jacobian) if a is not None]
        if jacobian is None and given and all(isinstance(a, np.ndarray) and a.dtype == np.float32 for a in given):
            # float32 host arrays travel as float32 and are widened on the device (same values as widening here first)
            ptrs, hold = [], []
            for a, trailing in ((scalar, ()), (vector, (n,))):
                if a is None:
                    ptrs.append(None)
                    continue
                h = np.ascontiguousarray(a)
                if h.size != int(np.prod(self._shape(trailing))):
                    raise ValueError(f"array has {h.size} elements, expected {int(np.prod(self._shape(trailing)))}")
                ptrs.append(h.ctypes.data)
                hold.append(h)
            self._check(L.lib().ftkb_push_snapshot_f32(self._h, ptrs[0], ptrs[1]))
            return
        ptrs, where, hold = [], None, []
        for a, trailing in ((scalar, ()), (vector, (n,)), (jacobian, (n, n))):
            if a is None:
                ptrs.append(None)
                continue
            dp = _dev_ptr(a)
            count = int(np.prod(self._shape(trailing)))
            if dp is not None:
                if int(np.prod(tuple(a.shape))) != count or (hasattr(a, "is_contiguous") and not a.is_contiguous()):
                    raise ValueError("device array has the wrong size or is not contiguous")
                kind = L.MEM_DEVICE_BORROW if borrow else L.MEM_DEVICE
                ptrs.append(dp)
                hold.append(a)
            else:
                h = np.ascontiguousarray(a, dtype=np.float64)
                if h.size != count:
                    raise ValueError(f"array has {h.size} elements, expected {count}")
                kind = L.MEM_HOST
                ptrs.append(h.ctypes.data)
                hold.append(h)
            if where is not None and where != kind:
                raise ValueError("scalar/vector/jacobian must all be host arrays or all be device arrays")
            where = kind
        if where == L.MEM_DEVICE_BORROW:
            self._keep.append(hold)
            self._keep = self._keep[-6:]          # a borrowed layer is read until its sweeps are confirmed (ftkb200.h)
        if where in (L.MEM_DEVICE, L.MEM_DEVICE_BORROW):
            self._order_after_producer(hold)
        # copied arrays (host, or device without borrow) are consumed before the call returns; `hold` lives until then
        self._check(L.lib().ftkb_push_snapshot(self._h, ptrs[0], ptrs[1], ptrs[2], where if where is not None else L.MEM_HOST))

    def _order_after_producer(self, arrays):
        """device inputs: make the context's stream wait for the stream that (may still be) writing them -- torch's current
        stream for torch tensors (ftkb_set_producer_stream); other producers synchronise before pushing"""
        stream = None
        for a in arrays:
            if getattr(a, "is_cuda", False) and hasattr(a, "data_ptr"):
                import torch
                stream = int(torch.cuda.current_stream(a.device).cuda_stream)
        if stream is not None:
            self._check(L.lib().ftkb_set_producer_stream(self._h, C.c_void_p(stream), 1))

    def push_device_pointers(self, scalar=0, vector=0, jacobian=0, stream=None):
        """Raw device pointers (ints), used in place (FTKB_MEM_DEVICE_BORROW): the thinnest wrapper over
        ftkb_push_snapshot for callers that keep their time series resident in HBM.  The arrays must stay
        valid and unchanged until three advance_timestep() calls later (or synchronize()).  stream: the CUDA stream
        (int handle) that produced them, if it has not been synchronised."""
        if stream is not None:
            self._check(L.lib().ftkb_set_producer_stream(self._h, C.c_void_p(int(stream)), 1))
        self._check(L.lib().ftkb_push_snapshot(self._h, scalar or None, vector or None, jacobian or None, L.MEM_DEVICE_BORROW))

    def export_layer_cells(self, index=0):
        """(device pointer, bytes, min non-zero |v|) of the range cells of resident layer `index`; the buffer stays alive until
        close() so that a neighbouring time slab can read it through NVLink peer memory (ftkb_export_layer_cells)"""
        ptr, nbytes, res = C.c_void_p(), C.c_uint64(), C.c_double()
        self._check(L.lib().ftkb_export_layer_cells(self._h, int(index), C.byref(ptr), C.byref(nbytes), C.byref(res)))
        return int(ptr.value), int(nbytes.value), float(res.value)

    def push_remote_snapshot(self, scalar=0, vector=0, cells=0, resolution=0.0):
        """a layer that lives in a peer process's memory (pointers from _lib.ipc_import) together with its range cells and
        its min non-zero |v|: the sweep reads the cells and the sparse vertices it needs over NVLink, nothing is copied"""
        self._check(L.lib().ftkb_push_snapshot_remote(self._h, scalar or None, vector or None, cells or None, float(resolution)))

    def push_scalar_field_snapshot(self, scalar, borrow=False):
        self.push_field_data_snapshot(scalar=scalar, borrow=borrow)

    def push_vector_field_snapshot(self, vector, borrow=False):
        self.push_field_data_snapshot(vector=vector, borrow=borrow)

    def push_synthetic_snapshot(self, kind, params, t):
        p = (C.c_double * max(len(params), 1))(*[float(v) for v in params])
        self._check(L.lib().ftkb_push_synthetic(self._h, int(kind), p, len(params), float(t)))

    def update_timestep(self):
        self._check(L.lib().ftkb_update_timestep(self._h))

    def advance_timestep(self):
        self._check(L.lib().ftkb_advance_timestep(self._h))

    def finalize(self):
        self._check(L.lib().ftkb_finalize(self._h))

    def synchronize(self):
        self._check(L.lib().ftkb_synchronize(self._h))

    @property
    def current_timestep(self):
        t = C.c_int32()
        self._check(L.lib().ftkb_current_timestep(self._h, C.byref(t)))
        return t.value

    def last_layer_resolution(self):
        r = C.c_double()
        self._check(L.lib().ftkb_last_layer_resolution(self._h, C.byref(r)))
        return r.value

    def set_resolution(self, r):
        self._check(L.lib().ftkb_set_resolution(self._h, float(r)))

    # ---- results -------------------------------------------------------------------------------
    def get_discrete_critical_points(self):
        """structured array (L.POINT_DTYPE) sorted by the reference's element order"""
        n = C.c_uint64()
        self._check(L.lib().ftkb_num_points(self._h, C.byref(n)))
        out = np.empty(n.value, L.POINT_DTYPE)       # filled completely by the copy below
        if n.value:
            self._check(L.lib().ftkb_get_points(self._h, out.ctypes.data, n.value))
        starts = self._array_domain.starts if self._array_domain is not None else []
        if n.value and any(starts):
            # the library works in array-relative indices; the reference's positions are absolute
            # (regular_tracker.hh:24-30; the C++ shim does the same in to_feature_point)
            for j, s0 in enumerate(starts):
                out["corner"][:, j] += s0
                if self._coords is None:
                    out["x"][:, j] += float(s0)
        return out

    get_critical_points = get_discrete_critical_points

    def import_points(self, pts):
        pts = np.ascontiguousarray(pts, dtype=L.POINT_DTYPE)
        starts = self._array_domain.starts if self._array_domain is not None else []
        if len(pts) and any(starts):          # back to the library's array-relative indices (see get_discrete_critical_points)
            pts = pts.copy()
            for j, s0 in enumerate(starts):
                pts["corner"][:, j] -= s0
                if self._coords is None:
                    pts["x"][:, j] -= float(s0)
        self._check(L.lib().ftkb_import_points(self._h, pts.ctypes.data, len(pts)))

    def get_trajectory_index(self):
        """-> list of (index array into get_discrete_critical_points(), loop flag)"""
        nt = C.c_uint64()
        self._check(L.lib().ftkb_num_trajectories(self._h, C.byref(nt)))
        n = C.c_uint64()
        self._check(L.lib().ftkb_num_points(self._h, C.byref(n)))
        npts = int(n.value)
        off = np.zeros(nt.value + 1, np.uint64)
        idx = np.zeros(max(npts, 1), np.uint64)
        loop = np.zeros(max(nt.value, 1), np.uint8)
        self._check(L.lib().ftkb_get_trajectories(self._h, off.ctypes.data, idx.ctypes.data, loop.ctypes.data))
        return [(idx[int(off[i]):int(off[i + 1])].astype(np.int64), bool(loop[i])) for i in range(nt.value)]

    def get_trajectory_complete(self):
        """feature_curve_t::complete of every trajectory (set by the streaming grow step; all False otherwise)"""
        nt = C.c_uint64()
        self._check(L.lib().ftkb_num_trajectories(self._h, C.byref(nt)))
        out = np.zeros(max(nt.value, 1), np.uint8)
        self._check(L.lib().ftkb_get_trajectory_complete(self._h, out.ctypes.data))
        return out[:nt.value].astype(bool)

    def live_curveset(self):
        """streaming trackers, at any time: (grown_through, CurveSet) -- the trajectories grown so far (the reference's
        traced_critical_points) and the last timestep whose grow step has run (start timestep - 1 before the first);
        CurveSet.slice(t) holds the points of timestep t once t <= grown_through.  Equal to CurveSet.from_tracker after finalize."""
        from .curves import CurveSet
        return CurveSet.live(L.lib().ftkb_get_live_curveset, self._h, self._check)

    def get_traced_critical_points(self):
        """list of trajectories, each a structured array of points in trace order (with .loop in the
        second tuple member); the counterpart of feature_curve_set_t"""
        pts = self.get_discrete_critical_points()
        return [(pts[idx], loop) for idx, loop in self.get_trajectory_index()]

    def get_component_labels(self):
        n = len(self.get_discrete_critical_points())
        out = np.zeros(max(n, 1), np.uint64)
        self._check(L.lib().ftkb_get_component_labels(self._h, out.ctypes.data))
        return out[:n]

    def get_degrees(self):
        n = len(self.get_discrete_critical_points())
        out = np.zeros(max(n, 1), np.int32)
        self._check(L.lib().ftkb_get_degrees(self._h, out.ctypes.data))
        return out[:n]

    def get_last_worklist(self):
        """diagnostic: linear corner indices (x fastest over the domain) the last scan left for the exact test"""
        n = C.c_uint64()
        self._check(L.lib().ftkb_get_last_worklist(self._h, None, 0, C.byref(n)))
        out = np.zeros(max(n.value, 1), np.uint64)
        self._check(L.lib().ftkb_get_last_worklist(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out[:n.value]

    def get_layer(self, index=0):
        """diagnostic: resident snapshot `index` (0 = current) copied to the host, in memory order -> (scalar, vector), None
        for a field the snapshot does not hold (what ftkb_push_synthetic generated on the device)"""
        n = self.ND
        out = []
        for trailing, src in (((), self._scalar_source), ((n,), self._vector_source)):
            if src != SOURCE_GIVEN:
                out.append(None)
                continue
            a = np.zeros(self._shape(trailing), np.float64)
            args = (a.ctypes.data, None) if not trailing else (None, a.ctypes.data)
            self._check(L.lib().ftkb_get_layer(self._h, int(index), *args))
            out.append(a)
        return tuple(out)

    def stats(self):
        s = L.Stats()
        self._check(L.lib().ftkb_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def timer_start(self):
        self._check(L.lib().ftkb_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_double()
        self._check(L.lib().ftkb_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def reset_stats(self):
        self._check(L.lib().ftkb_reset_stats(self._h))


class critical_point_tracker_2d_regular(_RegularTracker):
    ND = 2


class critical_point_tracker_3d_regular(_RegularTracker):
    ND = 3


def make_tracker(dims, field="scalar", lb=None, ub=None, jacobian_symmetric=None, robust=True, compute_degrees=False,
                 type_filter=None, start_timestep=0, device=0, resolution_init=0.0,
                 scalar_source=None, vector_source=None, jacobian_source=None, streaming=False, coords=None, point_capacity=0):
    """Configure a tracker the way the reference's front ends do (json_interface.hh:634-656):
    scalar input -> lattice({2,..}, {D-3,..}) = [2, D-2], derived gradient/Hessian, symmetric;
    vector input -> lattice({1,..}, {D-2,..}) = [1, D-2], derived Jacobian, non-symmetric."""
    nd = len(dims)
    tr = (critical_point_tracker_2d_regular if nd == 2 else critical_point_tracker_3d_regular)(device=device)
    if field == "scalar":
        ss, vs, js, sym, margin = SOURCE_GIVEN, SOURCE_DERIVED, SOURCE_DERIVED, True, 2
    else:
        ss, vs, js, sym, margin = SOURCE_NONE, SOURCE_GIVEN, SOURCE_DERIVED, False, 1
    tr.set_scalar_field_source(ss if scalar_source is None else scalar_source)
    tr.set_vector_field_source(vs if vector_source is None else vector_source)
    tr.set_jacobian_field_source(js if jacobian_source is None else jacobian_source)
    tr.set_jacobian_symmetric(sym if jacobian_symmetric is None else jacobian_symmetric)
    tr.set_enable_robust_detection(robust)
    tr.set_enable_computing_degrees(compute_degrees)
    if type_filter is not None:
        tr.set_type_filter(type_filter)
    lo = [margin] * nd if lb is None else list(lb)
    hi = [d - 2 for d in dims] if ub is None else list(ub)
    tr.set_domain(Lattice(lo, [h - l + 1 for l, h in zip(lo, hi)]))
    tr.set_array_domain(Lattice([0] * nd, dims))
    tr.set_start_timestep(start_timestep)
    tr.set_initial_resolution(resolution_init)
    tr.set_enable_streaming_trajectories(streaming)
    tr._point_capacity = int(point_capacity)      # initial size of the punctured-simplex buffer (grows on demand)
    if coords is not None:
        tr._coords = coords_arg(coords)
    tr.initialize()
    return tr


def coords_arg(coords):
    """("bounds" | "rectilinear" | "explicit", flat data in the reference's order) -> (COORDS_* mode, float64 array)"""
    return ({"bounds": L.COORDS_BOUNDS, "rectilinear": L.COORDS_RECTILINEAR, "explicit": L.COORDS_EXPLICIT}[coords[0]],
            np.ascontiguousarray(coords[1], np.float64).ravel())


def track(snapshots, dims, field="scalar", trace=True, **kw):
    """The reference's front-end loop (python/pyftk.cpp:110-117, json_interface.hh:699-706)."""
    tr = make_tracker(dims, field=field, **kw)
    snaps = list(snapshots)
    for k, s in enumerate(snaps):
        if field == "scalar":
            tr.push_scalar_field_snapshot(s)
        else:
            tr.push_vector_field_snapshot(s)
        if k != 0:
            tr.advance_timestep()
        if k == len(snaps) - 1:
            tr.update_timestep()
    if trace:
        tr.finalize()
    return tr
